// NCSN++ forward executor: topology, packed-weight table, per-(B,F,T) buffer plan and launch list.
//
// Mirrors `NCSNpp.__init__` / `NCSNpp.forward` (sgmse-bbed/sgmse/backbones/ncsnpp.py:45-245, 247-404) for the
// configuration the reference instantiates (biggan blocks, FIR resampling, input_skip / output_skip
// pyramids with 'sum' combiner, Fourier embedding), plus the head of `ScoreModel.forward`
// (sgmse-bbed/sgmse/model.py:481-543).
//
// Data layout: activations NHWC bf16 in one caller-provided workspace; `torch.cat([h, skip])`
// (ncsnpp.py:337) is never materialised -- both producers write straight into channel slices of a
// shared buffer (views with a pixel pitch).  4-channel pyramids, GroupNorm statistics, attention
// scores and the time-embedding biases are fp32.  Buffers are placed by a lifetime-interval
// first-fit allocator, all launches of one forward are recorded once per (B,F,T) and replayed
// (CUDA-graph capturable: no allocation, no sync, no host reads).
#include <algorithm>
#include <functional>
#include <initializer_list>
#include <map>
#include <string>
#include <tuple>
#include <vector>

#include "kernels.h"

namespace {

enum PackKind {       // how the host packs a reference state-dict tensor into the weight blob
    PK_RAW_F32 = 0,   // flat copy, fp32
    PK_CONV3_K_BF16 = 1,  // [Cout,Cin,3,3] -> bf16 rows [cout][k_off + (r*3+s)*Cin + cin], row pitch row_stride
    PK_CONV1_K_BF16 = 2,  // [Cout,Cin,1,1] -> bf16 rows [cout][k_off + cin]
    PK_NIN_K_BF16 = 3,    // W[in,out]      -> bf16 rows [out][k_off + in]
    PK_CONV3_TAP_F32 = 4, // [Cout,Cin,3,3] -> fp32 [cout][r][s][cin]
    PK_CONV3_K_BF16_HILO64 = 5  // [Cout,Cin<=4,3,3] -> bf16 rows [cout][(r*3+s)*64 + c], c < 2*Cin: w[cout][c % Cin][r][s]
};

struct Param {
    std::string name;
    int kind;
    int64_t offset;      // bytes into the blob
    int64_t row_stride;  // elements (bf16 kinds)
    int64_t k_offset;    // elements (bf16 kinds)
    int accumulate;      // 1: add into the destination (fused biases)
    int ndim;
    int64_t dims[4];     // shape of the reference state-dict tensor
};

struct Mod {
    int kind;  // 0 fourier 1 linear 2 conv_in 3 res 4 attn 5 combine 6 gn 7 conv_out
    int cin = 0, cout = 0, up = 0, down = 0, has_c2 = 0;
    int tb_row = 0;       // row offset into the concatenated Dense_0 matrix
    // blob offsets of the parameters
    int64_t gn_g = 0, gn_b = 0;    // GroupNorm affine: gn; GroupNorm_0 of res and attn
    int64_t w = 0, b = 0;          // fourier W; linear; conv_in / conv_out (fp32 taps); combine Conv_0; res Conv_0;
                                   // attn NIN_0..2 as one [3C][C] qkv matrix
    int64_t w_tc = 0;              // conv_in / conv_out: bf16 tensor-core copy of w
    int64_t gn1_g = 0, gn1_b = 0;  // res GroupNorm_1
    int64_t w1 = 0, b1 = 0;        // res Conv_1 (| Conv_2 along K; b1 holds b1 + b2); attn NIN_3
};
enum { M_FOURIER, M_LINEAR, M_CONV_IN, M_RES, M_ATTN, M_COMBINE, M_GN, M_CONV_OUT };

struct LT {  // logical tensor
    int B, H, W, C;
    int esize;  // bytes per element: 2 (bf16 act), 4 (f32; C counts floats per pixel)
    int parent = -1, coff = 0;
    int first = 1 << 30, last = -1;
    int64_t off = -1, bytes = 0;
};

struct Engine;

struct Plan {
    Engine* eng;
    int B, F, T, flags;
    bool cross_check = false;   // flags bit1: fp32 CUDA-core convolutions and attention
    std::vector<LT> tens;
    std::vector<std::function<int(Plan&)>> builders;
    std::vector<std::function<int(cudaStream_t)>> launches;
    std::map<int, int> taps;  // module index -> tensor id
    // GroupNorm statistics by tensor: entry index into the fixed-point statistics arena t_stats (zeroed at the start
    // of every forward; an entry holds [B][128 units][2] 64-bit sums)
    std::map<int, int> stats_of;
    int n_stat_entries = 0;
    unsigned long long* stat_ptr(int entry) const {
        return reinterpret_cast<unsigned long long*>(ws + tens[t_stats].off) + (int64_t)entry * B * 256;
    }
    std::map<int, std::pair<int, int>> cat_children;
    // every convolution rec_conv / rec_conv_out records, in order (snrse_ncsnpp_dbg_convs); tensor ids < 0 are absent
    struct ConvRec {
        int x, taps, shortcut, res, out, n_rows;
        int path;   // 0 2-CTA kernel, 1 CUDA cores, 2 single-CTA implicit GEMM (the path codes of snrse_dbg_conv)
        bool norm, stats, tbias, bias, out4, addend;
        float scale;
    };
    std::vector<ConvRec> convs;
    int step = 0;
    int64_t ws_bytes = 0;
    uint8_t* ws = nullptr;
    // fixed slots
    int t_x4, t_tb, t_tscr, t_stats, t_scsh;
    // bound per call
    const float* t_ptr = nullptr;
    const float2 *x_ptr = nullptr, *y_ptr = nullptr;
    float2* out_ptr = nullptr;
    int mode = 0;

    // per launch group: kind (LK_*), algorithmic flops and bytes -- read by the profiling entry point
    struct Info { int kind; double flops, bytes; };
    std::vector<Info> info;
    void add(int kind, double flops, double bytes, std::function<int(cudaStream_t)> f) {
        launches.push_back(std::move(f));
        info.push_back(Info{kind, flops, bytes});
    }

    int root(int id) const {
        while (tens[id].parent >= 0) id = tens[id].parent;
        return id;
    }
    int new_t(int b, int h, int w, int c, int esize) {
        LT t;
        t.B = b; t.H = h; t.W = w; t.C = c; t.esize = esize;
        t.bytes = (int64_t)b * h * w * c * esize;
        tens.push_back(t);
        return (int)tens.size() - 1;
    }
    // Record one step: every tensor it reads or writes (ids < 0 are absent operands) lives at least through this step,
    // and `build` appends the step's launches once the buffers are placed.
    void record(std::initializer_list<int> ids, std::function<int(Plan&)> build) {
        for (int id : ids) {
            if (id < 0) continue;
            LT& r = tens[root(id)];
            r.first = std::min(r.first, step);
            r.last = std::max(r.last, step);
        }
        step++;
        builders.push_back(std::move(build));
    }
    int concat(int a, int b) {
        LT &ta = tens[a], &tb = tens[b];
        int c = new_t(ta.B, ta.H, ta.W, ta.C + tb.C, 2);
        tens[c].first = std::min(tens[a].first, tens[b].first);
        tens[c].last = std::max(tens[a].last, tens[b].last);
        tens[a].parent = c; tens[a].coff = 0;
        tens[b].parent = c; tens[b].coff = tens[a].C;
        cat_children[c] = {a, b};
        return c;
    }
    int chan_off(int id) const {   // first channel of tensor id inside its root buffer
        int coff = 0;
        for (int r = id; tens[r].parent >= 0; r = tens[r].parent) coff += tens[r].coff;
        return coff;
    }
    ActView view(int id) const {
        const int r = root(id);
        ActView v;
        v.ptr = reinterpret_cast<bf16*>(ws + tens[r].off) + chan_off(id);
        v.B = tens[id].B; v.H = tens[id].H; v.W = tens[id].W; v.C = tens[id].C;
        v.ld = tens[r].C;
        return v;
    }
    float* fptr(int id) const { return reinterpret_cast<float*>(ws + tens[root(id)].off); }
};

struct Engine {
    int nf = 128, n_levels = 0, num_res_blocks = 2, image_size = 256;
    std::vector<int> ch_mult, attn_res;
    std::vector<Mod> mods;
    std::vector<Param> params;
    int64_t blob_bytes = 0;
    const uint8_t* blob = nullptr;
    int dense_rows = 0;
    int64_t dense_w_off = 0, dense_b_off = 0;
    int64_t out_w_off = 0, out_b_off = 0;
    std::map<std::tuple<int, int, int>, Plan*> plans;

    int64_t alloc(int64_t bytes) {
        int64_t o = blob_bytes;
        blob_bytes += (bytes + 255) / 256 * 256;
        return o;
    }
    void add_param(const std::string& name, std::vector<int64_t> shape, int kind, int64_t off, int64_t row_stride = 0,
                   int64_t k_off = 0, int acc = 0) {
        Param p{name, kind, off, row_stride, k_off, acc, (int)shape.size(), {1, 1, 1, 1}};
        for (size_t i = 0; i < shape.size(); ++i) p.dims[i] = shape[i];
        params.push_back(p);
    }
    const float* wf(int64_t off) const { return reinterpret_cast<const float*>(blob + off); }
    const bf16* wb(int64_t off) const { return reinterpret_cast<const bf16*>(blob + off); }
};

bool in_list(const std::vector<int>& v, int x) { return std::find(v.begin(), v.end(), x) != v.end(); }

// ------------------------------------------------------------------------------------------------
// Topology + weight table (ncsnpp.py:99-245)
// ------------------------------------------------------------------------------------------------
int build_topology(Engine& e, int image_size) {
    const int nf = e.nf, L = e.n_levels;
    std::vector<Mod>& m = e.mods;
    auto res = [&](int cin, int cout, int up, int down) {
        Mod r; r.kind = M_RES; r.cin = cin; r.cout = cout; r.up = up; r.down = down;
        r.has_c2 = (cin != cout || up || down) ? 1 : 0;
        m.push_back(r);
    };
    auto attn = [&](int c) { Mod r; r.kind = M_ATTN; r.cin = r.cout = c; m.push_back(r); };
    { Mod r; r.kind = M_FOURIER; r.cout = nf; m.push_back(r); }
    { Mod r; r.kind = M_LINEAR; r.cin = 2 * nf; r.cout = 4 * nf; m.push_back(r); }
    { Mod r; r.kind = M_LINEAR; r.cin = 4 * nf; r.cout = 4 * nf; m.push_back(r); }
    { Mod r; r.kind = M_CONV_IN; r.cin = 4; r.cout = nf; m.push_back(r); }
    std::vector<int> hs_c{nf};
    int in_ch = nf;
    for (int lv = 0; lv < L; ++lv) {
        const int resol = image_size >> lv;
        for (int b = 0; b < e.num_res_blocks; ++b) {
            const int out_ch = nf * e.ch_mult[lv];
            res(in_ch, out_ch, 0, 0);
            in_ch = out_ch;
            if (in_list(e.attn_res, resol)) attn(in_ch);
            hs_c.push_back(in_ch);
        }
        if (lv != L - 1) {
            res(in_ch, in_ch, 0, 1);
            { Mod r; r.kind = M_COMBINE; r.cin = 4; r.cout = in_ch; m.push_back(r); }
            hs_c.push_back(in_ch);
        }
    }
    in_ch = hs_c.back();
    res(in_ch, in_ch, 0, 0);
    attn(in_ch);
    res(in_ch, in_ch, 0, 0);
    for (int lv = L - 1; lv >= 0; --lv) {
        const int resol = image_size >> lv;
        for (int b = 0; b < e.num_res_blocks + 1; ++b) {
            const int out_ch = nf * e.ch_mult[lv];
            res(in_ch + hs_c.back(), out_ch, 0, 0);
            hs_c.pop_back();
            in_ch = out_ch;
        }
        if (in_list(e.attn_res, resol)) attn(in_ch);
        { Mod r; r.kind = M_GN; r.cin = r.cout = in_ch; m.push_back(r); }
        { Mod r; r.kind = M_CONV_OUT; r.cin = in_ch; r.cout = 4; m.push_back(r); }
        if (lv != 0) res(in_ch, in_ch, 1, 0);
    }
    if (!hs_c.empty()) {
        snrse_set_error("internal: skip stack not empty");
        return SNRSE_ERR_STATE;
    }
    // ---- weight blob layout + parameter table
    const int d = 4 * nf;
    e.out_w_off = e.alloc(2 * 4 * 4);
    e.out_b_off = e.alloc(2 * 4);
    e.add_param("dnn.output_layer.weight", {2, 4, 1, 1}, PK_RAW_F32, e.out_w_off);
    e.add_param("dnn.output_layer.bias", {2}, PK_RAW_F32, e.out_b_off);
    int rows = 0;
    for (auto& r : m)
        if (r.kind == M_RES) { r.tb_row = rows; rows += r.cout; }
    e.dense_rows = rows;
    e.dense_w_off = e.alloc((int64_t)rows * d * 4);
    e.dense_b_off = e.alloc((int64_t)rows * 4);
    for (size_t i = 0; i < m.size(); ++i) {
        Mod& r = m[i];
        const std::string p = "dnn.all_modules." + std::to_string(i) + ".";
        switch (r.kind) {
            case M_FOURIER:
                r.w = e.alloc(nf * 4);
                e.add_param(p + "W", {nf}, PK_RAW_F32, r.w);
                break;
            case M_LINEAR:
                r.w = e.alloc((int64_t)r.cout * r.cin * 4);
                r.b = e.alloc(r.cout * 4);
                e.add_param(p + "weight", {r.cout, r.cin}, PK_RAW_F32, r.w);
                e.add_param(p + "bias", {r.cout}, PK_RAW_F32, r.b);
                break;
            case M_CONV_IN:
            case M_CONV_OUT:
                r.w = e.alloc((int64_t)r.cout * r.cin * 9 * 4);
                r.b = e.alloc(r.cout * 4);
                e.add_param(p + "weight", {r.cout, r.cin, 3, 3}, PK_CONV3_TAP_F32, r.w);
                e.add_param(p + "bias", {r.cout}, PK_RAW_F32, r.b);
                if (r.kind == M_CONV_IN) {    // tensor-core copy for the 64-channel hi/lo operand (pack_input64)
                    r.w_tc = e.alloc((int64_t)r.cout * 9 * 64 * 2);
                    e.add_param(p + "weight", {r.cout, r.cin, 3, 3}, PK_CONV3_K_BF16_HILO64, r.w_tc, 9 * 64, 0);
                }
                if (r.kind == M_CONV_OUT) {   // tensor-core copy: bf16 K-major, 16 rows of which the first 4 are real
                    r.w_tc = e.alloc((int64_t)16 * 9 * r.cin * 2);
                    e.add_param(p + "weight", {r.cout, r.cin, 3, 3}, PK_CONV3_K_BF16, r.w_tc, 9 * (int64_t)r.cin, 0);
                }
                break;
            case M_GN:
                r.gn_g = e.alloc(r.cin * 4);
                r.gn_b = e.alloc(r.cin * 4);
                e.add_param(p + "weight", {r.cin}, PK_RAW_F32, r.gn_g);
                e.add_param(p + "bias", {r.cin}, PK_RAW_F32, r.gn_b);
                break;
            case M_COMBINE:
                r.w = e.alloc((int64_t)r.cout * 4 * 4);
                r.b = e.alloc(r.cout * 4);
                e.add_param(p + "Conv_0.weight", {r.cout, 4, 1, 1}, PK_RAW_F32, r.w);
                e.add_param(p + "Conv_0.bias", {r.cout}, PK_RAW_F32, r.b);
                break;
            case M_ATTN: {
                const int c = r.cin;
                r.gn_g = e.alloc(c * 4);
                r.gn_b = e.alloc(c * 4);
                r.w = e.alloc((int64_t)3 * c * c * 2);
                r.b = e.alloc(3 * c * 4);
                r.w1 = e.alloc((int64_t)c * c * 2);
                r.b1 = e.alloc(c * 4);
                e.add_param(p + "GroupNorm_0.weight", {c}, PK_RAW_F32, r.gn_g);
                e.add_param(p + "GroupNorm_0.bias", {c}, PK_RAW_F32, r.gn_b);
                for (int j = 0; j < 3; ++j) {
                    e.add_param(p + "NIN_" + std::to_string(j) + ".W", {c, c}, PK_NIN_K_BF16, r.w + (int64_t)j * c * c * 2, c, 0);
                    e.add_param(p + "NIN_" + std::to_string(j) + ".b", {c}, PK_RAW_F32, r.b + (int64_t)j * c * 4);
                }
                e.add_param(p + "NIN_3.W", {c, c}, PK_NIN_K_BF16, r.w1, c, 0);
                e.add_param(p + "NIN_3.b", {c}, PK_RAW_F32, r.b1);
                break;
            }
            case M_RES: {
                const int ci = r.cin, co = r.cout;
                const int64_t k1 = 9 * (int64_t)co + (r.has_c2 ? ci : 0);
                r.gn_g = e.alloc(ci * 4);
                r.gn_b = e.alloc(ci * 4);
                r.w = e.alloc((int64_t)co * 9 * ci * 2);
                r.b = e.alloc(co * 4);
                r.gn1_g = e.alloc(co * 4);
                r.gn1_b = e.alloc(co * 4);
                r.w1 = e.alloc((int64_t)co * k1 * 2);
                r.b1 = e.alloc(co * 4);
                e.add_param(p + "GroupNorm_0.weight", {ci}, PK_RAW_F32, r.gn_g);
                e.add_param(p + "GroupNorm_0.bias", {ci}, PK_RAW_F32, r.gn_b);
                e.add_param(p + "Conv_0.weight", {co, ci, 3, 3}, PK_CONV3_K_BF16, r.w, 9 * (int64_t)ci, 0);
                e.add_param(p + "Conv_0.bias", {co}, PK_RAW_F32, r.b);
                e.add_param(p + "Dense_0.weight", {co, d}, PK_RAW_F32, e.dense_w_off + (int64_t)r.tb_row * d * 4);
                e.add_param(p + "Dense_0.bias", {co}, PK_RAW_F32, e.dense_b_off + (int64_t)r.tb_row * 4);
                e.add_param(p + "GroupNorm_1.weight", {co}, PK_RAW_F32, r.gn1_g);
                e.add_param(p + "GroupNorm_1.bias", {co}, PK_RAW_F32, r.gn1_b);
                e.add_param(p + "Conv_1.weight", {co, co, 3, 3}, PK_CONV3_K_BF16, r.w1, k1, 0);
                e.add_param(p + "Conv_1.bias", {co}, PK_RAW_F32, r.b1);
                if (r.has_c2) {
                    e.add_param(p + "Conv_2.weight", {co, ci, 1, 1}, PK_CONV1_K_BF16, r.w1, k1, 9 * (int64_t)co);
                    e.add_param(p + "Conv_2.bias", {co}, PK_RAW_F32, r.b1, 0, 0, 1);
                }
                break;
            }
        }
    }
    return SNRSE_OK;
}

// ------------------------------------------------------------------------------------------------
// Plan recording helpers.  Each helper creates its output tensors and records its steps with Plan::record; the
// builders turn the steps into launch closures once the buffers are placed.
// ------------------------------------------------------------------------------------------------
const float INV_SQRT2 = 0.70710678118654752440f;
constexpr int MAX_STAT_ENTRIES = 192;   // tensors with GroupNorm statistics per forward (NCSN++ default: ~110)
enum { LK_OTHER = 0, LK_GEMM = 1, LK_GN = 2, LK_FIR = 3, LK_ATTN = 4, LK_THIN = 5, LK_HEAD = 6 };

// The kernel that runs a convolution, chosen once, when the step is recorded.  The steps around a convolution depend on
// it: only the 2-CTA kernel normalises its operand in flight and gathers the GroupNorm sums of its output.
enum ConvPath {
    CONV_SIMT,    // fp32 CUDA cores
    CONV_HALO2,   // 2-CTA (cta_group::2) tcgen05 halo kernel
    CONV_GEMM,    // single-CTA tcgen05 implicit GEMM
};
// Convolution of an H x W operand with `taps` taps (9: 3x3, 1: 1x1) to n_rows output channels:
//   - cross-check plans (flags bit1): CUDA cores everywhere; the input convolution reads the fp32 input (conv_in4)
//   - the C -> 4 output head (n_rows 4): the 2-CTA kernel with a 16-row weight tile where the map fits its tiles,
//     CUDA cores (conv_out4) otherwise
//   - every other convolution, the input convolution on its 64-channel hi/lo operand included: the 2-CTA kernel where
//     it is eligible, the single-CTA implicit GEMM otherwise
ConvPath conv_path(const Plan& P, int H, int W, int taps, int n_rows) {
    if (P.cross_check) return CONV_SIMT;
    if (n_rows == 4) return conv_halo2_fits(H, W) ? CONV_HALO2 : CONV_SIMT;
    return conv_halo2_eligible(H, W, taps, n_rows) ? CONV_HALO2 : CONV_GEMM;
}

// out = (conv(x) [+ conv1x1(shortcut)] + bias + time-embedding bias [+ res]) * scale; ids < 0 and offsets < 0 are absent
struct Conv {
    int x = -1;           // operand
    int taps = 9;         // taps of x: 9 (3x3, padding 1) or 1
    int shortcut = -1;    // 1x1 operand appended along K (Conv_2 of a residual block)
    int64_t w = -1;       // blob offset of the bf16 K-major weights [n_rows][taps * C(x) + C(shortcut)]
    int n_rows = 0;       // output channels
    int64_t bias = -1;    // blob offset of the fp32 bias
    int tb_row = -1;      // first row of this layer in the time-embedding bias block t_tb
    int res = -1;         // identity residual
    float scale = 1.0f;
    int out = -1;
    // channel count the ALGORITHM contracts over when x is a zero-padded copy (the 4-channel network input enters as a
    // 64-channel hi/lo tile): FLOPs and bytes are booked at algo_cin, not at the padded width
    int algo_cin = 0;
    bool norm = false;    // x is normalised in flight: GroupNorm + SiLU with the scale/shift in t_scsh
};

int dbg_path(ConvPath path) { return path == CONV_HALO2 ? 0 : path == CONV_SIMT ? 1 : 2; }

int rec_conv(Plan& P, const Conv& c) {
    const ConvPath path = conv_path(P, P.tens[c.x].H, P.tens[c.x].W, c.taps, c.n_rows);
    int st = -1;
    if (path == CONV_HALO2) {   // the epilogue also accumulates the GroupNorm sums of `out`
        st = P.n_stat_entries++;
        P.stats_of[c.out] = st;
    }
    P.convs.push_back({c.x, c.taps, c.shortcut, c.res, c.out, c.n_rows, dbg_path(path), c.norm, st >= 0, c.tb_row >= 0,
                       c.bias >= 0, false, false, c.scale});
    P.record({c.x, c.norm ? P.t_scsh : -1, c.shortcut, c.res, c.out, c.tb_row >= 0 ? P.t_tb : -1}, [=](Plan& p) -> int {
        Engine& e = *p.eng;
        ActView va0 = p.view(c.x), va1, vres, vout = p.view(c.out);
        if (c.shortcut >= 0) va1 = p.view(c.shortcut);
        if (c.res >= 0) vres = p.view(c.res);
        const float* bias = c.bias >= 0 ? e.wf(c.bias) : nullptr;
        const float* tb = c.tb_row >= 0 ? p.fptr(p.t_tb) + c.tb_row : nullptr;
        const int tb_stride = e.dense_rows;
        const double px = (double)va0.B * va0.H * va0.W;
        const int c1 = c.shortcut >= 0 ? va1.C : 0;
        if (path == CONV_SIMT) {
            const int64_t ktot = (int64_t)c.taps * va0.C + c1;
            for (int n0 = 0; n0 < c.n_rows; n0 += 256) {
                const int nn = std::min(256, c.n_rows - n0);
                const bf16* w = e.wb(c.w) + (int64_t)n0 * ktot;
                ActView r2 = vres;
                if (c.res >= 0) r2.ptr += n0;
                p.add(LK_GEMM, 2.0 * px * nn * (double)ktot, 0.0, [=](cudaStream_t s) {
                    return conv_simt_launch(&va0, c.taps, c.shortcut >= 0 ? &va1 : nullptr, w, nn,
                                            bias ? bias + n0 : nullptr, tb ? tb + n0 : nullptr, tb_stride,
                                            c.res >= 0 ? &r2 : nullptr, c.scale, vout.ptr + n0, vout.ld, s);
                });
            }
            return SNRSE_OK;
        }
        const double c0 = c.algo_cin > 0 ? c.algo_cin : va0.C;
        const double kt = (double)c.taps * c0 + c1;
        // algorithmic bytes: each operand / result once (bf16), weights once
        const double by = 2.0 * (px * (c0 + c1 + c.n_rows + (c.res >= 0 ? c.n_rows : 0)) + kt * c.n_rows);
        const ActView* a1 = c.shortcut >= 0 ? &va1 : nullptr;
        const ActView* res = c.res >= 0 ? &vres : nullptr;
        if (path == CONV_HALO2) {
            ConvHaloPlan hp;
            SNRSE_TRY(conv_halo2_make_plan(&hp, &va0, a1, e.wb(c.w), c.n_rows, bias, tb, tb_stride, res, c.scale,
                                           vout.ptr, vout.ld, c.norm ? p.fptr(p.t_scsh) : nullptr, p.stat_ptr(st)));
            p.add(LK_GEMM, 2.0 * px * c.n_rows * kt, by, [hp](cudaStream_t s) { return conv_halo2_launch(&hp, s); });
            return SNRSE_OK;
        }
        ConvGemmPlan g;
        SNRSE_TRY(conv_gemm_make_plan(&g, &va0, c.taps, a1, e.wb(c.w), c.n_rows, 0, 0, bias, tb, tb_stride, res, c.scale,
                                      vout.ptr, vout.ld, 0));
        p.add(LK_GEMM, 2.0 * px * c.n_rows * kt, by, [g](cudaStream_t s) { return conv_gemm_launch(&g, s); });
        return SNRSE_OK;
    });
    return c.out;
}

// Sums of tensor x for GroupNorm: accumulated by its writer when that was the 2-CTA convolution, otherwise by one
// stand-alone pass (cached: skip tensors are normalised twice, in the down path and inside a concatenation).
int get_stats(Plan& P, int x) {
    auto it = P.stats_of.find(x);
    if (it != P.stats_of.end()) return it->second;
    const int st = P.n_stat_entries++;
    P.stats_of[x] = st;
    P.record({x}, [=](Plan& p) -> int {
        const ActView vx = p.view(x);
        unsigned long long* dst = p.stat_ptr(st);
        const double el = (double)vx.B * vx.H * vx.W * vx.C;
        p.add(LK_GN, 0.0, 2.0 * el, [=](cudaStream_t s) { return gn_stats_launch(&vx, dst, s); });
        return SNRSE_OK;
    });
    return st;
}

// scale/shift of GroupNorm(x) into t_scsh; x may be a concatenation whose halves carry their own statistics
void rec_gn_finalize(Plan& P, int x, int64_t g_off, int64_t b_off) {
    int s0, s1 = -1, u0, u1 = 0;
    auto cc = P.cat_children.find(x);
    if (cc != P.cat_children.end()) {
        s0 = get_stats(P, cc->second.first);
        s1 = get_stats(P, cc->second.second);
        u0 = P.tens[cc->second.first].C / 4;
        u1 = P.tens[cc->second.second].C / 4;
    } else {
        s0 = get_stats(P, x);
        u0 = P.tens[x].C / 4;
    }
    const LT tx = P.tens[x];
    P.record({P.t_scsh}, [=](Plan& p) -> int {
        Engine& e = *p.eng;
        const unsigned long long* a0 = p.stat_ptr(s0);
        const unsigned long long* a1 = s1 >= 0 ? p.stat_ptr(s1) : nullptr;
        float* scsh = p.fptr(p.t_scsh);
        const float* gamma = e.wf(g_off);
        const float* beta = e.wf(b_off);
        const int64_t cnt = (int64_t)tx.H * tx.W * (tx.C / 32);
        const int B = tx.B;
        p.add(LK_GN, 0.0, 0.0, [=](cudaStream_t s) {
            return gn_finalize_launch(a0, u0, a1, u1, B, cnt, gamma, beta, 1e-6f, scsh, s);
        });
        return SNRSE_OK;
    });
}

// GroupNorm (+SiLU) as its own pass -> new dense tensor
int rec_gn(Plan& P, int x, int64_t g_off, int64_t b_off, int silu) {
    rec_gn_finalize(P, x, g_off, b_off);
    const LT tx = P.tens[x];
    const int out = P.new_t(tx.B, tx.H, tx.W, tx.C, 2);
    P.record({x, out, P.t_scsh}, [=](Plan& p) -> int {
        const ActView vx = p.view(x), vo = p.view(out);
        float* scsh = p.fptr(p.t_scsh);
        const double el = (double)vx.B * vx.H * vx.W * vx.C;
        p.add(LK_GN, 0.0, 2.0 * el * 2, [=](cudaStream_t s) { return gn_apply_launch(&vx, scsh, silu, &vo, s); });
        return SNRSE_OK;
    });
    return out;
}

// GroupNorm + SiLU of x for the convolution that reads it: in flight (scale/shift into t_scsh, x stays the operand),
// or as a pass of its own whose output is the operand
int rec_gn_silu_operand(Plan& P, int x, int64_t g_off, int64_t b_off, bool in_flight) {
    if (!in_flight) return rec_gn(P, x, g_off, b_off, 1);
    rec_gn_finalize(P, x, g_off, b_off);
    return x;
}

// a = FIR(silu(GroupNorm(x))) and xs = FIR(x) from ONE pass over x (scale/shift currently in t_scsh)
void rec_fir_dual(Plan& P, int x, int up, int* a, int* xs) {
    const LT tx = P.tens[x];
    const int on = up ? P.new_t(tx.B, tx.H * 2, tx.W * 2, tx.C, 2) : P.new_t(tx.B, tx.H / 2, tx.W / 2, tx.C, 2);
    const int orw = up ? P.new_t(tx.B, tx.H * 2, tx.W * 2, tx.C, 2) : P.new_t(tx.B, tx.H / 2, tx.W / 2, tx.C, 2);
    P.record({x, on, orw, P.t_scsh}, [=](Plan& p) -> int {
        const ActView vx = p.view(x), vn = p.view(on), vr = p.view(orw);
        const float* scsh = p.fptr(p.t_scsh);
        const double el = (double)vx.B * vx.H * vx.W * vx.C + 2.0 * vn.B * vn.H * vn.W * vn.C;
        p.add(LK_FIR, 0.0, 2.0 * el, [=](cudaStream_t s) { return fir_dual_launch(&vx, &vn, &vr, up, scsh, s); });
        return SNRSE_OK;
    });
    *a = on;
    *xs = orw;
}

int rec_resblock(Plan& P, const Mod& m, int x) {
    // GroupNorm_0 + SiLU (+ FIR resampling of both branches) + Conv_0 + Dense_0(temb)
    Conv c0{.w = m.w, .n_rows = m.cout, .bias = m.b, .tb_row = m.tb_row};
    int xs = x;
    if (m.up || m.down) {
        // one dual-output FIR launch over x produces both branches; every row segment is staged in shared memory once,
        // raw and normalised, so x comes from DRAM once instead of three times and SiLU is evaluated once per element
        rec_gn_finalize(P, x, m.gn_g, m.gn_b);
        rec_fir_dual(P, x, m.up ? 1 : 0, &c0.x, &xs);
    } else {
        c0.norm = conv_path(P, P.tens[x].H, P.tens[x].W, 9, m.cout) == CONV_HALO2;
        c0.x = rec_gn_silu_operand(P, x, m.gn_g, m.gn_b, c0.norm);
    }
    const LT ta = P.tens[c0.x];
    c0.out = P.new_t(ta.B, ta.H, ta.W, m.cout, 2);
    const int h = rec_conv(P, c0);
    // GroupNorm_1 + SiLU + Conv_1 (+ Conv_2 shortcut or identity residual), / sqrt(2)
    Conv c1{.w = m.w1, .n_rows = m.cout, .bias = m.b1, .scale = INV_SQRT2};
    c1.norm = conv_path(P, P.tens[h].H, P.tens[h].W, 9, m.cout) == CONV_HALO2;
    c1.x = rec_gn_silu_operand(P, h, m.gn1_g, m.gn1_b, c1.norm);
    if (m.has_c2) c1.shortcut = xs;
    else c1.res = xs;
    c1.out = P.new_t(ta.B, ta.H, ta.W, m.cout, 2);
    return rec_conv(P, c1);
}

int rec_attn(Plan& P, const Mod& m, int x) {
    const LT tx = P.tens[x];
    const int c = m.cin, n = tx.H * tx.W;
    const int a = rec_gn(P, x, m.gn_g, m.gn_b, 0);
    const int qkv = P.new_t(tx.B, tx.H, tx.W, 3 * c, 2);
    rec_conv(P, {.x = a, .taps = 1, .w = m.w, .n_rows = 3 * c, .bias = m.b, .out = qkv});
    const int sc = P.new_t(1, 1, 1, (int)((attention_workspace_bytes(tx.B, n, c) + 3) / 4), 4);   // scores | probabilities | V^T
    const int o = P.new_t(tx.B, tx.H, tx.W, c, 2);
    P.record({qkv, sc, o}, [=](Plan& p) -> int {
        const ActView vqkv = p.view(qkv), vo = p.view(o);
        ActView q = vqkv, k = vqkv, v = vqkv;
        q.C = k.C = v.C = c;
        k.ptr += c;
        v.ptr += 2 * c;
        float* scores = p.fptr(sc);
        const double nn = (double)q.H * q.W;
        const int tc = p.cross_check ? 0 : 1;   // cross-check mode keeps the fp32 CUDA-core kernels
        p.add(LK_ATTN, 4.0 * q.B * nn * nn * c, 2.0 * q.B * nn * c * 4, [=](cudaStream_t s) { return attention_launch(&q, &k, &v, scores, &vo, s, tc); });
        return SNRSE_OK;
    });
    const int out = P.new_t(tx.B, tx.H, tx.W, c, 2);
    return rec_conv(P, {.x = o, .taps = 1, .w = m.w1, .n_rows = c, .bias = m.b1, .res = x, .scale = INV_SQRT2, .out = out});
}

// input packing + time embedding (+ the bf16 hi/lo operand x64 of the tensor-core input convolution, when x64 >= 0)
void rec_pack_temb(Plan& P, int x64) {
    P.record({P.t_x4, P.t_tb, P.t_tscr, x64}, [=](Plan& p) -> int {
        Engine& e = *p.eng;
        Plan* pp = &p;
        float* x4 = p.fptr(p.t_x4);
        float* tb = p.fptr(p.t_tb);
        float* scr = p.fptr(p.t_tscr);
        bf16* x64p = x64 >= 0 ? p.view(x64).ptr : nullptr;
        const int64_t n = (int64_t)p.F * p.T;
        const Mod mf = e.mods[0], m1 = e.mods[1], m2 = e.mods[2];
        unsigned long long* stats0 = p.stat_ptr(0);
        const size_t stats_bytes = (size_t)p.n_stat_entries * p.B * 256 * 8;
        p.add(LK_HEAD, 0.0, (double)p.B * n * (32 + (x64p ? 128 : 0)), [=, &e](cudaStream_t s) {
            SNRSE_CUDA(cudaMemsetAsync(stats0, 0, stats_bytes, s));   // GroupNorm sums are accumulated with atomics
            if (x64p) SNRSE_TRY(pack_input64_launch(pp->x_ptr, pp->y_ptr, x4, x64p, pp->B, n, s));
            else SNRSE_TRY(pack_input_launch(pp->x_ptr, pp->y_ptr, x4, pp->B, n, s));
            return temb_launch(pp->t_ptr, pp->B, e.nf, e.wf(mf.w), e.wf(m1.w), e.wf(m1.b), e.wf(m2.w), e.wf(m2.b),
                               e.wf(e.dense_w_off), e.wf(e.dense_b_off), e.dense_rows, scr, tb, s);
        });
        return SNRSE_OK;
    });
}

// input conv 4 -> nf (ncsnpp.py:285): tensor cores on the 64-channel hi/lo operand x64, or fp32 CUDA cores on x4
int rec_conv_in(Plan& P, const Mod& m, int x64) {
    const int out = P.new_t(P.B, P.F, P.T, m.cout, 2);
    if (x64 >= 0) return rec_conv(P, {.x = x64, .w = m.w_tc, .n_rows = m.cout, .bias = m.b, .out = out, .algo_cin = 4});
    P.record({P.t_x4, out}, [=](Plan& p) -> int {
        Engine& e = *p.eng;
        const ActView vo = p.view(out);
        const float* x4 = p.fptr(p.t_x4);
        const double px = (double)vo.B * vo.H * vo.W;
        p.add(LK_THIN, 2.0 * px * 36 * vo.C, px * (16 + 2.0 * vo.C), [=, &e](cudaStream_t s) { return conv_in4_launch(x4, e.wf(m.w), e.wf(m.b), &vo, s); });
        return SNRSE_OK;
    });
    return out;
}

// input pyramid: FIR-downsample the 4-channel input *pyr, 1x1 conv 4->C, add to h (ncsnpp.py:310-311); *pyr becomes
// the downsampled level
int rec_combine(Plan& P, const Mod& m, int h, int* pyr) {
    const int src = *pyr, ih = P.tens[src].H, iw = P.tens[src].W;
    const int np = P.new_t(P.B, ih / 2, iw / 2, 4, 4);
    const int out = P.new_t(P.B, ih / 2, iw / 2, m.cout, 2);
    P.record({src, np, h, out}, [=](Plan& p) -> int {
        Engine& e = *p.eng;
        const float* sp = p.fptr(src);
        float* dp = p.fptr(np);
        const ActView vh = p.view(h), vo = p.view(out);
        const double px = (double)vh.B * vh.H * vh.W;
        p.add(LK_THIN, 2.0 * px * 4 * vh.C, px * (4.0 * vh.C + 16 + 64), [=, &e](cudaStream_t s) {
            SNRSE_TRY(fir_down2_f4_launch(sp, dp, vh.B, ih, iw, s));
            return combine4_launch(dp, &vh, e.wf(m.w), e.wf(m.b), &vo, s);
        });
        return SNRSE_OK;
    });
    *pyr = np;
    return out;
}

// GroupNorm + SiLU + conv3x3 C -> 4, added to the FIR-upsampled output pyramid prev (ncsnpp.py:348-366); returns the
// new pyramid level.  On the 2-CTA tensor-core kernel with the normalisation in flight when the map is large enough,
// CUDA cores otherwise.
int rec_conv_out(Plan& P, const Mod& mg, const Mod& mc, int h, int prev) {
    const LT th = P.tens[h];
    const bool tc = conv_path(P, th.H, th.W, 9, 4) == CONV_HALO2;
    const int a = rec_gn_silu_operand(P, h, mg.gn_g, mg.gn_b, tc);
    const int np = P.new_t(th.B, th.H, th.W, 4, 4);
    const int up = prev >= 0 ? P.new_t(th.B, th.H, th.W, 4, 4) : -1;
    P.convs.push_back({a, 9, -1, -1, np, 4, dbg_path(tc ? CONV_HALO2 : CONV_SIMT), tc, false, false, true, true, prev >= 0,
                       1.0f});
    P.record({a, np, tc ? P.t_scsh : -1, prev, up}, [=](Plan& p) -> int {
        Engine& e = *p.eng;
        const ActView va = p.view(a);
        float* dst = p.fptr(np);
        float* upp = up >= 0 ? p.fptr(up) : nullptr;
        const float* pv = prev >= 0 ? p.fptr(prev) : nullptr;
        const double px = (double)va.B * va.H * va.W;
        if (tc) {
            ConvHaloPlan hp;
            SNRSE_TRY(conv_halo2_make_plan_out4(&hp, &va, e.wb(mc.w_tc), e.wf(mc.b), upp, dst, p.fptr(p.t_scsh)));
            p.add(LK_THIN, 2.0 * px * 36 * va.C, px * (2.0 * va.C + 16 + (pv ? 20 : 0)), [=](cudaStream_t s) {
                if (pv) SNRSE_TRY(fir_up2_f4_launch(pv, upp, va.B, va.H / 2, va.W / 2, s));
                return conv_halo2_launch(&hp, s);
            });
            return SNRSE_OK;
        }
        p.add(LK_THIN, 2.0 * px * 36 * va.C, px * (2.0 * va.C + 16 + (pv ? 20 : 0)), [=, &e](cudaStream_t s) {
            if (pv) SNRSE_TRY(fir_up2_f4_launch(pv, upp, va.B, va.H / 2, va.W / 2, s));
            return conv_out4_launch(&va, e.wf(mc.w), e.wf(mc.b), upp, dst, s);
        });
        return SNRSE_OK;
    });
    return np;
}

// head: h / t, 1x1 conv 4->2, preconditioning (ncsnpp.py:398-403, model.py:488,537-541)
void rec_final(Plan& P, int pyr) {
    P.record({pyr}, [=](Plan& p) -> int {
        Engine& e = *p.eng;
        Plan* pp = &p;
        const float* pf = p.fptr(pyr);
        const int64_t n = (int64_t)p.F * p.T;
        p.add(LK_HEAD, 0.0, (double)p.B * n * 32, [=, &e](cudaStream_t s) {
            return final_launch(pf, pp->t_ptr, e.wf(e.out_w_off), e.wf(e.out_b_off), pp->x_ptr, pp->out_ptr, pp->B, n,
                                pp->mode, s);
        });
        return SNRSE_OK;
    });
}

int record_plan(Plan& P) {
    Engine& e = *P.eng;
    const int B = P.B, F = P.F, T = P.T, L = e.n_levels, nf = e.nf;
    P.t_x4 = P.new_t(B, F, T, 4, 4);
    P.t_tb = P.new_t(B, 1, 1, e.dense_rows, 4);
    P.t_tscr = P.new_t(B, 1, 1, 10 * nf, 4);   // act(temb) [4nf] | Fourier features [2nf] | hidden [4nf] per sample
    P.t_stats = P.new_t(B, 1, 1, MAX_STAT_ENTRIES * 512, 4);   // statistics arena: entries of [B][128 units][2] x 8 bytes
    P.t_scsh = P.new_t(B, 1, 1, 2 * 512, 4);
    const int persistent[] = {P.t_x4, P.t_tb, P.t_tscr, P.t_stats, P.t_scsh};
    // the tensor-core input convolution reads a 64-channel bf16 hi/lo copy of the input, written by the input packing
    const int x64 = conv_path(P, F, T, 9, nf) == CONV_SIMT ? -1 : P.new_t(B, F, T, 64, 2);
    rec_pack_temb(P, x64);   // modules 0-2: Fourier embedding and the two time-embedding layers
    size_t mi = 3;
    auto tap = [&](int t) {   // t is the output of module mi: keep it as the module's activation tap
        P.taps[(int)mi++] = t;
        return t;
    };
    int h = tap(rec_conv_in(P, e.mods[mi], x64));
    std::vector<int> hs{h};
    int ipyr = P.t_x4;
    for (int lv = 0; lv < L; ++lv) {
        for (int b = 0; b < e.num_res_blocks; ++b) {
            h = tap(rec_resblock(P, e.mods[mi], hs.back()));
            if (in_list(e.attn_res, P.tens[h].H)) h = tap(rec_attn(P, e.mods[mi], h));
            hs.push_back(h);
        }
        if (lv != L - 1) {
            h = tap(rec_resblock(P, e.mods[mi], hs.back()));
            h = tap(rec_combine(P, e.mods[mi], h, &ipyr));
            hs.push_back(h);
        }
    }
    h = tap(rec_resblock(P, e.mods[mi], hs.back()));
    h = tap(rec_attn(P, e.mods[mi], h));
    h = tap(rec_resblock(P, e.mods[mi], h));
    int pyr = -1;
    for (int lv = L - 1; lv >= 0; --lv) {
        for (int b = 0; b < e.num_res_blocks + 1; ++b) {
            const int cat = P.concat(h, hs.back());
            hs.pop_back();
            h = tap(rec_resblock(P, e.mods[mi], cat));
        }
        if (in_list(e.attn_res, P.tens[h].H)) h = tap(rec_attn(P, e.mods[mi], h));
        const Mod& gn = e.mods[mi++];   // the head's GroupNorm has no tap of its own
        pyr = tap(rec_conv_out(P, gn, e.mods[mi], h, pyr));
        if (lv != 0) h = tap(rec_resblock(P, e.mods[mi], h));
    }
    if (P.n_stat_entries > MAX_STAT_ENTRIES) {
        snrse_set_error("internal: %d GroupNorm statistics entries exceed the arena (%d)", P.n_stat_entries, MAX_STAT_ENTRIES);
        return SNRSE_ERR_STATE;
    }
    if (!hs.empty() || mi != e.mods.size()) {
        snrse_set_error("internal: plan/topology mismatch (mi=%d of %d)", (int)mi, (int)e.mods.size());
        return SNRSE_ERR_STATE;
    }
    rec_final(P, pyr);
    for (int id : persistent) { P.tens[id].first = 0; P.tens[id].last = 1 << 29; }
    if (P.flags & 1)
        for (auto& t : P.tens) t.last = 1 << 29;  // debug: keep every tensor alive (activation taps stay readable)
    // --- place root tensors: first-fit over lifetime intervals
    std::vector<int> roots;
    for (int i = 0; i < (int)P.tens.size(); ++i)
        if (P.tens[i].parent < 0 && P.tens[i].last >= 0) roots.push_back(i);
    std::sort(roots.begin(), roots.end(), [&](int a, int b) {
        if (P.tens[a].first != P.tens[b].first) return P.tens[a].first < P.tens[b].first;
        return P.tens[a].bytes > P.tens[b].bytes;
    });
    std::vector<int> placed;
    int64_t top = 0;
    for (int id : roots) {
        LT& t = P.tens[id];
        const int64_t sz = (t.bytes + 1023) / 1024 * 1024;
        std::vector<std::pair<int64_t, int64_t>> busy;
        for (int o : placed) {
            const LT& u = P.tens[o];
            if (u.last < t.first || u.first > t.last) continue;
            busy.push_back({u.off, u.off + (u.bytes + 1023) / 1024 * 1024});
        }
        std::sort(busy.begin(), busy.end());
        int64_t off = 0;
        for (auto& iv : busy) {
            if (off + sz <= iv.first) break;
            off = std::max(off, iv.second);
        }
        t.off = off;
        top = std::max(top, off + sz);
        placed.push_back(id);
    }
    P.ws_bytes = top + 1024;
    return SNRSE_OK;
}

__global__ void tap_bf16_kernel(const bf16* __restrict__ x, int ld, int C, int64_t hw, float* __restrict__ out, int64_t total) {
    pdl_sync();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int64_t p = i % hw;
    const int64_t bc = i / hw;
    const int c = (int)(bc % C);
    const int64_t b = bc / C;
    out[i] = __bfloat162float(x[(b * hw + p) * ld + c]);
}
__global__ void tap_f32_kernel(const float* __restrict__ x, int C, int64_t hw, float* __restrict__ out, int64_t total) {
    pdl_sync();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int64_t p = i % hw;
    const int64_t bc = i / hw;
    const int c = (int)(bc % C);
    const int64_t b = bc / C;
    out[i] = x[(b * hw + p) * C + c];
}

// F and T positive multiples of 2^(levels-1), F the image size the attention placement was built for, known flags
bool plan_args_ok(const Engine* e, int B, int F, int T, int flags) {
    if (flags & ~3) {
        snrse_set_error("plan: unknown flags 0x%x (bit0: keep every activation, bit1: CUDA-core cross-check)", flags);
        return false;
    }
    if (!e || B < 1 || F < 1 || T < 1 || (F % (1 << (e->n_levels - 1))) || (T % (1 << (e->n_levels - 1)))) {
        snrse_set_error("plan: F and T must be positive multiples of 2^(levels-1) (got B=%d F=%d T=%d)", B, F, T);
        return false;
    }
    if (F != e->image_size) {
        snrse_set_error("plan: F=%d differs from the image_size=%d the attention placement was built for", F, e->image_size);
        return false;
    }
    return true;
}

// One row of snrse_ncsnpp_dbg_convs (snrse_conv_row of include/snrse_b200_plans.h mirrors this struct)
struct ConvRow {
    int path, out4, B, H, W;
    int c0, ld0, off0, c1, ld1, off1, res, ld_res, off_res, ld_out, off_out;
    int taps, n, norm, bias, tbias, tb_stride, stats, addend;
    float scale;
    ConvPlanFields plan;
};

Plan* find_plan(Engine* e, int B, int F, int T) {
    auto it = e->plans.find(std::make_tuple(B, F, T));
    return it == e->plans.end() ? nullptr : it->second;
}

}  // namespace

// ================================================================================================
// C-ABI (declared in include/snrse_b200.h)
// ================================================================================================
extern "C" {

int snrse_ncsnpp_create(void** handle, int nf, const int* ch_mult, int n_levels, int num_res_blocks,
                        const int* attn_resolutions, int n_attn, int image_size) {
    SNRSE_CHECK_ARG(handle && ch_mult && n_levels >= 1 && n_levels <= 8, "ncsnpp_create: bad arguments");
    SNRSE_CHECK_ARG(nf == 128, "ncsnpp_create: nf must be 128 (GroupNorm/implicit-GEMM kernels assume 32 groups, C %% 128 == 0)");
    Engine* e = new Engine();
    e->nf = nf;
    e->n_levels = n_levels;
    e->num_res_blocks = num_res_blocks;
    e->image_size = image_size;
    e->ch_mult.assign(ch_mult, ch_mult + n_levels);
    if (attn_resolutions) e->attn_res.assign(attn_resolutions, attn_resolutions + n_attn);
    const int rc = build_topology(*e, image_size);
    if (rc != SNRSE_OK) {
        delete e;
        return rc;
    }
    *handle = e;
    return SNRSE_OK;
}

void snrse_ncsnpp_destroy(void* handle) {
    Engine* e = static_cast<Engine*>(handle);
    if (!e) return;
    for (auto& kv : e->plans) delete kv.second;
    delete e;
}

int snrse_ncsnpp_num_modules(void* handle) { return (int)static_cast<Engine*>(handle)->mods.size(); }
int snrse_ncsnpp_num_params(void* handle) { return (int)static_cast<Engine*>(handle)->params.size(); }
int64_t snrse_ncsnpp_weight_bytes(void* handle) { return static_cast<Engine*>(handle)->blob_bytes; }

int snrse_ncsnpp_param_info(void* handle, int i, char* name, int name_cap, int* kind, int64_t* offset,
                            int64_t* row_stride, int64_t* k_offset, int* accumulate) {
    Engine* e = static_cast<Engine*>(handle);
    SNRSE_CHECK_ARG(e && i >= 0 && i < (int)e->params.size(), "param_info: index out of range");
    const Param& p = e->params[i];
    SNRSE_CHECK_ARG((int)p.name.size() + 1 <= name_cap, "param_info: name buffer too small");
    memcpy(name, p.name.c_str(), p.name.size() + 1);
    *kind = p.kind;
    *offset = p.offset;
    *row_stride = p.row_stride;
    *k_offset = p.k_offset;
    *accumulate = p.accumulate;
    return SNRSE_OK;
}

int snrse_ncsnpp_param_shape(void* handle, int i, int64_t* dims, int* ndim) {
    Engine* e = static_cast<Engine*>(handle);
    SNRSE_CHECK_ARG(e && i >= 0 && i < (int)e->params.size(), "param_shape: index out of range");
    for (int j = 0; j < 4; ++j) dims[j] = e->params[i].dims[j];
    *ndim = e->params[i].ndim;
    return SNRSE_OK;
}

int snrse_ncsnpp_set_weights(void* handle, const void* device_blob) {
    Engine* e = static_cast<Engine*>(handle);
    SNRSE_CHECK_ARG(e && device_blob, "set_weights: null");
    SNRSE_CHECK_ARG((reinterpret_cast<uintptr_t>(device_blob) & 255) == 0, "set_weights: blob must be 256-byte aligned");
    e->blob = static_cast<const uint8_t*>(device_blob);
    for (auto& kv : e->plans) {  // launch closures captured weight pointers: rebuild lazily
        kv.second->launches.clear();
        kv.second->info.clear();
        kv.second->ws = nullptr;
    }
    return SNRSE_OK;
}

// flags: bit0 = keep every activation alive (debug taps), bit1 = fp32 CUDA-core cross-check path (convolutions,
//        attention and input packing); no other bit is defined
int64_t snrse_ncsnpp_plan_bytes(void* handle, int B, int F, int T, int flags) {
    Engine* e = static_cast<Engine*>(handle);
    if (!plan_args_ok(e, B, F, T, flags)) return -1;
    Plan* p = find_plan(e, B, F, T);
    if (p && p->flags != flags) {
        delete p;
        e->plans.erase(std::make_tuple(B, F, T));
        p = nullptr;
    }
    if (!p) {
        p = new Plan();
        p->eng = e; p->B = B; p->F = F; p->T = T; p->flags = flags;
        p->cross_check = (flags & 2) != 0;
        if (record_plan(*p) != SNRSE_OK) {
            delete p;
            return -1;
        }
        e->plans[std::make_tuple(B, F, T)] = p;
    }
    return p->ws_bytes;
}

int snrse_ncsnpp_plan_bind(void* handle, int B, int F, int T, void* workspace, int64_t bytes) {
    Engine* e = static_cast<Engine*>(handle);
    Plan* p = e ? find_plan(e, B, F, T) : nullptr;
    SNRSE_CHECK_ARG(p, "plan_bind: call snrse_ncsnpp_plan_bytes first");
    SNRSE_CHECK_ARG(e->blob, "plan_bind: weights not set");
    SNRSE_CHECK_ARG(workspace && bytes >= p->ws_bytes, "plan_bind: workspace too small (%lld < %lld)", (long long)bytes,
                    (long long)p->ws_bytes);
    SNRSE_CHECK_ARG((reinterpret_cast<uintptr_t>(workspace) & 1023) == 0, "plan_bind: workspace must be 1024-byte aligned");
    p->ws = static_cast<uint8_t*>(workspace);
    p->launches.clear();
    p->info.clear();
    for (auto& b : p->builders) SNRSE_TRY(b(*p));
    return SNRSE_OK;
}

// x, y, out: complex64 [B, F, T] (torch layout); t: [B] f32 (device).  mode: 0 raw dnn, 1 sebridge precond, 2 -dnn.
int snrse_ncsnpp_forward(void* handle, int B, int F, int T, const void* x, const void* y, const float* t, void* out,
                         int mode, void* stream) {
    Engine* e = static_cast<Engine*>(handle);
    Plan* p = e ? find_plan(e, B, F, T) : nullptr;
    SNRSE_CHECK_ARG(p && p->ws && !p->launches.empty(), "forward: no bound plan for B=%d F=%d T=%d", B, F, T);
    SNRSE_CHECK_ARG(x && y && t && out, "forward: null pointer");
    p->x_ptr = static_cast<const float2*>(x);
    p->y_ptr = static_cast<const float2*>(y);
    p->t_ptr = t;
    p->out_ptr = static_cast<float2*>(out);
    p->mode = mode;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    for (auto& l : p->launches) SNRSE_TRY(l(s));
    return SNRSE_OK;
}

// Eager forward with a CUDA event between launch groups: per group kind (0 other, 1 implicit-GEMM conv,
// 2 GroupNorm+SiLU, 3 FIR, 4 attention core, 5 thin convs, 6 pack/temb/head), algorithmic flops / bytes and
// measured milliseconds on `stream`.  Synchronises the stream (measurement only; not graph-capturable).
int snrse_ncsnpp_profile_forward(void* handle, int B, int F, int T, const void* x, const void* y, const float* t,
                                 void* out, int mode, void* stream, int cap, int* kinds, double* flops, double* bytes,
                                 float* ms, int* n_groups) {
    Engine* e = static_cast<Engine*>(handle);
    Plan* p = e ? find_plan(e, B, F, T) : nullptr;
    SNRSE_CHECK_ARG(p && p->ws && !p->launches.empty(), "profile_forward: no bound plan");
    const int n = (int)p->launches.size();
    SNRSE_CHECK_ARG(cap >= n, "profile_forward: arrays too small (%d groups)", n);
    p->x_ptr = static_cast<const float2*>(x);
    p->y_ptr = static_cast<const float2*>(y);
    p->t_ptr = t;
    p->out_ptr = static_cast<float2*>(out);
    p->mode = mode;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    std::vector<cudaEvent_t> ev(n + 1);
    for (auto& v : ev) SNRSE_CUDA(cudaEventCreate(&v));
    SNRSE_CUDA(cudaEventRecord(ev[0], s));
    for (int i = 0; i < n; ++i) {
        SNRSE_TRY(p->launches[i](s));
        SNRSE_CUDA(cudaEventRecord(ev[i + 1], s));
    }
    SNRSE_CUDA(cudaStreamSynchronize(s));
    for (int i = 0; i < n; ++i) {
        SNRSE_CUDA(cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]));
        kinds[i] = p->info[i].kind;
        flops[i] = p->info[i].flops;
        bytes[i] = p->info[i].bytes;
    }
    for (auto& v : ev) cudaEventDestroy(v);
    *n_groups = n;
    return SNRSE_OK;
}

// Debug: the convolutions of the (B,F,T) plan with these flags, recorded as snrse_ncsnpp_plan_bytes records them but
// into a plan of its own (nothing cached, no weights, no device), with their plan fields for num_sms SMs.
int snrse_ncsnpp_dbg_convs(void* handle, int B, int F, int T, int flags, int num_sms, void* rows, int cap, int* n) {
    Engine* e = static_cast<Engine*>(handle);
    SNRSE_CHECK_ARG(n && num_sms >= 2, "dbg_convs: bad arguments");
    if (!plan_args_ok(e, B, F, T, flags)) return SNRSE_ERR_ARG;
    Plan P;
    P.eng = e; P.B = B; P.F = F; P.T = T; P.flags = flags;
    P.cross_check = (flags & 2) != 0;
    SNRSE_TRY(record_plan(P));
    *n = (int)P.convs.size();
    if (!rows) return SNRSE_OK;
    SNRSE_CHECK_ARG(cap >= *n, "dbg_convs: %d rows do not fit %d", *n, cap);
    ConvRow* out = static_cast<ConvRow*>(rows);
    for (const Plan::ConvRec& c : P.convs) {
        ConvRow r{};
        const LT& x = P.tens[c.x];
        r.path = c.path; r.out4 = c.out4; r.B = x.B; r.H = x.H; r.W = x.W;
        r.c0 = x.C; r.ld0 = P.tens[P.root(c.x)].C; r.off0 = P.chan_off(c.x);
        if (c.shortcut >= 0) {
            r.c1 = P.tens[c.shortcut].C; r.ld1 = P.tens[P.root(c.shortcut)].C; r.off1 = P.chan_off(c.shortcut);
        }
        if (c.res >= 0) {
            r.res = 1; r.ld_res = P.tens[P.root(c.res)].C; r.off_res = P.chan_off(c.res);
        }
        r.ld_out = P.tens[P.root(c.out)].C; r.off_out = P.chan_off(c.out);
        r.taps = c.taps; r.n = c.n_rows; r.norm = c.norm; r.bias = c.bias; r.tbias = c.tbias;
        r.tb_stride = c.tbias ? e->dense_rows : 0;
        r.stats = c.stats; r.addend = c.addend; r.scale = c.scale;
        if (c.path == 0) {
            ConvHaloPlan hp;
            SNRSE_TRY(c.out4 ? conv_halo2_plan_shape_out4(&hp, r.B, r.H, r.W, r.c0, num_sms)
                             : conv_halo2_plan_shape(&hp, r.B, r.H, r.W, r.c0, r.c1, r.n, r.norm, num_sms));
            r.plan = conv_plan_fields(hp);
        } else if (c.path == 2) {
            ConvGemmPlan gp;
            SNRSE_TRY(conv_gemm_plan_shape(&gp, r.B, r.H, r.W, r.taps, r.c0, r.c1, r.n, num_sms));
            r.plan = conv_plan_fields(gp);
        }
        *out++ = r;
    }
    return SNRSE_OK;
}

int snrse_ncsnpp_num_launch_groups(void* handle, int B, int F, int T) {
    Engine* e = static_cast<Engine*>(handle);
    Plan* p = e ? find_plan(e, B, F, T) : nullptr;
    return p ? (int)p->launches.size() : -1;
}

// Debug: copy the output activation of module `module_idx` as fp32 NCHW into `out` (device).  Needs a
// plan made with flags bit0.  dims receives {B, C, H, W}.
int snrse_ncsnpp_read_tap(void* handle, int B, int F, int T, int module_idx, float* out, int64_t cap_elems,
                          int64_t* dims, void* stream) {
    Engine* e = static_cast<Engine*>(handle);
    Plan* p = e ? find_plan(e, B, F, T) : nullptr;
    SNRSE_CHECK_ARG(p && p->ws, "read_tap: no bound plan");
    SNRSE_CHECK_ARG(p->flags & 1, "read_tap: plan was not created with the keep-all flag");
    auto it = p->taps.find(module_idx);
    SNRSE_CHECK_ARG(it != p->taps.end(), "read_tap: module %d has no tap", module_idx);
    const LT& t = p->tens[it->second];
    const int64_t total = (int64_t)t.B * t.C * t.H * t.W;
    dims[0] = t.B; dims[1] = t.C; dims[2] = t.H; dims[3] = t.W;
    SNRSE_CHECK_ARG(cap_elems >= total, "read_tap: output buffer too small");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int64_t hw = (int64_t)t.H * t.W;
    if (t.esize == 2) {
        const ActView v = p->view(it->second);
        snrse_launch(tap_bf16_kernel, dim3((unsigned)cdiv64(total, 256)), dim3(256), 0, s, v.ptr, v.ld, v.C, hw, out, total);
    } else {
        snrse_launch(tap_f32_kernel, dim3((unsigned)cdiv64(total, 256)), dim3(256), 0, s, p->fptr(it->second), t.C, hw, out, total);
    }
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}

}  // extern "C"
