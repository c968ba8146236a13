// FIR x2 resampling with the [1,3,3,1] (x) [1,3,3,1] / 64 kernel, NHWC.
// Replaces `upsample_2d` / `downsample_2d` (sgmse-bbed/sgmse/backbones/ncsnpp_utils/up_or_down_sampling.py:195-257)
// and the reference's own CUDA op `upfirdn2d_kernel` modes 3 and 5
// (ncsnpp_utils/op/upfirdn2d_kernel.cu:107-207,264-283) for exactly the two configurations NCSN++ uses:
//   up  : zero-insert x2, pad (2,1), gain 4  ->  per axis  out[2i]   = (x[i-1] + 3 x[i]) / 4
//                                                           out[2i+1] = (3 x[i] + x[i+1]) / 4
//   down: pad (1,1), keep every 2nd sample   ->  per axis  out[j] = (x[2j-1] + 3 x[2j] + 3 x[2j+1] + x[2j+2]) / 8
// with zeros outside the image.
#include "kernels.h"

namespace {

struct V8 {
    float f[8];
};
__device__ __forceinline__ V8 ld8(const bf16* p) {
    V8 r;
    unpack8(__ldg(reinterpret_cast<const uint4*>(p)), r.f);
    return r;
}

// Both bf16 kernels are separable and walk a band of rows with a sliding window in registers: thread = (column,
// 8-channel chunk); every input row is filtered horizontally once (3 or 4 loads, neighbours shared through L1)
// and reused by the two output rows it contributes to, so the kernels move ~1x the tensor instead of issuing
// 16 (down) / 4 (up) loads per output chunk.  grid = (column blocks, row bands, B).
constexpr int FIR_BAND = 16;   // rows per block (output rows for down, input rows for up)

__device__ __forceinline__ void zero8(float* a) {
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] = 0.f;
}

// raw 16-byte loads of the 4 input columns around output column wo of input row hh (zero outside the image)
__device__ __forceinline__ void load_row_down(const bf16* __restrict__ img, int ld, int H, int W, int hh, int wo, int c0,
                                              uint4* raw) {
    const bool row_ok = hh >= 0 && hh < H;
    const bf16* row = img + (int64_t)(row_ok ? hh : 0) * W * ld + c0;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const int ww = 2 * wo - 1 + t;
        const bool ok = row_ok && ww >= 0 && ww < W;
        raw[t] = ok ? __ldg(reinterpret_cast<const uint4*>(row + (int64_t)ww * ld)) : make_uint4(0, 0, 0, 0);
    }
}
// horizontal [1,3,3,1]/8
__device__ __forceinline__ void hfilt_down(const uint4* raw, float* r) {
    float f0[8], f1[8], f2[8], f3[8];
    unpack8(raw[0], f0);
    unpack8(raw[1], f1);
    unpack8(raw[2], f2);
    unpack8(raw[3], f3);
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = fmaf(0.125f, f3[j], fmaf(0.375f, f2[j], fmaf(0.375f, f1[j], fmaf(0.125f, f0[j], 0.f))));
}

// interior rows / columns: four unconditional 16-byte loads, no masks
__device__ __forceinline__ void load_row_down_fast(const bf16* __restrict__ p, int ld, uint4* raw) {
#pragma unroll
    for (int t = 0; t < 4; ++t) raw[t] = __ldg(reinterpret_cast<const uint4*>(p + (int64_t)t * ld));
}

__device__ __forceinline__ void fir_down2_body(const bf16* __restrict__ x, int ld, int C, int H, int W, bf16* __restrict__ out,
                                               int out_ld, int band) {
    const int tpp = C >> 3, cols = blockDim.x / tpp;
    const int c0 = (threadIdx.x % tpp) * 8;
    const int Ho = H >> 1, Wo = W >> 1;
    const int wo = blockIdx.x * cols + threadIdx.x / tpp;
    if (wo >= Wo) return;
    const int b = blockIdx.z;
    const bf16* img = x + (int64_t)b * H * W * ld;
    const int ho0 = blockIdx.y * band;
    const int ho1 = min(ho0 + band, Ho);
    // columns 2wo-1 .. 2wo+2 all inside the image: rows inside the image need no bounds logic at all
    const bool col_in = wo > 0 && 2 * wo + 2 < W;
    const int64_t rstride = (int64_t)W * ld;
    const bf16* pcol = img + (int64_t)(2 * wo - 1) * ld + c0;   // column 2wo-1 of row 0 (only dereferenced when col_in)
    auto load_row = [&](int hh, uint4* raw) {
        if (col_in && hh >= 0 && hh < H) load_row_down_fast(pcol + hh * rstride, ld, raw);
        else load_row_down(img, ld, H, W, hh, wo, c0, raw);
    };
    float r0[8], r1[8], r2[8], r3[8];   // horizontally filtered rows 2ho-1 .. 2ho+2
    uint4 ra[4], rb[4];
    load_row(2 * ho0 - 1, ra);
    load_row(2 * ho0, rb);
    hfilt_down(ra, r0);
    hfilt_down(rb, r1);
    load_row(2 * ho0 + 1, ra);   // the two new rows of the first output row
    load_row(2 * ho0 + 2, rb);
    bf16* op = out + (((int64_t)b * Ho + ho0) * Wo + wo) * out_ld + c0;
    const int64_t ostride = (int64_t)Wo * out_ld;
    for (int ho = ho0; ho < ho1; ++ho, op += ostride) {
        hfilt_down(ra, r2);
        hfilt_down(rb, r3);
        if (ho + 1 < ho1) {   // next output row's loads are in flight while this one is finished
            load_row(2 * ho + 3, ra);
            load_row(2 * ho + 4, rb);
        }
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = 0.125f * (r0[j] + r3[j]) + 0.375f * (r1[j] + r2[j]);
        *reinterpret_cast<uint4*>(op) = pack8(o);
#pragma unroll
        for (int j = 0; j < 8; ++j) { r0[j] = r2[j]; r1[j] = r3[j]; }
    }
}

// horizontal interpolation of input row hh at input column wi: ea -> output column 2wi, eb -> 2wi+1
__device__ __forceinline__ void hfilt_up(const bf16* __restrict__ img, int ld, int H, int W, int hh, int wi, int c0, float* ea,
                                         float* eb) {
    zero8(ea);
    zero8(eb);
    if (hh < 0 || hh >= H) return;
    const bf16* row = img + (int64_t)hh * W * ld + c0;
    float m[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(row + (int64_t)wi * ld)), m);
#pragma unroll
    for (int j = 0; j < 8; ++j) { ea[j] = 0.75f * m[j]; eb[j] = 0.75f * m[j]; }
    if (wi > 0) {
        float l[8];
        unpack8(__ldg(reinterpret_cast<const uint4*>(row + (int64_t)(wi - 1) * ld)), l);
#pragma unroll
        for (int j = 0; j < 8; ++j) ea[j] = fmaf(0.25f, l[j], ea[j]);
    }
    if (wi + 1 < W) {
        float rr[8];
        unpack8(__ldg(reinterpret_cast<const uint4*>(row + (int64_t)(wi + 1) * ld)), rr);
#pragma unroll
        for (int j = 0; j < 8; ++j) eb[j] = fmaf(0.25f, rr[j], eb[j]);
    }
}

__device__ __forceinline__ void fir_up2_body(const bf16* __restrict__ x, int ld, int C, int H, int W, bf16* __restrict__ out,
                                             int out_ld, int band) {
    const int tpp = C >> 3, cols = blockDim.x / tpp;
    const int c0 = (threadIdx.x % tpp) * 8;
    const int wi = blockIdx.x * cols + threadIdx.x / tpp;
    if (wi >= W) return;
    const int b = blockIdx.z;
    const int Wo = 2 * W;
    const bf16* img = x + (int64_t)b * H * W * ld;
    bf16* oimg = out + (int64_t)b * (2 * H) * Wo * out_ld + c0;
    const int h0 = blockIdx.y * band;
    const int h1 = min(h0 + band, H);
    float pa[8], pb[8], ca[8], cb[8], na[8], nb[8];   // rows hi-1, hi, hi+1 (a: even output column, b: odd)
    hfilt_up(img, ld, H, W, h0 - 1, wi, c0, pa, pb);
    hfilt_up(img, ld, H, W, h0, wi, c0, ca, cb);
    for (int hi = h0; hi < h1; ++hi) {
        hfilt_up(img, ld, H, W, hi + 1, wi, c0, na, nb);
        float o[8];
        bf16* r_even = oimg + ((int64_t)(2 * hi) * Wo + 2 * wi) * out_ld;
        bf16* r_odd = r_even + (int64_t)Wo * out_ld;
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = fmaf(0.25f, pa[j], 0.75f * ca[j]);
        *reinterpret_cast<uint4*>(r_even) = pack8(o);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = fmaf(0.25f, pb[j], 0.75f * cb[j]);
        *reinterpret_cast<uint4*>(r_even + out_ld) = pack8(o);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = fmaf(0.25f, na[j], 0.75f * ca[j]);
        *reinterpret_cast<uint4*>(r_odd) = pack8(o);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = fmaf(0.25f, nb[j], 0.75f * cb[j]);
        *reinterpret_cast<uint4*>(r_odd + out_ld) = pack8(o);
#pragma unroll
        for (int j = 0; j < 8; ++j) { pa[j] = ca[j]; pb[j] = cb[j]; ca[j] = na[j]; cb[j] = nb[j]; }
    }
}

__global__ void __launch_bounds__(256)
fir_down2_kernel(const bf16* __restrict__ x, int ld, int C, int H, int W, bf16* __restrict__ out, int out_ld, int band) {
    pdl_sync();
    fir_down2_body(x, ld, C, H, W, out, out_ld, band);
}
__global__ void __launch_bounds__(256)
fir_up2_kernel(const bf16* __restrict__ x, int ld, int C, int H, int W, bf16* __restrict__ out, int out_ld, int band) {
    pdl_sync();
    fir_up2_body(x, ld, C, H, W, out, out_ld, band);
}

// ---- dual-output variants for the up / down residual blocks (layerspp.py:245-257): the block filters BOTH
// h = silu(GroupNorm(x)) and the raw x with the same FIR.  One launch produces FIR(h) and FIR(x) from ONE pass over x:
// every input row segment of the block (its columns + halo, all channels) is staged in shared memory once, raw and
// normalised (silu(x*scale + shift) rounded to bf16 -- what the separate GroupNorm pass would have stored), and both
// filters read their taps from there.  Rows are staged so that each element is normalised once per block: neighbouring
// output columns share input columns, so normalising the taps as they are loaded would evaluate SiLU 2x (down) / 3x (up)
// per element.  Against the three-pass form (gn_apply: read x, write h; FIR: read h; FIR: read x) the DRAM traffic per
// element of x drops from 3 reads + 1 write (+ outputs) to 1 read (+ outputs).  Same arithmetic and rounding points:
// bit-identical results.

// GroupNorm scale / shift of one 8-channel chunk (per (sample, channel), from gn_finalize)
struct Norm8 {
    float sc[8], sh[8];
};
__device__ __forceinline__ Norm8 load_norm(const float* __restrict__ scsh, int b, int C, int c0) {
    Norm8 n;
    const float4* a = reinterpret_cast<const float4*>(scsh + ((int64_t)b * 2) * C + c0);
    const float4* c = reinterpret_cast<const float4*>(scsh + ((int64_t)b * 2 + 1) * C + c0);
    const float4 a0 = __ldg(a), a1 = __ldg(a + 1), c0v = __ldg(c), c1 = __ldg(c + 1);
    n.sc[0] = a0.x; n.sc[1] = a0.y; n.sc[2] = a0.z; n.sc[3] = a0.w; n.sc[4] = a1.x; n.sc[5] = a1.y; n.sc[6] = a1.z; n.sc[7] = a1.w;
    n.sh[0] = c0v.x; n.sh[1] = c0v.y; n.sh[2] = c0v.z; n.sh[3] = c0v.w; n.sh[4] = c1.x; n.sh[5] = c1.y; n.sh[6] = c1.z; n.sh[7] = c1.w;
    return n;
}
// unpack 8 bf16, normalise + SiLU and round to bf16: the same arithmetic as gn_apply_kernel and its bf16 store
__device__ __forceinline__ void unpack_norm(const uint4& raw, const Norm8& n, float* f) {
    unpack8(raw, f);
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = __bfloat162float(__float2bfloat16(silu_f(fmaf(f[j], n.sc[j], n.sh[j]))));
}

// Staging is split in two so that the global loads of the NEXT rows are in flight while the current rows are filtered:
// fir_stage_load issues up to MAXI 16-byte loads of a row segment into registers (nothing depends on them yet),
// fir_stage_store normalises them and writes the raw and the normalised copy to shared memory.
template <int MAXI>
struct StageRegs {
    uint4 raw[MAXI];
    unsigned ok;      // bit i: item i lies inside the image (others are stored as zeros)
};
template <int MAXI>
__device__ __forceinline__ void fir_stage_load(const bf16* __restrict__ img, int ld, int H, int W, int hh, int wbase, int ncol,
                                               int tpp, int chunk, StageRegs<MAXI>& r) {
    const bool row_ok = hh >= 0 && hh < H;
    const int cstep = blockDim.x / tpp;
    r.ok = 0;
#pragma unroll
    for (int i = 0; i < MAXI; ++i) {
        const int col = threadIdx.x / tpp + i * cstep, ww = wbase + col;
        r.raw[i] = make_uint4(0, 0, 0, 0);
        if (col < ncol && row_ok && ww >= 0 && ww < W) {
            r.raw[i] = __ldg(reinterpret_cast<const uint4*>(img + ((int64_t)hh * W + ww) * ld + chunk * 8));
            r.ok |= 1u << i;
        }
    }
}
template <int MAXI>
__device__ __forceinline__ void fir_stage_store(const StageRegs<MAXI>& r, int ncol, int tpp, int chunk, const Norm8& nm,
                                                uint4* __restrict__ s_raw, uint4* __restrict__ s_nrm) {
    const int cstep = blockDim.x / tpp;
#pragma unroll
    for (int i = 0; i < MAXI; ++i) {
        const int col = threadIdx.x / tpp + i * cstep;
        if (col < ncol) {
            uint4 nr = make_uint4(0, 0, 0, 0);
            if ((r.ok >> i) & 1u) {
                float f[8];
                unpack_norm(r.raw[i], nm, f);
                nr = pack8(f);                     // already bf16 values: exact
            }
            s_raw[col * tpp + chunk] = r.raw[i];
            s_nrm[col * tpp + chunk] = nr;
        }
    }
}
// horizontal [1,3,3,1]/8 over four staged columns (stride tpp); zeros stand for positions outside the image
__device__ __forceinline__ void hfilt_down_s(const uint4* __restrict__ p, int tpp, float* r) {
    float f0[8], f1[8], f2[8], f3[8];
    unpack8(p[0], f0);
    unpack8(p[tpp], f1);
    unpack8(p[2 * tpp], f2);
    unpack8(p[3 * tpp], f3);
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = fmaf(0.125f, f3[j], fmaf(0.375f, f2[j], fmaf(0.375f, f1[j], fmaf(0.125f, f0[j], 0.f))));
}

__global__ void __launch_bounds__(256, 2)
fir_down2_dual_kernel(const bf16* __restrict__ x, int ld, int C, int H, int W, bf16* __restrict__ out_n, int out_n_ld,
                      bf16* __restrict__ out_r, int out_r_ld, int band, const float* __restrict__ scsh) {
    pdl_sync();
    extern __shared__ __align__(16) uint4 fir_sm[];
    const int tpp = C >> 3, cols = blockDim.x / tpp;
    const int chunk = threadIdx.x % tpp, tcol = threadIdx.x / tpp, c0 = chunk * 8;
    const int Ho = H >> 1, Wo = W >> 1;
    const int wo = blockIdx.x * cols + tcol;          // >= Wo: the thread only helps staging
    const int b = blockIdx.z;
    const bf16* img = x + (int64_t)b * H * W * ld;
    const int ho0 = blockIdx.y * band, ho1 = min(ho0 + band, Ho);
    const Norm8 nm = load_norm(scsh, b, C, c0);
    const int ncol = 2 * cols + 2, wbase = 2 * blockIdx.x * cols - 1, rowsz = ncol * tpp;
    // [slot 2][row of the pair 2][raw | normalised][rowsz]
    auto S = [&](int slot, int r, int kind) { return fir_sm + ((slot * 2 + r) * 2 + kind) * rowsz; };
    StageRegs<3> ga, gb;                              // ncol = 2 cols + 2 <= 3 cols for cols >= 2 (checked by the launcher)
    auto load_pair = [&](int hh) {
        fir_stage_load<3>(img, ld, H, W, hh, wbase, ncol, tpp, chunk, ga);
        fir_stage_load<3>(img, ld, H, W, hh + 1, wbase, ncol, tpp, chunk, gb);
    };
    auto store_pair = [&](int slot) {
        fir_stage_store<3>(ga, ncol, tpp, chunk, nm, S(slot, 0, 0), S(slot, 0, 1));
        fir_stage_store<3>(gb, ncol, tpp, chunk, nm, S(slot, 1, 0), S(slot, 1, 1));
    };
    const int my = 2 * tcol * tpp + chunk;            // first of this thread's four staged columns
    load_pair(2 * ho0 - 1);
    store_pair(0);
    load_pair(2 * ho0 + 1);
    store_pair(1);
    __syncthreads();
    float n0[8], n1[8], q0[8], q1[8];                 // horizontally filtered rows 2ho-1, 2ho (normalised / raw)
    hfilt_down_s(S(0, 0, 1) + my, tpp, n0);
    hfilt_down_s(S(0, 1, 1) + my, tpp, n1);
    hfilt_down_s(S(0, 0, 0) + my, tpp, q0);
    hfilt_down_s(S(0, 1, 0) + my, tpp, q1);
    const bool live = wo < Wo;
    bf16* on = out_n + (((int64_t)b * Ho + ho0) * Wo + (live ? wo : 0)) * out_n_ld + c0;
    bf16* orw = out_r + (((int64_t)b * Ho + ho0) * Wo + (live ? wo : 0)) * out_r_ld + c0;
    for (int ho = ho0; ho < ho1; ++ho, on += (int64_t)Wo * out_n_ld, orw += (int64_t)Wo * out_r_ld) {
        const int slot = (ho - ho0 + 1) & 1;          // the pair holding rows 2ho+1, 2ho+2
        __syncthreads();                              // that pair is complete; the other slot is no longer being read
        const bool more = ho + 1 < ho1;               // block-uniform
        if (more) load_pair(2 * ho + 3);              // next pair's loads are in flight while this row is finished
        float t2[8], t3[8], o[8];
        hfilt_down_s(S(slot, 0, 1) + my, tpp, t2);
        hfilt_down_s(S(slot, 1, 1) + my, tpp, t3);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = 0.125f * (n0[j] + t3[j]) + 0.375f * (n1[j] + t2[j]);
        if (live) *reinterpret_cast<uint4*>(on) = pack8(o);
#pragma unroll
        for (int j = 0; j < 8; ++j) { n0[j] = t2[j]; n1[j] = t3[j]; }
        hfilt_down_s(S(slot, 0, 0) + my, tpp, t2);
        hfilt_down_s(S(slot, 1, 0) + my, tpp, t3);
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = 0.125f * (q0[j] + t3[j]) + 0.375f * (q1[j] + t2[j]);
        if (live) *reinterpret_cast<uint4*>(orw) = pack8(o);
#pragma unroll
        for (int j = 0; j < 8; ++j) { q0[j] = t2[j]; q1[j] = t3[j]; }
        if (more) store_pair(slot ^ 1);
    }
}

// horizontal interpolation of a staged row at this thread's column (p: the column left of it): ea -> output column 2wi,
// eb -> 2wi+1; the same operations in the same order as hfilt_up
__device__ __forceinline__ void hfilt_up_s(const uint4* __restrict__ p, int tpp, bool row_ok, bool has_l, bool has_r, float* ea,
                                           float* eb) {
    zero8(ea);
    zero8(eb);
    if (!row_ok) return;
    float m[8];
    unpack8(p[tpp], m);
#pragma unroll
    for (int j = 0; j < 8; ++j) { ea[j] = 0.75f * m[j]; eb[j] = 0.75f * m[j]; }
    if (has_l) {
        float l[8];
        unpack8(p[0], l);
#pragma unroll
        for (int j = 0; j < 8; ++j) ea[j] = fmaf(0.25f, l[j], ea[j]);
    }
    if (has_r) {
        float rr[8];
        unpack8(p[2 * tpp], rr);
#pragma unroll
        for (int j = 0; j < 8; ++j) eb[j] = fmaf(0.25f, rr[j], eb[j]);
    }
}

__global__ void __launch_bounds__(256, 2)
fir_up2_dual_kernel(const bf16* __restrict__ x, int ld, int C, int H, int W, bf16* __restrict__ out_n, int out_n_ld,
                    bf16* __restrict__ out_r, int out_r_ld, int band, const float* __restrict__ scsh) {
    pdl_sync();
    extern __shared__ __align__(16) uint4 fir_sm[];
    const int tpp = C >> 3, cols = blockDim.x / tpp;
    const int chunk = threadIdx.x % tpp, tcol = threadIdx.x / tpp, c0 = chunk * 8;
    const int wi = blockIdx.x * cols + tcol;          // >= W: the thread only helps staging
    const int b = blockIdx.z, Wo = 2 * W;
    const bf16* img = x + (int64_t)b * H * W * ld;
    const int h0 = blockIdx.y * band, h1 = min(h0 + band, H);
    const Norm8 nm = load_norm(scsh, b, C, c0);
    const int ncol = cols + 2, wbase = blockIdx.x * cols - 1, rowsz = ncol * tpp;
    // ring of three rows: row r lives in slot (r - (h0 - 1)) % 3;  [slot 3][raw | normalised][rowsz]
    auto S = [&](int row, int kind) { return fir_sm + (((row - (h0 - 1)) % 3) * 2 + kind) * rowsz; };
    StageRegs<2> gr;                                  // ncol = cols + 2 <= 2 cols for cols >= 2 (checked by the launcher)
    auto stage_load = [&](int row) { fir_stage_load<2>(img, ld, H, W, row, wbase, ncol, tpp, chunk, gr); };
    auto stage_store = [&](int row) { fir_stage_store<2>(gr, ncol, tpp, chunk, nm, S(row, 0), S(row, 1)); };
    auto stage = [&](int row) { stage_load(row); stage_store(row); };
    const int my = tcol * tpp + chunk;                // the column left of this thread's input column
    const bool live = wi < W, has_l = wi > 0, has_r = wi + 1 < W;
    stage(h0 - 1);
    stage(h0);
    stage(h0 + 1);
    __syncthreads();
    float pa[8], pb[8], ca[8], cb[8], qa[8], qb[8], da[8], db[8];   // rows hi-1 / hi, normalised (p, c) and raw (q, d)
    hfilt_up_s(S(h0 - 1, 1) + my, tpp, h0 - 1 >= 0, has_l, has_r, pa, pb);
    hfilt_up_s(S(h0, 1) + my, tpp, true, has_l, has_r, ca, cb);
    hfilt_up_s(S(h0 - 1, 0) + my, tpp, h0 - 1 >= 0, has_l, has_r, qa, qb);
    hfilt_up_s(S(h0, 0) + my, tpp, true, has_l, has_r, da, db);
    bf16* on = out_n + (int64_t)b * (2 * H) * Wo * out_n_ld + c0;
    bf16* orw = out_r + (int64_t)b * (2 * H) * Wo * out_r_ld + c0;
    for (int hi = h0; hi < h1; ++hi) {
        __syncthreads();                              // row hi+1 is complete; the slot of row hi-1's predecessor is free
        const bool more = hi + 2 <= h1;               // block-uniform: row hi+2 is needed by the next trip
        if (more) stage_load(hi + 2);                 // its loads overlap this row's arithmetic
        float na[8], nb[8], o[8];
        const bool nrow = hi + 1 < H;
        hfilt_up_s(S(hi + 1, 1) + my, tpp, nrow, has_l, has_r, na, nb);
        if (live) {
            bf16* r_even = on + ((int64_t)(2 * hi) * Wo + 2 * wi) * out_n_ld;
            bf16* r_odd = r_even + (int64_t)Wo * out_n_ld;
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = fmaf(0.25f, pa[j], 0.75f * ca[j]);
            *reinterpret_cast<uint4*>(r_even) = pack8(o);
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = fmaf(0.25f, pb[j], 0.75f * cb[j]);
            *reinterpret_cast<uint4*>(r_even + out_n_ld) = pack8(o);
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = fmaf(0.25f, na[j], 0.75f * ca[j]);
            *reinterpret_cast<uint4*>(r_odd) = pack8(o);
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = fmaf(0.25f, nb[j], 0.75f * cb[j]);
            *reinterpret_cast<uint4*>(r_odd + out_n_ld) = pack8(o);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) { pa[j] = ca[j]; pb[j] = cb[j]; ca[j] = na[j]; cb[j] = nb[j]; }
        hfilt_up_s(S(hi + 1, 0) + my, tpp, nrow, has_l, has_r, na, nb);
        if (live) {
            bf16* r_even = orw + ((int64_t)(2 * hi) * Wo + 2 * wi) * out_r_ld;
            bf16* r_odd = r_even + (int64_t)Wo * out_r_ld;
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = fmaf(0.25f, qa[j], 0.75f * da[j]);
            *reinterpret_cast<uint4*>(r_even) = pack8(o);
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = fmaf(0.25f, qb[j], 0.75f * db[j]);
            *reinterpret_cast<uint4*>(r_even + out_r_ld) = pack8(o);
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = fmaf(0.25f, na[j], 0.75f * da[j]);
            *reinterpret_cast<uint4*>(r_odd) = pack8(o);
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = fmaf(0.25f, nb[j], 0.75f * db[j]);
            *reinterpret_cast<uint4*>(r_odd + out_r_ld) = pack8(o);
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) { qa[j] = da[j]; qb[j] = db[j]; da[j] = na[j]; db[j] = nb[j]; }
        if (more) stage_store(hi + 2);
    }
}

__global__ void __launch_bounds__(256)
fir_down2_f4_kernel(const float4* __restrict__ x, int H, int W, float4* __restrict__ out, int64_t total) {
    pdl_sync();
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int Ho = H >> 1, Wo = W >> 1;
    int64_t pix = idx;
    const int wo = (int)(pix % Wo);
    pix /= Wo;
    const int ho = (int)(pix % Ho);
    const int b = (int)(pix / Ho);
    const float k[4] = {0.125f, 0.375f, 0.375f, 0.125f};
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int hh = 2 * ho - 1 + a;
        if (hh < 0 || hh >= H) continue;
#pragma unroll
        for (int bb = 0; bb < 4; ++bb) {
            const int ww = 2 * wo - 1 + bb;
            if (ww < 0 || ww >= W) continue;
            const float4 v = __ldg(x + ((int64_t)b * H + hh) * W + ww);
            const float kw = k[a] * k[bb];
            acc.x = fmaf(kw, v.x, acc.x);
            acc.y = fmaf(kw, v.y, acc.y);
            acc.z = fmaf(kw, v.z, acc.z);
            acc.w = fmaf(kw, v.w, acc.w);
        }
    }
    out[idx] = acc;
}

__global__ void __launch_bounds__(256)
fir_up2_f4_kernel(const float4* __restrict__ x, int H, int W, float4* __restrict__ out, int64_t total) {
    pdl_sync();
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int Ho = H * 2, Wo = W * 2;
    int64_t pix = idx;
    const int wo = (int)(pix % Wo);
    pix /= Wo;
    const int ho = (int)(pix % Ho);
    const int b = (int)(pix / Ho);
    const int hi = ho >> 1, wi = wo >> 1;
    const int ha = (ho & 1) ? hi : hi - 1;
    const int wa = (wo & 1) ? wi : wi - 1;
    const float kha = (ho & 1) ? 0.75f : 0.25f;
    const float kwa = (wo & 1) ? 0.75f : 0.25f;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int a = 0; a < 2; ++a) {
        const int hh = ha + a;
        if (hh < 0 || hh >= H) continue;
        const float kh = a == 0 ? kha : 1.0f - kha;
#pragma unroll
        for (int bb = 0; bb < 2; ++bb) {
            const int ww = wa + bb;
            if (ww < 0 || ww >= W) continue;
            const float kk = kh * (bb == 0 ? kwa : 1.0f - kwa);
            const float4 v = __ldg(x + ((int64_t)b * H + hh) * W + ww);
            acc.x = fmaf(kk, v.x, acc.x);
            acc.y = fmaf(kk, v.y, acc.y);
            acc.z = fmaf(kk, v.z, acc.z);
            acc.w = fmaf(kk, v.w, acc.w);
        }
    }
    out[idx] = acc;
}

// General upfirdn2d (ncsnpp_utils/op/upfirdn2d.cpp:12-23; the "large" path of op/upfirdn2d_kernel.cu:25-104 and the
// pure-torch statement op/upfirdn2d.py:159-200): zero-insertion upsampling by (up_x, up_y), padding (negative = crop),
// correlation with the flipped kernel, decimation by (down_x, down_y).  fp32 planes [major][in_h][in_w] (the reference
// always passes minor = 1).  One thread per output sample, filter taps from shared memory; only the taps that land on
// a real (non-inserted) input sample are visited.
__global__ void __launch_bounds__(256)
upfirdn2d_kernel(const float* __restrict__ x, const float* __restrict__ k, float* __restrict__ out, int in_h, int in_w,
                 int kh, int kw, int up_x, int up_y, int down_x, int down_y, int pad_x0, int pad_y0, int out_h, int out_w,
                 int64_t total) {
    pdl_sync();
    extern __shared__ float ks[];
    for (int i = threadIdx.x; i < kh * kw; i += blockDim.x) ks[i] = k[i];
    __syncthreads();
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int ox = (int)(idx % out_w);
    const int64_t r = idx / out_w;
    const int oy = (int)(r % out_h);
    const int64_t m = r / out_h;
    const float* xp = x + m * in_h * in_w;
    // output (oy, ox) = sum_{ky,kx} k[kh-1-ky][kw-1-kx] * U[oy*down_y + ky - pad_y0][ox*down_x + kx - pad_x0],
    // U[uy][ux] = x[uy/up_y][ux/up_x] when both divide exactly and the indices are inside the image, else 0
    const int by = oy * down_y - pad_y0, bx = ox * down_x - pad_x0;
    int ky0 = ((-by) % up_y + up_y) % up_y;        // first ky with (by + ky) % up_y == 0
    int kx0 = ((-bx) % up_x + up_x) % up_x;
    float acc = 0.f;
    for (int ky = ky0; ky < kh; ky += up_y) {
        const int uy = by + ky;
        if (uy < 0) continue;
        const int iy = uy / up_y;
        if (iy >= in_h) break;
        for (int kx = kx0; kx < kw; kx += up_x) {
            const int ux = bx + kx;
            if (ux < 0) continue;
            const int ix = ux / up_x;
            if (ix >= in_w) break;
            acc = fmaf(xp[(int64_t)iy * in_w + ix], ks[(kh - 1 - ky) * kw + (kw - 1 - kx)], acc);
        }
    }
    out[idx] = acc;
}

}  // namespace

int upfirdn2d_launch(const float* x, const float* kernel, float* out, int64_t major, int in_h, int in_w, int kh, int kw,
                     int up_x, int up_y, int down_x, int down_y, int pad_x0, int pad_x1, int pad_y0, int pad_y1,
                     cudaStream_t s) {
    SNRSE_CHECK_ARG(major > 0 && in_h > 0 && in_w > 0 && kh > 0 && kw > 0, "upfirdn2d: empty input or kernel");
    SNRSE_CHECK_ARG(up_x >= 1 && up_y >= 1 && down_x >= 1 && down_y >= 1, "upfirdn2d: up / down factors must be >= 1");
    SNRSE_CHECK_ARG(kh * kw <= 4096, "upfirdn2d: kernel larger than 4096 taps");
    const int out_h = (in_h * up_y + pad_y0 + pad_y1 - kh) / down_y + 1;
    const int out_w = (in_w * up_x + pad_x0 + pad_x1 - kw) / down_x + 1;
    SNRSE_CHECK_ARG(in_h * up_y + pad_y0 + pad_y1 >= kh && in_w * up_x + pad_x0 + pad_x1 >= kw && out_h > 0 && out_w > 0,
                    "upfirdn2d: padded input smaller than the kernel");
    const int64_t total = major * out_h * out_w;
    snrse_launch(upfirdn2d_kernel, dim3((unsigned)cdiv64(total, 256)), dim3(256), kh * kw * sizeof(float), s, 
        x, kernel, out, in_h, in_w, kh, kw, up_x, up_y, down_x, down_y, pad_x0, pad_y0, out_h, out_w, total);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}

int fir_down2_launch(const ActView* x, const ActView* out, cudaStream_t s) {
    SNRSE_CHECK_ARG(x->H % 2 == 0 && x->W % 2 == 0 && x->C % 8 == 0, "fir_down2: H, W must be even, C %% 8 == 0");
    SNRSE_CHECK_ARG(x->C <= 2048 && x->B <= 65535, "fir_down2: C <= 2048, B <= 65535");
    const int tpp = x->C / 8, nthr = tpp * (256 / tpp > 0 ? 256 / tpp : 1), cols = nthr / tpp;
    // rows per block: as many as keep >= ~4 blocks per SM in flight (small maps would otherwise use a handful of SMs)
    int band = FIR_BAND;
    while (band > 1 && (int64_t)cdiv(x->W / 2, cols) * cdiv(x->H / 2, band) * x->B < 592) band >>= 1;
    dim3 grid((unsigned)cdiv(x->W / 2, cols), (unsigned)cdiv(x->H / 2, band), (unsigned)x->B);
    snrse_launch(fir_down2_kernel, dim3(grid), dim3(nthr), 0, s, x->ptr, x->ld, x->C, x->H, x->W, out->ptr, out->ld, band);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}

int fir_up2_launch(const ActView* x, const ActView* out, cudaStream_t s) {
    SNRSE_CHECK_ARG(x->C % 8 == 0, "fir_up2: C %% 8 == 0");
    SNRSE_CHECK_ARG(x->C <= 2048 && x->B <= 65535, "fir_up2: C <= 2048, B <= 65535");
    const int tpp = x->C / 8, nthr = tpp * (256 / tpp > 0 ? 256 / tpp : 1), cols = nthr / tpp;
    int band = FIR_BAND;
    while (band > 1 && (int64_t)cdiv(x->W, cols) * cdiv(x->H, band) * x->B < 592) band >>= 1;
    dim3 grid((unsigned)cdiv(x->W, cols), (unsigned)cdiv(x->H, band), (unsigned)x->B);
    snrse_launch(fir_up2_kernel, dim3(grid), dim3(nthr), 0, s, x->ptr, x->ld, x->C, x->H, x->W, out->ptr, out->ld, band);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}

int fir_dual_launch(const ActView* x, const ActView* out_n, const ActView* out_r, int up, const float* scsh, cudaStream_t s) {
    SNRSE_CHECK_ARG(scsh != nullptr, "fir_dual: GroupNorm scale / shift required");
    SNRSE_CHECK_ARG(x->C % 8 == 0 && x->C <= 1024 && x->B <= 65535, "fir_dual: C %% 8 == 0, C <= 1024, B <= 65535");
    SNRSE_CHECK_ARG(up || (x->H % 2 == 0 && x->W % 2 == 0), "fir_dual (down): H, W must be even");
    const int tpp = x->C / 8, nthr = tpp * (256 / tpp > 0 ? 256 / tpp : 1), cols = nthr / tpp;
    const int wcols = up ? x->W : x->W / 2, hrows = up ? x->H : x->H / 2;
    int band = FIR_BAND;
    while (band > 1 && (int64_t)cdiv(wcols, cols) * cdiv(hrows, band) * x->B < 592) band >>= 1;
    dim3 grid((unsigned)cdiv(wcols, cols), (unsigned)cdiv(hrows, band), (unsigned)x->B);
    // staged rows: down 2 slots x 2 rows, up a ring of 3 rows; raw + normalised copies, 16 bytes per (column, 8 channels)
    const size_t smem = (size_t)(up ? 3 * 2 * (cols + 2) : 2 * 2 * 2 * (2 * cols + 2)) * tpp * 16;
    static bool attr_set = false;
    if (!attr_set) {
        SNRSE_CUDA(cudaFuncSetAttribute(fir_down2_dual_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
        SNRSE_CUDA(cudaFuncSetAttribute(fir_up2_dual_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
        attr_set = true;
    }
    SNRSE_CHECK_ARG(smem <= 160 * 1024, "fir_dual: row staging does not fit shared memory");
    if (up) snrse_launch(fir_up2_dual_kernel, dim3(grid), dim3(nthr), smem, s, x->ptr, x->ld, x->C, x->H, x->W, out_n->ptr, out_n->ld, out_r->ptr, out_r->ld, band, scsh);
    else snrse_launch(fir_down2_dual_kernel, dim3(grid), dim3(nthr), smem, s, x->ptr, x->ld, x->C, x->H, x->W, out_n->ptr, out_n->ld, out_r->ptr, out_r->ld, band, scsh);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}

int fir_down2_f4_launch(const float* x, float* out, int B, int H, int W, cudaStream_t s) {
    SNRSE_CHECK_ARG(H % 2 == 0 && W % 2 == 0, "fir_down2_f4: H, W must be even");
    const int64_t total = (int64_t)B * (H / 2) * (W / 2);
    snrse_launch(fir_down2_f4_kernel, dim3((unsigned)cdiv64(total, 256)), dim3(256), 0, s, reinterpret_cast<const float4*>(x), H, W,
                                                                     reinterpret_cast<float4*>(out), total);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}

int fir_up2_f4_launch(const float* x, float* out, int B, int H, int W, cudaStream_t s) {
    const int64_t total = (int64_t)B * (H * 2) * (W * 2);
    snrse_launch(fir_up2_f4_kernel, dim3((unsigned)cdiv64(total, 256)), dim3(256), 0, s, reinterpret_cast<const float4*>(x), H, W,
                                                                   reinterpret_cast<float4*>(out), total);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}
