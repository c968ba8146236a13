// Implicit-GEMM convolution for the NCSN++ 3x3 / 1x1 / NIN contractions on the sm_100a tensor cores.
//
// Replaces the cuDNN / cuBLAS calls behind `ddpm_conv3x3`, `ddpm_conv1x1` and `NIN`
// (reference: sgmse-bbed/sgmse/backbones/ncsnpp_utils/layers.py:100-124,537-555) as used by
// `ResnetBlockBigGANpp` / `AttnBlockpp` (layerspp.py:64-93,244-276).
//
// Formulation (NHWC bf16 activations, fp32 accumulation in TMEM):
//   M = 128 output pixels per CTA, arranged as a th x tw patch of one image (th*tw = 128);
//   N = output channels handled by the CTA (64 / 128 / 256);
//   K = walked in blocks of 64 input channels: segment 0 visits `taps0` filter taps (9 for 3x3,
//       pad 1) x C0/64 channel chunks, an optional segment 1 (the fused 1x1 shortcut `Conv_2`)
//       visits C1/64 chunks of a second input with a single tap.
//   A operand: one 4-D TMA box {64 ch, tw, th, 1} per K block, fetched at the tap-shifted pixel
//       coordinate; out-of-image rows are zero-filled by TMA, which is exactly the conv padding,
//       so no im2col buffer ever exists.  The box lands in shared memory as 128 rows x 128 B with
//       the 128-byte swizzle == the canonical K-major UMMA operand layout.
//   B operand: weights pre-packed [Cout][tap][cin] (K-major), a {64, N} TMA box per K block.
//   tcgen05.mma (cta_group::1, kind::f16, M=128, N, K=16) x 4 per K block, accumulator in TMEM.
//   Warp roles: warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer, warps 2-5 = epilogue
//   (tcgen05.ld -> +bias +time-embedding bias +residual, *scale -> bf16/f32 global stores).
#include <cuda.h>

#include "kernels.h"
#include "ptx.cuh"
#include "tma_host.h"

namespace {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;                      // bf16 elements = 128 bytes = one swizzle row
constexpr int A_STAGE_BYTES = BLOCK_M * BLOCK_K * 2;  // 16 KB
constexpr int NUM_THREADS = 224;   // warp 0: activation TMA, 1: MMA, 2-5: epilogue, 6: weight TMA
constexpr int MAX_STAGES = 8;

struct GemmArgs {
    int taps0, c0_chunks, c1_chunks;
    int H, W;
    int th_log2, tw_log2, tiles_h, tiles_w;
    int N, n_tile, b_batched;
    const float* bias;
    const float* tbias;
    int tb_stride;
    const bf16* res;
    int res_ld;
    float scale;
    void* out;
    int out_ld;
    int out_f32;
    int stages;
    int a_box_bytes;   // bytes one activation TMA box delivers (rows of the tile that exist in the image)
    long long* dbg;
};

__global__ void __launch_bounds__(NUM_THREADS, 1)
conv_gemm_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                 const __grid_constant__ CUtensorMap mapB, const GemmArgs g) {
    pdl_trigger();   // the next kernel may become resident; it blocks in its own pdl_wait()
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[MAX_STAGES];
    __shared__ __align__(8) uint64_t empty_bar[MAX_STAGES];
    __shared__ __align__(8) uint64_t accum_bar;
    __shared__ uint32_t tmem_base_smem;

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);   // provably warp-uniform (uniform-register descriptors)
    const int lane = threadIdx.x & 31;

    // ---- tile coordinates
    int tile = blockIdx.x;
    const int tw_idx = tile % g.tiles_w;
    tile /= g.tiles_w;
    const int th_idx = tile % g.tiles_h;
    const int b = tile / g.tiles_h;
    const int h0 = th_idx << g.th_log2;
    const int w0 = tw_idx << g.tw_log2;
    const int n0 = blockIdx.y * g.n_tile;

    const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;  // 128B-swizzle atoms need 1024B alignment
    const uint32_t b_stage_bytes = (uint32_t)g.n_tile * BLOCK_K * 2;
    const uint32_t stage_bytes = A_STAGE_BYTES + b_stage_bytes;
    const int nkb0 = g.taps0 * g.c0_chunks;
    const int nkb = nkb0 + g.c1_chunks;
    const uint32_t tmem_cols = (uint32_t)g.n_tile;  // 64 / 128 / 256: already a power of two >= 32

    if (warp == 1) {
        if (lane == 0) {
            for (int s = 0; s < g.stages; ++s) {
                ptx::mbar_init(ptx::smem_u32(&full_bar[s]), 2);   // one arrival per producer warp
                ptx::mbar_init(ptx::smem_u32(&empty_bar[s]), 1);
            }
            ptx::mbar_init(ptx::smem_u32(&accum_bar), 1);
            ptx::fence_barrier_init();
        }
        __syncwarp();
        ptx::tmem_alloc(ptx::smem_u32(&tmem_base_smem), tmem_cols);
        ptx::tmem_relinquish();
    } else if (warp == 0 && lane == 0) {
        ptx::prefetch_tensormap(&mapA0);
        ptx::prefetch_tensormap(&mapB);
        if (g.c1_chunks > 0) ptx::prefetch_tensormap(&mapA1);
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, tmem_base_smem, 0);
    // Programmatic dependent launch: barrier init, TMEM allocation and descriptor prefetch above overlap the predecessor's
    // tail; the weight producer streams its (constant) tiles right away, everyone else waits for the predecessor's data
    if (!(warp == 6 && !g.b_batched)) pdl_wait();

    if (warp == 0) {
        // =========================== TMA producer ===========================
        // the whole warp walks the loop (uniform control flow), one elected lane issues
        const bool elected = ptx::elect_one();
        long long w_empty = 0, t_begin = g.dbg ? clock64() : 0;
        // ring slot / phase and (tap, chunk) are carried incrementally: a runtime integer division costs ~150 clk of
        // exposed latency in this single-warp loop, and four of them per K block made the producer (570 clk per block),
        // not the tensor pipe (130 clk), the bound of the small-map layers
        int s = 0, tap = 0, chunk = 0;
        uint32_t ph = 0;
        for (int kb = 0; kb < nkb; ++kb) {
            long long t0 = g.dbg ? clock64() : 0;
            ptx::mbar_wait(ptx::smem_u32(&empty_bar[s]), ph ^ 1u);
            if (g.dbg) w_empty += clock64() - t0;
            const uint32_t fb = ptx::smem_u32(&full_bar[s]);
            const uint32_t sa = smem_base + (uint32_t)s * stage_bytes;
            const bool seg0 = kb < nkb0;
            int dh = 0, dw = 0;
            if (seg0 && g.taps0 == 9) {
                const int t3 = (tap * 11) >> 5;          // tap / 3 for tap in 0..8
                dh = t3 - 1;
                dw = tap - 3 * t3 - 1;
            }
            if (elected) {
                ptx::mbar_arrive_expect_tx(fb, (uint32_t)g.a_box_bytes);
                if (seg0) ptx::tma_load_4d(sa, &mapA0, fb, chunk * BLOCK_K, w0 + dw, h0 + dh, b);
                else ptx::tma_load_4d(sa, &mapA1, fb, chunk * BLOCK_K, w0, h0, b);
            }
            __syncwarp();
            if (++s == g.stages) { s = 0; ph ^= 1u; }
            if (seg0) {
                if (++chunk == g.c0_chunks) { chunk = 0; ++tap; }
                if (kb + 1 == nkb0) chunk = 0;           // second segment (1x1 shortcut operand) restarts at chunk 0
            } else {
                ++chunk;
            }
        }
        if (g.dbg && elected && blockIdx.y == 0) {
            g.dbg[blockIdx.x * 8 + 0] = w_empty;
            g.dbg[blockIdx.x * 8 + 1] = clock64() - t_begin;
        }
    } else if (warp == 6) {
        // =========================== TMA producer, weights ===========================
        // the two operands get a producer warp each: every producer step is a chain of dependent special instructions
        // (barrier wait ~130 clk, expect-tx, TMA issue), and the small-map layers are bound by that chain, not by data
        const bool elected = ptx::elect_one();
        int s = 0;
        uint32_t ph = 0;
        for (int kb = 0; kb < nkb; ++kb) {
            ptx::mbar_wait(ptx::smem_u32(&empty_bar[s]), ph ^ 1u);
            const uint32_t fb = ptx::smem_u32(&full_bar[s]);
            const uint32_t sa = smem_base + (uint32_t)s * stage_bytes;
            if (elected) {
                ptx::mbar_arrive_expect_tx(fb, b_stage_bytes);
                ptx::tma_load_3d(sa + A_STAGE_BYTES, &mapB, fb, kb * BLOCK_K, n0, g.b_batched ? b : 0);
            }
            __syncwarp();
            if (++s == g.stages) { s = 0; ph ^= 1u; }
        }
    } else if (warp == 1) {
        // =========================== MMA issuer ===========================
        const uint32_t idesc = ptx::umma_idesc_bf16(BLOCK_M, (uint32_t)g.n_tile);
        const bool elected = ptx::elect_one();
        long long w_full = 0, w_first = 0, t_begin = g.dbg ? clock64() : 0;
        int s = 0;
        uint32_t ph = 0;
        for (int kb = 0; kb < nkb; ++kb) {
            long long t0 = g.dbg ? clock64() : 0;
            ptx::mbar_wait(ptx::smem_u32(&full_bar[s]), ph);
            if (g.dbg) { const long long d = clock64() - t0; w_full += d; if (kb == 0) w_first = d; }
            ptx::tc_fence_after();
            const uint32_t sa = smem_base + (uint32_t)s * stage_bytes;
            const uint64_t da = ptx::umma_desc_k_sw128(sa);
            const uint64_t db = ptx::umma_desc_k_sw128(sa + A_STAGE_BYTES);
            if (elected) {
                // advance 16 bf16 = 32 bytes along K inside the swizzle atom: +2 in the (addr>>4) field
                ptx::mma_bf16_ss(tmem_base, da, db, idesc, kb > 0 ? 1u : 0u);
                ptx::mma_bf16_ss(tmem_base, da + 2, db + 2, idesc, 1u);
                ptx::mma_bf16_ss(tmem_base, da + 4, db + 4, idesc, 1u);
                ptx::mma_bf16_ss(tmem_base, da + 6, db + 6, idesc, 1u);
                ptx::mma_commit(ptx::smem_u32(&empty_bar[s]));  // frees the smem stage when these MMAs retire
            }
            __syncwarp();
            if (++s == g.stages) { s = 0; ph ^= 1u; }
        }
        if (elected) ptx::mma_commit(ptx::smem_u32(&accum_bar));  // accumulator complete
        __syncwarp();
        if (g.dbg && elected && blockIdx.y == 0) {
            g.dbg[blockIdx.x * 8 + 2] = w_full;
            g.dbg[blockIdx.x * 8 + 3] = clock64() - t_begin;
            g.dbg[blockIdx.x * 8 + 4] = w_first;
        }
    } else {
        // =========================== epilogue (warps 2..5) ===========================
        const int quarter = warp & 3;  // TMEM lane quarter this warp may access
        const int row = quarter * 32 + lane;
        const int hl = row >> g.tw_log2;
        const int wl = row & ((1 << g.tw_log2) - 1);
        const int h = h0 + hl, w = w0 + wl;
        const bool valid = (h < g.H) && (w < g.W);
        const int64_t pix = ((int64_t)b * g.H + h) * g.W + w;
        ptx::mbar_wait(ptx::smem_u32(&accum_bar), 0);
        ptx::tc_fence_after();
        const float* tb = g.tbias ? g.tbias + (int64_t)b * g.tb_stride : nullptr;
        for (int c0 = 0; c0 < g.n_tile; c0 += 32) {
            uint32_t v[32];
            ptx::tmem_ld_32x32(tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)c0, v);
            ptx::tmem_ld_wait();
            const int n = n0 + c0;
            if (valid && n < g.N) {
                float f[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
                if (g.bias) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] += __ldg(g.bias + n + j);
                }
                if (tb) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) f[j] += __ldg(tb + n + j);
                }
                if (g.res) {
                    const uint4* rp = reinterpret_cast<const uint4*>(g.res + pix * g.res_ld + n);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        float r[8];
                        unpack8(__ldg(rp + q), r);
#pragma unroll
                        for (int j = 0; j < 8; ++j) f[q * 8 + j] += r[j];
                    }
                }
#pragma unroll
                for (int j = 0; j < 32; ++j) f[j] *= g.scale;
                if (g.out_f32) {
                    float4* op = reinterpret_cast<float4*>(reinterpret_cast<float*>(g.out) + pix * g.out_ld + n);
#pragma unroll
                    for (int q = 0; q < 8; ++q) op[q] = make_float4(f[4 * q], f[4 * q + 1], f[4 * q + 2], f[4 * q + 3]);
                } else {
                    uint4* op = reinterpret_cast<uint4*>(reinterpret_cast<bf16*>(g.out) + pix * g.out_ld + n);
#pragma unroll
                    for (int q = 0; q < 4; ++q) op[q] = pack8(f + 8 * q);
                }
            }
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        __syncwarp();
        ptx::tmem_dealloc(tmem_base, tmem_cols);
    }
}

}  // namespace
extern long long* g_halo_dbg_shared;
namespace {
int ilog2(int v) {
    int l = 0;
    while ((1 << l) < v) ++l;
    return l;
}

}  // namespace

int conv_gemm_make_plan(ConvGemmPlan* p, const ActView* a0, int taps0, const ActView* a1, const bf16* wt, int n_rows,
                        int64_t wt_batch_stride, int b_batched, const float* bias, const float* tbias, int tb_stride,
                        const ActView* res, float scale, void* out, int out_ld, int out_f32) {
    return conv_gemm_make_plan_ex(p, a0, taps0, a1, wt, n_rows, wt_batch_stride, b_batched, bias, tbias, tb_stride, res,
                                  scale, out, out_ld, out_f32, 0);
}

int conv_gemm_plan_shape(ConvGemmPlan* p, int B, int H, int W, int taps0, int C0, int C1, int n_rows, int num_sms) {
    SNRSE_CHECK_ARG(taps0 == 1 || taps0 == 9, "conv_gemm: taps0 must be 1 or 9");
    SNRSE_CHECK_ARG(C0 % 64 == 0, "conv_gemm: Cin must be a multiple of 64 (got %d)", C0);
    SNRSE_CHECK_ARG(C1 % 64 == 0, "conv_gemm: Cin1 must be a multiple of 64");
    SNRSE_CHECK_ARG(n_rows % 32 == 0, "conv_gemm: N must be a multiple of 32 (got %d)", n_rows);
    memset(p, 0, sizeof(*p));
    p->taps0 = taps0;
    p->c0_chunks = C0 / 64;
    p->c1_chunks = C1 / 64;
    p->B = B;
    p->H = H;
    p->W = W;
    // tile shape: th*tw = 128, fewest tiles; ties -> prefer 8x16 (small halo for the 3x3 taps)
    int best_tw = 128, best_tiles = 1 << 30, best_rank = 1 << 30;
    for (int tw = 1; tw <= 128; tw <<= 1) {
        const int th = 128 / tw;
        const int tiles = cdiv(H, th) * cdiv(W, tw);
        const int rank = abs(ilog2(tw) - 4);
        if (tiles < best_tiles || (tiles == best_tiles && rank < best_rank)) {
            best_tiles = tiles;
            best_tw = tw;
            best_rank = rank;
        }
    }
    const int tw = best_tw, th = 128 / tw;
    p->tw_log2 = ilog2(tw);
    p->th_log2 = ilog2(th);
    p->tiles_h = cdiv(H, th);
    p->tiles_w = cdiv(W, tw);
    p->N = n_rows;
    p->n_tile = n_rows >= 256 ? 256 : (n_rows >= 128 ? 128 : 64);
    // Few pixel tiles (small feature maps): one CTA walks the whole K loop alone and is bound by the TMA latency per
    // K block, not by the tensor pipe.  Split N into 64-column tiles (4x the CTAs, a quarter of the MMA time each) and
    // give every CTA a whole SM's shared memory for a deep TMA ring.
    const int64_t pixel_tiles = (int64_t)B * p->tiles_h * p->tiles_w;
    const bool small = pixel_tiles * cdiv(n_rows, p->n_tile) * 2 <= num_sms && n_rows % 64 == 0;
    if (small) p->n_tile = 64;
    p->small = small;
    const int stage_bytes = A_STAGE_BYTES + p->n_tile * BLOCK_K * 2;
    // two CTAs per SM when possible (overlaps one tile's epilogue with the other's main loop)
    int stages = ((small ? 196 : 110) * 1024) / stage_bytes;
    if (stages > MAX_STAGES) stages = MAX_STAGES;
    if (stages < 2) stages = 2;
    const int nkb = taps0 * p->c0_chunks + p->c1_chunks;
    if (stages > nkb) stages = nkb < 2 ? 2 : nkb;
    p->stages = stages;
    p->smem_bytes = stages * stage_bytes + 1024;
    p->a_box_bytes = th * tw * 128;
    return SNRSE_OK;
}

int conv_gemm_make_plan_ex(ConvGemmPlan* p, const ActView* a0, int taps0, const ActView* a1, const bf16* wt, int n_rows,
                           int64_t wt_batch_stride, int b_batched, const float* bias, const float* tbias, int tb_stride,
                           const ActView* res, float scale, void* out, int out_ld, int out_f32, int64_t wt_row_pitch) {
    SNRSE_CHECK_ARG(a0->ld % 8 == 0, "conv_gemm: the operand pitch must be a multiple of 8");
    SNRSE_CHECK_ARG(!a1 || a1->ld % 8 == 0, "conv_gemm: the shortcut operand pitch must be a multiple of 8");
    SNRSE_CHECK_ARG(!a1 || (a1->B == a0->B && a1->H == a0->H && a1->W == a0->W), "conv_gemm: segment shapes differ");
    SNRSE_CHECK_ARG(out_ld % (out_f32 ? 4 : 8) == 0, "conv_gemm: output pitch must be a multiple of 16 bytes");
    SNRSE_CHECK_ARG(!res || res->ld % 8 == 0, "conv_gemm: residual pitch must be a multiple of 8");
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    SNRSE_TRY(conv_gemm_plan_shape(p, a0->B, a0->H, a0->W, taps0, a0->C, a1 ? a1->C : 0, n_rows, sms));
    p->b_batched = b_batched;
    p->bias = bias;
    p->tbias = tbias;
    p->tb_stride = tb_stride;
    p->res = res ? res->ptr : nullptr;
    p->res_ld = res ? res->ld : 0;
    p->scale = scale;
    p->out = out;
    p->out_ld = out_ld;
    p->out_f32 = out_f32;
    const int64_t ktot = (int64_t)64 * (taps0 * p->c0_chunks + p->c1_chunks);
    const int tw = 1 << p->tw_log2, th = 1 << p->th_log2;
    SNRSE_TRY(tma_make_act_map(&p->mapA0, a0->ptr, a0->C, a0->W, a0->H, a0->B, a0->ld, 64, tw, th));
    if (a1) {
        SNRSE_TRY(tma_make_act_map(&p->mapA1, a1->ptr, a1->C, a1->W, a1->H, a1->B, a1->ld, 64, tw, th));
    } else {
        p->mapA1 = p->mapA0;
    }
    const int nb = b_batched ? a0->B : 1;
    SNRSE_TRY(tma_make_wt_map(&p->mapB, wt, ktot, n_rows, nb, b_batched ? wt_batch_stride : ktot * n_rows, 64, p->n_tile,
                              wt_row_pitch));
    return SNRSE_OK;
}

int conv_gemm_launch(const ConvGemmPlan* p, cudaStream_t s) {
    static bool attr_set = false;
    if (!attr_set) {
        // opt-in limit is 227 KB per block INCLUDING the kernel's static shared memory (barriers)
        SNRSE_CUDA(cudaFuncSetAttribute(conv_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        attr_set = true;
    }
    GemmArgs g;
    g.taps0 = p->taps0;
    g.c0_chunks = p->c0_chunks;
    g.c1_chunks = p->c1_chunks;
    g.H = p->H;
    g.W = p->W;
    g.th_log2 = p->th_log2;
    g.tw_log2 = p->tw_log2;
    g.tiles_h = p->tiles_h;
    g.tiles_w = p->tiles_w;
    g.N = p->N;
    g.n_tile = p->n_tile;
    g.b_batched = p->b_batched;
    g.bias = p->bias;
    g.tbias = p->tbias;
    g.tb_stride = p->tb_stride;
    g.res = p->res;
    g.res_ld = p->res_ld;
    g.scale = p->scale;
    g.out = p->out;
    g.out_ld = p->out_ld;
    g.out_f32 = p->out_f32;
    g.stages = p->stages;
    g.a_box_bytes = p->a_box_bytes;
    g.dbg = g_halo_dbg_shared;
    dim3 grid((unsigned)(p->B * p->tiles_h * p->tiles_w), (unsigned)cdiv(p->N, p->n_tile));
    snrse_launch_m(2, conv_gemm_kernel, dim3(grid), dim3(NUM_THREADS), p->smem_bytes, s, p->mapA0, p->mapA1, p->mapB, g);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}
