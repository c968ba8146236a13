// Persistent 2-CTA (cta_group::2) implicit-GEMM 3x3 convolution for sm_100a (tcgen05 + TMEM + TMA).
//
// Same contract as conv_gemm.cu (ddpm_conv3x3 of sgmse-bbed/sgmse/backbones/ncsnpp_utils/layers.py:118-124,
// with the fused 1x1 shortcut / bias / time-embedding bias / residual epilogue of layerspp.py:262-276).
// Design facts it is built on (profiles/r01_mma_probe.md):
//   * a single CTA with both operands in shared memory tops out at 60 % (N=128) / 75 % (N=256) of the tensor
//     peak; a CTA pair (M=256 across two SMs, each SM streaming its 128 pixel rows and HALF of the weight tile)
//     reaches 100 % at N=128 and N=256  -> two CTAs of one TPC form a cluster, the leader issues the MMAs;
//   * a SWIZZLE_128B K-major UMMA descriptor may start at any 128-byte row of a TMA-written tile and use any
//     multiple of 128 B as the stride between 8-row groups  -> ONE halo tile per 64-channel chunk serves all
//     nine taps: sub-tile = 16 image rows x 8 pixels (M = 128, one 8-row group per image row), halo tile =
//     [16*SUB+2 rows][10 pixels][64 ch]; tap (r,s) of sub-tile u is the same buffer addressed from row
//     ((r + 16u)*10 + s) with a group stride of 10 rows (1280 B).  L2->SM traffic per output pixel drops from
//     9 (first kernel) / 3.4 (three column-shifted copies) to 1.33 tile loads;
//   * the MMA / TMA issue loops are warp-uniform (descriptors in uniform registers, one elected lane issues).
//
// Super-tile = SUB (1 or 2) sub-tiles stacked in H sharing every weight tile; SUB accumulators of 128 lanes x N
// columns per CTA in TMEM, double-buffered when SUB*N <= 256 so the epilogue of tile i overlaps tile i+1.
// Two TMA rings: A (halo tiles, one per channel chunk) and B (per-tap weight tiles, N/2 rows per CTA); both
// CTAs' loads complete on the LEADER's barriers, tcgen05.commit multicasts to both CTAs.  The 128-output-channel
// layers with a fused 1x1 shortcut add a third ring for the shortcut operand's bare tiles (16 KB per sub-tile) and
// interleave those chunks behind the 3x3 chunks in the K loop; the A producer walks both rings with non-blocking
// barrier probes (see conv_halo2_make_plan).
// Programmatic dependent launch: the kernel triggers its successor at once and waits for its predecessor only after
// its own prologue; the weight producer never waits (weights are constants of the captured graph).
//
// Warp roles (12 warps): 0..7 = epilogue (TMEM lane quarter = warp & 3: 4 image rows x 8 pixels; column half =
// warp >> 2), 8 = A producer, 9 = B producer, 10 / 11 = MMA issuers of sub-tile 0 / 1 (11 owns TMEM).
// Each epilogue warp owns private 4 KB staging tiles (32 pixels x 64 channels, 128-byte swizzle): the residual
// arrives there by TMA, the warp adds accumulator / bias / time-embedding bias in place, one elected lane sends
// it out with a TMA store (full 128-byte lines, ragged edges clipped by the tensor map).
#include <cuda.h>
#include <stdlib.h>

#include "gn_fixed.cuh"
#include "kernels.h"
#include "ptx.cuh"
#include "tma_host.h"

namespace {

constexpr int HALO_THREADS = 384;        // + 256 (warps 12..19) when GroupNorm+SiLU is applied to the operand in flight
constexpr int NORM_WARP0 = 12, NORM_THREADS = 256;
constexpr int EPI_WARPS = 8;
// The warp scheduler favours the highest warp id of a sub-partition: the single-lane issue warps sit above the
// epilogue warps so that their (few) instructions never queue behind epilogue arithmetic.
constexpr int W_PROD_A = 8, W_PROD_B = 9, W_MMA0 = 10, W_MMA1 = 11;
constexpr int MAX_A = 3, MAX_B = 8, MAX_SC = 2;
constexpr int TW = 8, SUB_ROWS = 16, HALO_W = TW + 2;
constexpr uint32_t ROW_B = 128;                       // one pixel = 64 bf16 channels = one swizzle row

struct Halo2Args {
    int c0_chunks, c1_chunks;
    unsigned char seq[16];         // order of the channel chunks in the K loop: chunk | 0x80 for the 1x1 shortcut operand
    int H, W, B;
    int sub;                       // sub-tiles per super-tile (1 or 2)
    int tiles_h, tiles_w, n_tiles;
    int N;                         // columns per accumulator (128 or 256) == output channels / nsplit
    int nsplit, n_total;           // small maps: the clusters of the upper half of the grid take output channels N..2N-1
    int na, nb;                    // ring depths
    int nsc;                       // > 0: the 1x1 shortcut operand tiles travel through their own ring of nsc slots
    int acc_bufs;                  // 1 or 2 TMEM accumulator sets
    int stg_bufs;                  // 1 or 2 staging tiles per epilogue warp
    int has_res;
    float4* out4;                  // N == 16 only: fp32 4-channel output [B,H,W,4] = acc[:, 0:4] + bias (+ addend4)
    const float4* addend4;
    unsigned long long* ustats;    // null, or GroupNorm sums of the result, accumulated: [B][N/4][2] fixed point (gn_fixed.cuh)
    const float* scsh;             // null, or GroupNorm scale/shift [B][2][norm_c] applied (+SiLU) to operand 0 in shared memory
    int norm_c;
    const float* bias;
    const float* tbias;
    int tb_stride;
    float scale;
    long long* dbg;                // optional per-CTA cycle counters [grid][8] (measurement builds only)
};

#define DBG_T0() long long t0__ = g.dbg ? clock64() : 0
#define DBG_ADD(acc) do { if (g.dbg) { const long long t1__ = clock64(); acc += t1__ - t0__; t0__ = t1__; } } while (0)

__host__ __device__ inline uint32_t halo_stage_bytes(int sub) {   // halo tile rounded up to the 1 KB swizzle atom
    return (((uint32_t)(SUB_ROWS * sub + 2) * HALO_W * ROW_B) + 1023u) & ~1023u;
}

__host__ __device__ inline uint32_t halo_bsum_bytes(int n_cols) {   // EPI_WARPS slices of max(N/2, 32) floats
    return (uint32_t)(8 * (n_cols / 2 < 32 ? 32 : n_cols / 2) * 4);
}

// K-major SWIZZLE_128B descriptor with an explicit 8-row-group stride (bytes); start may be any 128-byte row
__device__ __forceinline__ uint64_t umma_desc_rows(uint32_t smem_addr, uint32_t group_stride) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(group_stride >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// Sum v[0..15] over the 32 lanes of the warp with a transpose-reduce butterfly (16 shuffles instead of 80): after
// it, lane l holds the warp total of element ((l>>1) & 15) [bit 4 of l = element bit 3, ... bit 1 = element bit 0;
// lanes l and l^1 hold the same value].  Fixed order -> deterministic.
__device__ __forceinline__ float warp_transpose_reduce16(float* v, int lane) {
    {
        const bool up = lane & 16;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float keep = up ? v[i + 8] : v[i], send = up ? v[i] : v[i + 8];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
    }
    {
        const bool up = lane & 8;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float keep = up ? v[i + 4] : v[i], send = up ? v[i] : v[i + 4];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
    }
    {
        const bool up = lane & 4;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const float keep = up ? v[i + 2] : v[i], send = up ? v[i] : v[i + 2];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
        }
    }
    {
        const bool up = lane & 2;
        const float keep = up ? v[1] : v[0], send = up ? v[0] : v[1];
        v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 2);
    }
    return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 1);
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(HALO_THREADS + NORM_THREADS, 1)
conv_halo2_kernel(const __grid_constant__ CUtensorMap mapA0, const __grid_constant__ CUtensorMap mapA1,
                  const __grid_constant__ CUtensorMap mapB, const __grid_constant__ CUtensorMap mapOut,
                  const __grid_constant__ CUtensorMap mapRes, const Halo2Args g) {
    pdl_trigger();   // the next kernel may become resident; it blocks in its own pdl_wait()
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t a_full[MAX_A], a_empty[MAX_A], a_land[MAX_A], b_full[MAX_B], b_empty[MAX_B];
    __shared__ __align__(8) uint64_t acc_full[2], acc_empty[2], res_bar[EPI_WARPS], sc_full[MAX_SC], sc_empty[MAX_SC];
    __shared__ uint32_t tmem_base_smem;

    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // provably warp-uniform
    const uint32_t rank = blockIdx.x & 1u;   // == %cluster_ctarank for cluster dims (2,1,1); 0 = leader (issues the MMAs)
    // N-split (maps too small to fill the GPU with pixel tiles): cluster c < n_ctiles computes output channels 0..N-1 of
    // tile c, cluster n_ctiles + c channels N..2N-1 of the same tile; each cluster then walks exactly one tile
    const int n_ctiles = (g.n_tiles + 1) >> 1;   // cluster tiles = pairs of super-tiles
    const int nhalf = (g.nsplit == 2 && (int)(blockIdx.x >> 1) >= n_ctiles) ? 1 : 0;
    const int cluster_id = (int)(blockIdx.x >> 1) - nhalf * n_ctiles;
    const int n_clusters = g.nsplit == 2 ? n_ctiles : (int)(gridDim.x >> 1);
    const int n_off = nhalf * g.N;               // first output channel of this cluster
    const uint32_t smem_base = (ptx::smem_u32(smem_raw) + 1023u) & ~1023u;
    const uint32_t a_bytes = halo_stage_bytes(g.sub);                                   // ring slot
    const uint32_t a_tx = (uint32_t)(SUB_ROWS * g.sub + 2) * HALO_W * ROW_B;            // bytes one halo TMA box delivers
    const uint32_t a1_tx = (uint32_t)(SUB_ROWS * g.sub) * TW * ROW_B;                   // shortcut operand: no halo
    const uint32_t b_bytes = (uint32_t)(g.N / 2) * ROW_B;   // this CTA's half of the weight tile
    // shared-memory map: halo ring | shortcut ring | weight ring | epilogue staging | per-warp additive terms
    const uint32_t a_base = smem_base, sc_base = a_base + (uint32_t)g.na * a_bytes;
    const uint32_t sc_bytes = a1_tx;                        // 16 KB per sub-tile: a multiple of the 1 KB swizzle atom
    const uint32_t b_base = sc_base + (uint32_t)g.nsc * sc_bytes;
    const uint32_t stg_base = b_base + (uint32_t)g.nb * b_bytes;
    const int n_astage = g.c0_chunks + g.c1_chunks;   // halo tiles consumed per super-tile
    const uint32_t acc_cols = (uint32_t)(g.sub * g.N);
    const uint32_t tmem_cols = acc_cols * (uint32_t)g.acc_bufs;  // 128/256/512: power of two
    const bool norm_on = g.scsh != nullptr;                      // GroupNorm + SiLU applied to operand 0 in flight
    // per epilogue warp: (bias + time-embedding bias) * scale for its N/2 columns
    const uint32_t bs_base = stg_base + (uint32_t)(EPI_WARPS * g.stg_bufs) * 4096u;

    if (warp == W_MMA1) {
        if (lane == 0) {
            for (int i = 0; i < g.na; ++i) {
                ptx::mbar_init(ptx::smem_u32(&a_full[i]), 2);   // one arrival per CTA (producer, or normalising warps)
                ptx::mbar_init(ptx::smem_u32(&a_land[i]), 1);   // local: raw tile landed, to be normalised
                ptx::mbar_init(ptx::smem_u32(&a_empty[i]), (uint32_t)g.sub);   // one commit per issuing warp
            }
            for (int i = 0; i < g.nb; ++i) {
                ptx::mbar_init(ptx::smem_u32(&b_full[i]), 1);
                ptx::mbar_init(ptx::smem_u32(&b_empty[i]), (uint32_t)g.sub);
            }
            for (int i = 0; i < 2; ++i) {
                ptx::mbar_init(ptx::smem_u32(&acc_full[i]), (uint32_t)g.sub);
                ptx::mbar_init(ptx::smem_u32(&acc_empty[i]), 2 * EPI_WARPS);   // one arrive per epilogue warp of BOTH CTAs
            }
            for (int i = 0; i < EPI_WARPS; ++i) ptx::mbar_init(ptx::smem_u32(&res_bar[i]), 1);
            for (int i = 0; i < g.nsc; ++i) {
                ptx::mbar_init(ptx::smem_u32(&sc_full[i]), 2);                 // one expect-tx arrival per CTA's producer
                ptx::mbar_init(ptx::smem_u32(&sc_empty[i]), (uint32_t)g.sub);
            }
            ptx::fence_barrier_init();
        }
        __syncwarp();
        ptx::tmem_alloc2(ptx::smem_u32(&tmem_base_smem), tmem_cols);
        ptx::tmem_relinquish2();
    } else if (warp == W_PROD_A && lane == 0) {
        ptx::prefetch_tensormap(&mapA0);
        if (g.c1_chunks > 0) ptx::prefetch_tensormap(&mapA1);
    } else if (warp == W_PROD_B && lane == 0) {
        ptx::prefetch_tensormap(&mapB);
    } else if (warp == W_MMA0 && lane == 0) {
        ptx::prefetch_tensormap(&mapOut);
        if (g.has_res) ptx::prefetch_tensormap(&mapRes);
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::cluster_sync();             // both CTAs' barriers are initialised before any remote signal
    ptx::tc_fence_after();
    const uint32_t tmem_base = __shfl_sync(0xffffffffu, tmem_base_smem, 0);
    const int tiles_per_img = g.tiles_h * g.tiles_w;
    // Programmatic dependent launch: everything above (barriers, TMEM, descriptor prefetch, cluster handshake) overlaps the
    // predecessor's tail.  The weight producer starts filling its ring at once (weights are constants of the graph); every
    // other role first waits until the predecessor's activations / statistics / time-embedding biases are visible.
    if (warp != W_PROD_B) pdl_wait();

    if (warp == W_PROD_A) {
        // =========================== A producer: one halo tile per channel chunk ===========================
        const bool elected = ptx::elect_one();
        // ring slot and phase are carried incrementally in every role below: `it % n`, `it / n` with a runtime n are two
        // integer divisions (~100 clk of exposed latency each) per K step on a single warp's critical path
        uint32_t s = 0, ph = 0;
        long long w_a = 0;
        DBG_T0();
        const uint32_t fb0 = ptx::mapa_rank0(ptx::smem_u32(&a_full[0]));   // leader's barriers (8 B apart)
        if (g.nsc > 0) {
            // Two rings, one warp: a cursor per ring walks (tile, chunk) on its own and issues whenever ITS slot is free, so
            // a full shortcut ring never holds back the next halo tile (and vice versa).  Shortcut tiles go straight to
            // the leader's barrier (never normalised); halo tiles take the route of the shared ring below.
            const uint32_t sfb0 = ptx::mapa_rank0(ptx::smem_u32(&sc_full[0]));
            uint32_t s2 = 0, ph2 = 0;
            int ct_h = cluster_id, i_h = 0, ct_s = cluster_id, i_s = 0;
            uint32_t spins = 0;
            while (ct_h < n_ctiles || ct_s < n_ctiles) {
                bool progress = false;
                if (ct_h < n_ctiles && __shfl_sync(0xffffffffu, ptx::mbar_test_wait(ptx::smem_u32(&a_empty[s]), ph ^ 1u), 0)) {
                    const int tile = 2 * ct_h + (int)rank;
                    const int b = tile / tiles_per_img, rem = tile % tiles_per_img;   // tile == n_tiles -> b == B: zero fill
                    const int h0 = (rem / g.tiles_w) * SUB_ROWS * g.sub, w0 = (rem % g.tiles_w) * TW;
                    const uint32_t dst = a_base + s * a_bytes;
                    if (elected) {
                        if (norm_on) {
                            ptx::mbar_arrive_expect_tx(ptx::smem_u32(&a_land[s]), a_tx);
                            ptx::tma_load_4d(dst, &mapA0, ptx::smem_u32(&a_land[s]), i_h * 64, w0 - 1, h0 - 1, b);
                        } else {
                            ptx::mbar_arrive_expect_tx_remote(fb0 + 8u * s, a_tx);
                            ptx::tma_load_4d_2sm(dst, &mapA0, fb0 + 8u * s, i_h * 64, w0 - 1, h0 - 1, b);
                        }
                    }
                    __syncwarp();
                    if (++s == (uint32_t)g.na) { s = 0; ph ^= 1u; }
                    if (++i_h == g.c0_chunks) { i_h = 0; ct_h += n_clusters; }
                    progress = true;
                }
                if (ct_s < n_ctiles && __shfl_sync(0xffffffffu, ptx::mbar_test_wait(ptx::smem_u32(&sc_empty[s2]), ph2 ^ 1u), 0)) {
                    const int tile = 2 * ct_s + (int)rank;
                    const int b = tile / tiles_per_img, rem = tile % tiles_per_img;
                    const int h0 = (rem / g.tiles_w) * SUB_ROWS * g.sub, w0 = (rem % g.tiles_w) * TW;
                    if (elected) {
                        ptx::mbar_arrive_expect_tx_remote(sfb0 + 8u * s2, a1_tx);
                        ptx::tma_load_4d_2sm(sc_base + s2 * sc_bytes, &mapA1, sfb0 + 8u * s2, i_s * 64, w0, h0, b);
                    }
                    __syncwarp();
                    if (++s2 == (uint32_t)g.nsc) { s2 = 0; ph2 ^= 1u; }
                    if (++i_s == g.c1_chunks) { i_s = 0; ct_s += n_clusters; }
                    progress = true;
                }
                if (progress) spins = 0;
                else if (++spins > (1u << 26)) asm volatile("trap;");   // a protocol bug must fault, never hang
            }
        } else
        for (int ct = cluster_id; ct < n_ctiles; ct += n_clusters) {
            const int tile = 2 * ct + (int)rank;
            const int b = tile / tiles_per_img, rem = tile % tiles_per_img;   // tile == n_tiles -> b == B: zero fill
            const int h0 = (rem / g.tiles_w) * SUB_ROWS * g.sub, w0 = (rem % g.tiles_w) * TW;
            for (int j = 0; j < n_astage; ++j) {
                const bool seg0 = !(g.seq[j] & 0x80);
                const int chunk = g.seq[j] & 0x7f;
                if (g.dbg) t0__ = clock64();
                ptx::mbar_wait(ptx::smem_u32(&a_empty[s]), ph ^ 1u);
                DBG_ADD(w_a);
                const uint32_t dst = a_base + s * a_bytes;
                if (elected) {
                    // 3x3 operand: halo origin (w0-1, h0-1), rows / columns outside the image are zero-filled == conv padding;
                    // 1x1 shortcut operand: the bare tile (8 x 16*SUB pixels)
                    if (norm_on) {
                        // tile -> this CTA's own barrier; the normalising warps publish it to the leader afterwards
                        // (shortcut tiles take the same route untouched, so every ring slot follows one protocol)
                        ptx::mbar_arrive_expect_tx(ptx::smem_u32(&a_land[s]), seg0 ? a_tx : a1_tx);
                        if (seg0) ptx::tma_load_4d(dst, &mapA0, ptx::smem_u32(&a_land[s]), chunk * 64, w0 - 1, h0 - 1, b);
                        else ptx::tma_load_4d(dst, &mapA1, ptx::smem_u32(&a_land[s]), chunk * 64, w0, h0, b);
                    } else {
                        ptx::mbar_arrive_expect_tx_remote(fb0 + 8u * s, seg0 ? a_tx : a1_tx);
                        if (seg0) ptx::tma_load_4d_2sm(dst, &mapA0, fb0 + 8u * s, chunk * 64, w0 - 1, h0 - 1, b);
                        else ptx::tma_load_4d_2sm(dst, &mapA1, fb0 + 8u * s, chunk * 64, w0, h0, b);
                    }
                }
                __syncwarp();
                if (++s == (uint32_t)g.na) { s = 0; ph ^= 1u; }
            }
        }
        if (g.dbg && elected && !norm_on) g.dbg[blockIdx.x * 8 + 6] = w_a;
    } else if (warp == W_PROD_B) {
        // =========================== B producer: weight tiles ===========================
        const bool elected = ptx::elect_one();
        uint32_t s = 0, ph = 0;
        long long w_b = 0;
        DBG_T0();
        const uint32_t fb0 = ptx::mapa_rank0(ptx::smem_u32(&b_full[0]));
        for (int ct = cluster_id; ct < n_ctiles; ct += n_clusters) {
            for (int j = 0; j < n_astage; ++j) {
                const bool seg0 = !(g.seq[j] & 0x80);
                const int chunk = g.seq[j] & 0x7f;
                const int ntap = seg0 ? 9 : 1;
                for (int tap = 0; tap < ntap; ++tap) {
                    if (g.dbg) t0__ = clock64();
                    ptx::mbar_wait(ptx::smem_u32(&b_empty[s]), ph ^ 1u);
                    DBG_ADD(w_b);
                    // K layout of the packed weights: [tap = r*3 + s][cin], then the shortcut channels
                    const int kb = seg0 ? (tap * g.c0_chunks + chunk) : (9 * g.c0_chunks + chunk);
                    if (elected) {
                        if (rank == 0) ptx::mbar_arrive_expect_tx(ptx::smem_u32(&b_full[s]), 2 * b_bytes);
                        ptx::tma_load_3d_2sm(b_base + s * b_bytes, &mapB, fb0 + 8u * s, kb * 64, n_off + (int)rank * (g.N / 2), 0);
                    }
                    __syncwarp();
                    if (++s == (uint32_t)g.nb) { s = 0; ph ^= 1u; }
                }
            }
        }
        if (g.dbg && elected && !norm_on) g.dbg[blockIdx.x * 8 + 7] = w_b;
    } else if (warp == W_MMA0 || warp == W_MMA1) {
        // =========================== MMA issuers (leader CTA only) ===========================
        // One issuing warp per sub-tile (accumulator): measured (profiles/r01_mma_probe.md), the issuing thread's
        // barrier waits do not overlap its own MMAs -- tcgen05.mma issue blocks while the pipe is busy -- so with
        // 64-clock MMAs (N=128) a single issuer leaves the pipe idle ~30 % of the time.  Two independent streams
        // into different accumulators interleave in the pipe and cover each other's waits; results do not depend
        // on the interleaving.  The whole warp walks the loops (uniform control flow, descriptors in uniform
        // registers); one elected lane issues the MMAs and the commits.
        const int u = warp - W_MMA0;
        if (rank == 0 && u < g.sub) {
            const uint32_t idesc = ptx::umma_idesc_bf16(256, (uint32_t)g.N);
            const bool elected = ptx::elect_one();
            uint32_t sa = 0, pha = 0, sb = 0, phb = 0, ssc = 0, phsc = 0, itt = 0;
            long long w_a = 0, w_b = 0, w_acc = 0;
            const long long t_start = g.dbg ? clock64() : 0;
            DBG_T0();
            for (int ct = cluster_id; ct < n_ctiles; ct += n_clusters, ++itt) {
                const uint32_t buf = g.acc_bufs == 2 ? (itt & 1u) : 0u;
                const uint32_t use = g.acc_bufs == 2 ? (itt >> 1) : itt;   // how often this buffer was used before
                if (g.dbg) t0__ = clock64();
                ptx::mbar_wait(ptx::smem_u32(&acc_empty[buf]), (use & 1u) ^ 1u);
                DBG_ADD(w_acc);
                const uint32_t d = tmem_base + buf * acc_cols + (uint32_t)(u * g.N);
                for (int j = 0; j < n_astage; ++j) {
                    const bool seg0 = !(g.seq[j] & 0x80);
                    const bool own_ring = !seg0 && g.nsc > 0;      // shortcut tile from the shortcut ring
                    if (g.dbg) t0__ = clock64();
                    if (own_ring) ptx::mbar_wait(ptx::smem_u32(&sc_full[ssc]), phsc);
                    else ptx::mbar_wait(ptx::smem_u32(&a_full[sa]), pha);
                    DBG_ADD(w_a);
                    const uint32_t tile_base = own_ring ? sc_base + ssc * sc_bytes : a_base + sa * a_bytes;
                    const int ntap = seg0 ? 9 : 1;
                    for (int t = 0; t < ntap; ++t) {
                        const uint32_t r = (uint32_t)t / 3u, sft = (uint32_t)t - 3u * r;
                        const uint64_t db = ptx::umma_desc_k_sw128(b_base + sb * b_bytes);
                        const uint32_t acc = (j > 0 || t > 0) ? 1u : 0u;
                        // 3x3: first pixel row of this sub-tile's tap window in the halo tile, 8-row groups 10 rows apart;
                        // 1x1 shortcut: the bare tile, sub-tile u starts at row 16*8*u, groups 8 rows apart
                        const uint32_t row0 = seg0 ? (r + (uint32_t)(SUB_ROWS * u)) * HALO_W + sft : (uint32_t)(SUB_ROWS * TW * u);
                        const uint64_t da = umma_desc_rows(tile_base + row0 * ROW_B, (seg0 ? HALO_W : TW) * ROW_B);
                        if (g.dbg) t0__ = clock64();
                        ptx::mbar_wait(ptx::smem_u32(&b_full[sb]), phb);
                        DBG_ADD(w_b);
                        ptx::tc_fence_after();
                        if (elected) {
                            ptx::mma_bf16_ss_2sm(d, da, db, idesc, acc);
                            ptx::mma_bf16_ss_2sm(d, da + 2, db + 2, idesc, 1u);
                            ptx::mma_bf16_ss_2sm(d, da + 4, db + 4, idesc, 1u);
                            ptx::mma_bf16_ss_2sm(d, da + 6, db + 6, idesc, 1u);
                            ptx::mma_commit_2sm(ptx::smem_u32(&b_empty[sb]));
                        }
                        __syncwarp();
                        if (++sb == (uint32_t)g.nb) { sb = 0; phb ^= 1u; }
                    }
                    if (own_ring) {
                        if (elected) ptx::mma_commit_2sm(ptx::smem_u32(&sc_empty[ssc]));
                        if (++ssc == (uint32_t)g.nsc) { ssc = 0; phsc ^= 1u; }
                    } else {
                        if (elected) ptx::mma_commit_2sm(ptx::smem_u32(&a_empty[sa]));
                        if (++sa == (uint32_t)g.na) { sa = 0; pha ^= 1u; }
                    }
                }
                if (elected) ptx::mma_commit_2sm(ptx::smem_u32(&acc_full[buf]));
                __syncwarp();
            }
            if (g.dbg && elected && u == 0) {
                g.dbg[blockIdx.x * 8 + 0] = w_a;
                g.dbg[blockIdx.x * 8 + 1] = w_b;
                if (!norm_on) g.dbg[blockIdx.x * 8 + 2] = w_acc;
                g.dbg[blockIdx.x * 8 + 3] = clock64() - t_start;
            }
        }
    } else if (warp >= NORM_WARP0) {
        // =========================== GroupNorm + SiLU on the operand in flight ===========================
        // y = silu(x * scale[b,c] + shift[b,c]) (ncsnpp_utils/layerspp.py:245,266) applied in place to every raw halo
        // tile: 256 threads, thread = (16-byte chunk q of 8 channels, row group), rows strided by 32.  Pixels outside
        // the image stay zero (the convolution pads the NORMALISED activation).  Same arithmetic as gn_apply_kernel.
        if (norm_on) {
            const int tid = (warp - NORM_WARP0) * 32 + lane;
            const uint32_t q = (uint32_t)(tid & 7);
            const int rg = tid >> 3;
            const int rows_total = (SUB_ROWS * g.sub + 2) * HALO_W;
            const uint32_t fb0 = ptx::mapa_rank0(ptx::smem_u32(&a_full[0]));
            uint32_t s = 0, ph = 0;
            long long w_land = 0, t_xf = 0, t_sync = 0;
            DBG_T0();
            for (int ct = cluster_id; ct < n_ctiles; ct += n_clusters) {
                const int tile = 2 * ct + (int)rank;
                const int b = tile / tiles_per_img, rem = tile % tiles_per_img;
                const int h0 = (rem / g.tiles_w) * SUB_ROWS * g.sub, w0 = (rem % g.tiles_w) * TW;
                for (int j = 0; j < n_astage; ++j) {
                    if ((g.seq[j] & 0x80) && g.nsc > 0) continue;        // shortcut tiles bypass the halo ring
                    const bool live = (b < g.B) && !(g.seq[j] & 0x80);   // the 1x1 shortcut operand is used raw
                    const int chunk = g.seq[j] & 0x7f;
                    // h = x * (scale/2) + shift/2  ==  (x*scale + shift)/2 exactly;  silu(t) = h + h*tanh(h)  (silu_f)
                    float sc[8], sh[8];
                    if (live) {
                        const float4* pa = reinterpret_cast<const float4*>(g.scsh + ((int64_t)b * 2) * g.norm_c + chunk * 64 + q * 8);
                        const float4* pc = reinterpret_cast<const float4*>(g.scsh + ((int64_t)b * 2 + 1) * g.norm_c + chunk * 64 + q * 8);
                        const float4 a0 = __ldg(pa), a1 = __ldg(pa + 1), c0 = __ldg(pc), c1 = __ldg(pc + 1);
                        sc[0] = a0.x; sc[1] = a0.y; sc[2] = a0.z; sc[3] = a0.w; sc[4] = a1.x; sc[5] = a1.y; sc[6] = a1.z; sc[7] = a1.w;
                        sh[0] = c0.x; sh[1] = c0.y; sh[2] = c0.z; sh[3] = c0.w; sh[4] = c1.x; sh[5] = c1.y; sh[6] = c1.z; sh[7] = c1.w;
#pragma unroll
                        for (int i = 0; i < 8; ++i) { sc[i] *= 0.5f; sh[i] *= 0.5f; }
                    }
                    if (g.dbg) t0__ = clock64();
                    ptx::mbar_wait(ptx::smem_u32(&a_land[s]), ph);
                    DBG_ADD(w_land);
                    // rows advance by 32 (a multiple of 8): the swizzle term of this thread's chunk never changes
                    const uint32_t addr0 = a_base + s * a_bytes + (uint32_t)rg * ROW_B + ((q ^ ((uint32_t)rg & 7u)) << 4);
                    if (live) {
                        const bool interior = h0 >= 1 && h0 + SUB_ROWS * g.sub + 1 <= g.H && w0 >= 1 && w0 + TW + 1 <= g.W;
                        // NR rows per trip: independent dependency chains hide the LDS / MUFU latency (only two normalising
                        // warps share a scheduler, so instruction-level parallelism has to come from within the thread)
                        constexpr int NR = 4;
                        for (int r = rg; r < rows_total; r += 32 * NR) {
                            bool ok[NR];
                            uint4 raw[NR];
#pragma unroll
                            for (int k = 0; k < NR; ++k) {
                                const int rr = r + 32 * k;
                                ok[k] = rr < rows_total;
                                if (!interior) {   // border tile: padding pixels stay zero
                                    const int hh = rr / HALO_W, ww = rr - hh * HALO_W;
                                    const int ih = h0 - 1 + hh, iw = w0 - 1 + ww;
                                    ok[k] = ok[k] && ih >= 0 && ih < g.H && iw >= 0 && iw < g.W;
                                }
                                if (ok[k]) raw[k] = ptx::lds128(addr0 + (uint32_t)(rr - rg) * ROW_B);
                            }
#pragma unroll
                            for (int k = 0; k < NR; ++k) {
                                if (ok[k]) {
                                    const uint32_t w[4] = {raw[k].x, raw[k].y, raw[k].z, raw[k].w};
                                    uint4 o;
                                    uint32_t* ow = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
                                    for (int i = 0; i < 4; ++i) {
                                        const float h0f = fmaf(__uint_as_float(w[i] << 16), sc[2 * i], sh[2 * i]);
                                        const float h1f = fmaf(__uint_as_float(w[i] & 0xffff0000u), sc[2 * i + 1], sh[2 * i + 1]);
                                        float t0, t1;
                                        asm("tanh.approx.f32 %0, %1;" : "=f"(t0) : "f"(h0f));
                                        asm("tanh.approx.f32 %0, %1;" : "=f"(t1) : "f"(h1f));
                                        const __nv_bfloat162 pk = __floats2bfloat162_rn(fmaf(h0f, t0, h0f), fmaf(h1f, t1, h1f));
                                        ow[i] = *reinterpret_cast<const uint32_t*>(&pk);
                                    }
                                    ptx::sts128(addr0 + (uint32_t)(r + 32 * k - rg) * ROW_B, o);
                                }
                            }
                        }
                    }
                    DBG_ADD(t_xf);
                    ptx::fence_proxy_async();                       // generic-proxy writes -> visible to the tensor core
                    asm volatile("bar.sync 1, 256;" ::: "memory");   // all eight normalising warps are done with the tile
                    if (tid == 0) ptx::mbar_arrive_remote(fb0 + 8u * s);
                    DBG_ADD(t_sync);
                    if (++s == (uint32_t)g.na) { s = 0; ph ^= 1u; }
                }
            }
            if (g.dbg && tid == 0) {   // measurement builds: replaces the producers' counters
                g.dbg[blockIdx.x * 8 + 6] = w_land;
                g.dbg[blockIdx.x * 8 + 7] = t_xf;
                g.dbg[blockIdx.x * 8 + 2] = t_sync;
            }
        }
    } else if (warp < EPI_WARPS) {
        // =========================== epilogue ===========================
        const int e = warp, quarter = warp & 3, half = e >> 2;
        const int n_pass = g.N >> 7;                   // passes of 64 channels per column half
        const int half_cols = g.N >> 1;
        const bool elected = ptx::elect_one();
        const uint32_t my_stg = stg_base + (uint32_t)(e * g.stg_bufs) * 4096u;
        const uint32_t my_rbar = ptx::smem_u32(&res_bar[e]);
        const uint32_t row_off = (uint32_t)lane * ROW_B, sw = (uint32_t)(lane & 7);
        float* bs = reinterpret_cast<float*>(smem_raw + (bs_base - ptx::smem_u32(smem_raw))) + e * (half_cols < 32 ? 32 : half_cols);
        uint32_t itt = 0, cnt = 0, rphase = 0;
        int last_b = -1;
        long long w_full = 0, t_body = 0;
        const int units = g.N >> 2;
        DBG_T0();
        for (int ct = cluster_id; ct < n_ctiles; ct += n_clusters, ++itt) {
            const int tile = 2 * ct + (int)rank;
            const int b = tile / tiles_per_img, rem = tile % tiles_per_img;
            const int h0 = (rem / g.tiles_w) * SUB_ROWS * g.sub, w0 = (rem % g.tiles_w) * TW;
            const uint32_t buf = g.acc_bufs == 2 ? (itt & 1u) : 0u;
            const uint32_t use = g.acc_bufs == 2 ? (itt >> 1) : itt;
            if (g.out4) {
                // Thin output convolution (C -> 4, the pyramid heads of ncsnpp.py:350-366): N = 16 accumulator columns
                // of which 4 are real; fp32 result + bias (+ the up-sampled pyramid) written straight from registers.
                // Column half h of the warp grid takes sub-tile h.
                ptx::mbar_wait(ptx::smem_u32(&acc_full[buf]), use & 1u);
                ptx::tc_fence_after();
                if (half < g.sub) {
                    const int hh = h0 + SUB_ROWS * half + 4 * quarter + (lane >> 3), ww = w0 + (lane & 7);
                    uint32_t v[4];
                    ptx::tmem_ld_32x32_x4(tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * acc_cols + (uint32_t)(half * g.N), v);
                    ptx::tmem_ld_wait();
                    if (b < g.B && hh < g.H && ww < g.W) {
                        const int64_t pix = ((int64_t)b * g.H + hh) * g.W + ww;
                        float4 r = make_float4(__uint_as_float(v[0]) + __ldg(g.bias), __uint_as_float(v[1]) + __ldg(g.bias + 1),
                                               __uint_as_float(v[2]) + __ldg(g.bias + 2), __uint_as_float(v[3]) + __ldg(g.bias + 3));
                        if (g.addend4) {
                            const float4 ad = __ldg(g.addend4 + pix);
                            r.x += ad.x; r.y += ad.y; r.z += ad.z; r.w += ad.w;
                        }
                        g.out4[pix] = r;
                    }
                }
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive_remote(ptx::mapa_rank0(ptx::smem_u32(&acc_empty[buf])));
                continue;
            }
            if (b != last_b) {   // new image: refresh this warp's slice of the per-channel additive term
                last_b = b;
                const int bb = b < g.B ? b : g.B - 1;
                __syncwarp();
                for (int i = lane; i < half_cols; i += 32) {
                    const int ch = n_off + half * half_cols + i;
                    float v = g.bias ? __ldg(g.bias + ch) : 0.f;
                    if (g.tbias) v += __ldg(g.tbias + (int64_t)bb * g.tb_stride + ch);
                    bs[i] = v * g.scale;
                }
                __syncwarp();
            }
            if (g.dbg) t0__ = clock64();
            ptx::mbar_wait(ptx::smem_u32(&acc_full[buf]), use & 1u);
            DBG_ADD(w_full);
            ptx::tc_fence_after();
            // GroupNorm sums of this tile (pass 0 / 1), already in fixed point: integer adds keep them independent of SUB
            unsigned long long tile_s0 = 0, tile_q0 = 0, tile_s1 = 0, tile_q1 = 0;
            for (int u = 0; u < g.sub; ++u) {
                const int hrow = h0 + SUB_ROWS * u + 4 * quarter;   // this warp's four image rows (32 pixels)
                for (int p = 0; p < n_pass; ++p, ++cnt) {
                    const int cl = 64 * p, cbase = half * half_cols + cl;   // column within the half / the tensor
                    const uint32_t stg = my_stg + (g.stg_bufs == 2 ? (cnt & 1u) * 4096u : 0u);
                    // the TMA store that last read this staging tile has drained it
                    if (elected) {
                        if (g.stg_bufs == 2) ptx::bulk_wait_group_read<1>(); else ptx::bulk_wait_group_read<0>();
                    }
                    __syncwarp();
                    if (g.has_res && elected) {
                        ptx::mbar_arrive_expect_tx(my_rbar, 4096u);
                        ptx::tma_load_4d(stg, &mapRes, my_rbar, n_off + cbase, w0, hrow, b);
                    }
                    const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * acc_cols + (uint32_t)(u * g.N + cbase);
                    float us[16], uq[16];   // this pixel's unit sums / sums of squares for the 64 channels of the pass
                    const bool pix_ok = b < g.B && (hrow + (lane >> 3)) < g.H && (w0 + (lane & 7)) < g.W;
#pragma unroll
                    for (int hq = 0; hq < 2; ++hq) {   // 32 accumulator columns at a time (register budget: 640 threads)
                        uint32_t v[32];
                        ptx::tmem_ld_32x32(taddr + 32u * hq, v);
                        ptx::tmem_ld_wait();
                        if (hq == 0 && g.has_res) {
                            ptx::mbar_wait(my_rbar, rphase);
                            rphase ^= 1u;
                        }
#pragma unroll
                        for (int qq = 0; qq < 4; ++qq) {
                            const int q = 4 * hq + qq;
                            const float4 b0 = *reinterpret_cast<const float4*>(bs + cl + 8 * q);
                            const float4 b1 = *reinterpret_cast<const float4*>(bs + cl + 8 * q + 4);
                            float f[8];
                            f[0] = fmaf(__uint_as_float(v[8 * qq + 0]), g.scale, b0.x);
                            f[1] = fmaf(__uint_as_float(v[8 * qq + 1]), g.scale, b0.y);
                            f[2] = fmaf(__uint_as_float(v[8 * qq + 2]), g.scale, b0.z);
                            f[3] = fmaf(__uint_as_float(v[8 * qq + 3]), g.scale, b0.w);
                            f[4] = fmaf(__uint_as_float(v[8 * qq + 4]), g.scale, b1.x);
                            f[5] = fmaf(__uint_as_float(v[8 * qq + 5]), g.scale, b1.y);
                            f[6] = fmaf(__uint_as_float(v[8 * qq + 6]), g.scale, b1.z);
                            f[7] = fmaf(__uint_as_float(v[8 * qq + 7]), g.scale, b1.w);
                            const uint32_t addr = stg + row_off + (((uint32_t)q ^ sw) << 4);   // 128-byte swizzle
                            if (g.has_res) {
                                float rr[8];
                                unpack8(ptx::lds128(addr), rr);
#pragma unroll
                                for (int i = 0; i < 8; ++i) f[i] = fmaf(rr[i], g.scale, f[i]);
                            }
                            ptx::sts128(addr, pack8(f));
                            if (g.ustats) {
                                us[2 * q] = (f[0] + f[1]) + (f[2] + f[3]);
                                us[2 * q + 1] = (f[4] + f[5]) + (f[6] + f[7]);
                                uq[2 * q] = fmaf(f[0], f[0], f[1] * f[1]) + fmaf(f[2], f[2], f[3] * f[3]);
                                uq[2 * q + 1] = fmaf(f[4], f[4], f[5] * f[5]) + fmaf(f[6], f[6], f[7] * f[7]);
                            }
                        }
                    }
                    if (g.ustats) {
                        if (!pix_ok) {
#pragma unroll
                            for (int i = 0; i < 16; ++i) us[i] = uq[i] = 0.f;
                        }
                        // warp totals over its 32 pixels (fixed order), then exact integer accumulation: the statistics
                        // do not depend on which CTA handled which tile
                        const float ts = warp_transpose_reduce16(us, lane), tq = warp_transpose_reduce16(uq, lane);
                        if (p == 0) { tile_s0 += gn_fix_sum(ts); tile_q0 += gn_fix_sq(tq); }
                        else { tile_s1 += gn_fix_sum(ts); tile_q1 += gn_fix_sq(tq); }
                    }
                    ptx::fence_proxy_async();
                    __syncwarp();
                    if (elected) {
                        ptx::tma_store_4d(&mapOut, stg, n_off + cbase, w0, hrow, b);
                        ptx::bulk_commit_group();
                    }
                }
            }
            // all TMEM reads of this accumulator set are complete: hand it back to the MMA warp
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive_remote(ptx::mapa_rank0(ptx::smem_u32(&acc_empty[buf])));
            if (g.ustats && !(lane & 1) && b < g.B) {   // lane l holds unit ((l>>1)&15) of each 64-channel pass
                unsigned long long* dst = g.ustats + ((int64_t)b * (g.n_total >> 2) + (n_off >> 2) + half * (units >> 1) + ((lane >> 1) & 15)) * 2;
                atomicAdd(dst, tile_s0);
                atomicAdd(dst + 1, tile_q0);
                if (n_pass == 2) {
                    atomicAdd(dst + 32, tile_s1);
                    atomicAdd(dst + 33, tile_q1);
                }
            }
            DBG_ADD(t_body);
        }
        if (elected) ptx::bulk_wait_group_read<0>();   // staging tiles must outlive the last stores' reads
        if (g.dbg && threadIdx.x == 0) {
            g.dbg[blockIdx.x * 8 + 4] = w_full;
            g.dbg[blockIdx.x * 8 + 5] = t_body;
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::cluster_sync();             // the peer's TMEM / smem stay valid until the leader's last MMA retired
    if (warp == W_MMA1) {
        __syncwarp();
        ptx::tmem_dealloc2(tmem_base, tmem_cols);
    }
}

int g_num_sms2 = 0;

int device_num_sms() {
    if (g_num_sms2 == 0) {
        int dev = 0;
        SNRSE_CUDA(cudaGetDevice(&dev));
        SNRSE_CUDA(cudaDeviceGetAttribute(&g_num_sms2, cudaDevAttrMultiProcessorCount, dev));
    }
    return g_num_sms2;
}

// Zeroes the plan and fills in what both plans share: the tiling (SUB, tile counts), the N split, the TMEM
// accumulator count and the persistent grid.
void halo_plan_tiles(ConvHaloPlan* p, int B, int H, int W, int C0, int n_rows, int num_sms) {
    memset(p, 0, sizeof(*p));
    const int tiles_w = cdiv(W, TW);
    int sub = 2;
    if (H < 2 * SUB_ROWS || (int64_t)B * cdiv(H, 2 * SUB_ROWS) * tiles_w < num_sms) sub = 1;
    p->sub = sub;
    p->c0_chunks = C0 / 64;
    p->B = B; p->H = H; p->W = W;
    p->tiles_h = cdiv(H, SUB_ROWS * sub);
    p->tiles_w = tiles_w;
    p->n_tiles = B * p->tiles_h * p->tiles_w;
    // N-split: with so few pixel tiles that twice as many clusters still fit the GPU, every tile is computed by two
    // clusters, 128 output channels each (half the MMA and weight-tile time per cluster on the latency-bound small maps)
    const int n_ctiles = (p->n_tiles + 1) / 2, max_clusters = num_sms / 2;
    p->nsplit = (n_rows == 256 && 2 * n_ctiles <= max_clusters) ? 2 : 1;
    p->n_total = n_rows;
    p->N = n_rows / p->nsplit;
    p->acc_bufs = (sub * p->N <= 256) ? 2 : 1;
    p->grid = p->nsplit == 2 ? 4 * n_ctiles : 2 * (n_ctiles < max_clusters ? n_ctiles : max_clusters);
}
}  // namespace
extern long long* g_halo_dbg_shared;

bool conv_halo2_fits(int H, int W) { return W >= TW && H >= 8; }

bool conv_halo2_eligible(int H, int W, int taps0, int n_rows) {
    return taps0 == 9 && conv_halo2_fits(H, W) && (n_rows == 128 || n_rows == 256);
}

int conv_halo2_plan_shape(ConvHaloPlan* p, int B, int H, int W, int C0, int C1, int n_rows, int norm, int num_sms) {
    SNRSE_CHECK_ARG(conv_halo2_eligible(H, W, 9, n_rows), "conv_halo2: shape not eligible");
    SNRSE_CHECK_ARG(C0 % 64 == 0 && C1 % 64 == 0, "conv_halo2: channel counts must be multiples of 64");
    SNRSE_CHECK_ARG(C0 / 64 + C1 / 64 <= 16, "conv_halo2: at most 16 channel chunks (1024 channels)");
    halo_plan_tiles(p, B, H, W, C0, n_rows, num_sms);
    p->c1_chunks = C1 / 64;
    const int sub = p->sub, n_loc = p->N;
    const int a_bytes = (int)halo_stage_bytes(sub), b_bytes = (n_loc / 2) * 128;
    // dynamic shared memory (static: barriers + per-warp bias slices, ~4.3 KB)
    const int budget = 220 * 1024;
    // One A slot feeds 9 taps x SUB x 4 MMAs (>= 2300 clk): two slots hide the next tile's load.  With in-flight
    // normalisation the slot also waits for the normalising warps (load + ~2500 clk); at N=128 (64-clock MMAs) that
    // needs a third slot, paid for with single-buffered epilogue staging.
    int na = 2, stg = 2, nsc = 0;
    if (norm && n_loc == 128 && sub == 2) { na = 3; stg = 1; }
    int nb = (budget - na * a_bytes - stg * EPI_WARPS * 4096) / b_bytes;
    if (nb < 6 && stg == 2) {
        stg = 1;
        nb = (budget - na * a_bytes - stg * EPI_WARPS * 4096) / b_bytes;
    }
    if (nb > MAX_B) nb = MAX_B;
    SNRSE_CHECK_ARG(nb >= 4, "conv_halo2: shared memory budget");
    if (na < MAX_A && (budget - (na + 1) * a_bytes - stg * EPI_WARPS * 4096 - nb * b_bytes) >= 0) ++na;
    // Fused 1x1 shortcut: its operand tiles (16 KB per sub-tile, one 4-MMA group each) go through a ring of their own and
    // are interleaved with the 3x3 chunks in the K loop (conv_halo2_launch).  In the shared ring every shortcut stage
    // (512 clk of MMA work at N = 128) waited a full load latency for its slot: 40-45 % of the MMA warp's time
    // (profiles/r02_conv_ncu.md).  Two halo slots + two shortcut slots + a shorter weight ring need the whole 227 KB.
    // Only for the 128-output-channel layers (where N = 128 whatever the batch): the K order then depends on the layer alone,
    // never on the batch-dependent tiling, so results stay batch-invariant bit for bit.  The 256-channel layers keep the
    // shared ring: at N = 256 / SUB = 2 two extra slots leave room for only two weight slots.
    if (C1 > 0 && n_rows == 128) {
        const int sc_bytes = SUB_ROWS * sub * TW * 128;
        const int limit = 227 * 1024 - 1024 /*alignment*/ - 768 /*static: barriers*/ - (int)halo_bsum_bytes(n_loc);
        const int nb2 = (limit - 2 * a_bytes - MAX_SC * sc_bytes - EPI_WARPS * 4096) / b_bytes;
        if (nb2 >= 4) { na = 2; nsc = MAX_SC; stg = 1; nb = nb2 > MAX_B ? MAX_B : nb2; }
    }
    p->na = na; p->nb = nb; p->stg_bufs = stg; p->nsc = nsc;
    p->smem_bytes = na * a_bytes + nsc * SUB_ROWS * sub * TW * 128 + nb * b_bytes + stg * EPI_WARPS * 4096 +
                    (int)halo_bsum_bytes(n_loc) + 1024;
    return SNRSE_OK;
}

int conv_halo2_make_plan(ConvHaloPlan* p, const ActView* a0, const ActView* a1, const bf16* wt, int n_rows,
                         const float* bias, const float* tbias, int tb_stride, const ActView* res, float scale, bf16* out,
                         int out_ld, const float* scsh, unsigned long long* ustats) {
    SNRSE_CHECK_ARG(a0->ld % 8 == 0, "conv_halo2: the operand pitch must be a multiple of 8");
    SNRSE_CHECK_ARG(!a1 || (a1->ld % 8 == 0 && a1->H == a0->H && a1->W == a0->W && a1->B == a0->B),
                    "conv_halo2: bad shortcut operand");
    SNRSE_CHECK_ARG(out_ld % 8 == 0 && (!res || res->ld % 8 == 0), "conv_halo2: pitches must be multiples of 8");
    SNRSE_TRY(conv_halo2_plan_shape(p, a0->B, a0->H, a0->W, a0->C, a1 ? a1->C : 0, n_rows, scsh != nullptr,
                                    device_num_sms()));
    const int sub = p->sub, n_loc = p->N;
    p->bias = bias; p->tbias = tbias; p->tb_stride = tb_stride;
    p->res = res ? res->ptr : nullptr; p->res_ld = res ? res->ld : 0;
    p->scale = scale; p->out = out; p->out_ld = out_ld;
    p->scsh = scsh;
    p->ustats = ustats;
    const int box_h = SUB_ROWS * sub + 2;
    SNRSE_TRY(tma_make_act_map(&p->mapA0, a0->ptr, a0->C, a0->W, a0->H, a0->B, a0->ld, 64, HALO_W, box_h));
    if (a1) SNRSE_TRY(tma_make_act_map(&p->mapA1, a1->ptr, a1->C, a1->W, a1->H, a1->B, a1->ld, 64, TW, SUB_ROWS * sub));
    else p->mapA1 = p->mapA0;
    const int64_t ktot = 64 * (int64_t)(9 * p->c0_chunks + p->c1_chunks);
    SNRSE_TRY(tma_make_wt_map(&p->mapB, wt, ktot, n_rows, 1, ktot * n_rows, 64, n_loc / 2));
    // epilogue tiles: 32 pixels (4 image rows x 8) x 64 channels
    SNRSE_TRY(tma_make_act_map(&p->mapOut, out, n_rows, a0->W, a0->H, a0->B, out_ld, 64, TW, 4));
    if (res) SNRSE_TRY(tma_make_act_map(&p->mapRes, res->ptr, n_rows, a0->W, a0->H, a0->B, res->ld, 64, TW, 4));
    else p->mapRes = p->mapOut;
    return SNRSE_OK;
}

// Thin output convolution on the same kernel: 3x3, C -> 4 (weights packed as 16 rows, rows 4..15 zero), optional
// GroupNorm+SiLU of the operand in flight, fp32 output [B,H,W,4] = conv + bias (+ addend4).
int conv_halo2_plan_shape_out4(ConvHaloPlan* p, int B, int H, int W, int C0, int num_sms) {
    SNRSE_CHECK_ARG(conv_halo2_fits(H, W) && C0 % 64 == 0 && C0 / 64 <= 16, "conv_halo2 out4: shape not eligible");
    halo_plan_tiles(p, B, H, W, C0, 16, num_sms);
    p->na = 3; p->nb = MAX_B; p->stg_bufs = 0;   // no epilogue staging: the result leaves from registers
    p->smem_bytes = p->na * (int)halo_stage_bytes(p->sub) + p->nb * 1024 + (int)halo_bsum_bytes(16) + 1024;
    return SNRSE_OK;
}

int conv_halo2_make_plan_out4(ConvHaloPlan* p, const ActView* a0, const bf16* wt16, const float* bias4, const float* addend4,
                              float* out4, const float* scsh) {
    SNRSE_CHECK_ARG(a0->ld % 8 == 0, "conv_halo2 out4: the operand pitch must be a multiple of 8");
    SNRSE_CHECK_ARG(bias4 && out4, "conv_halo2 out4: null pointer");
    SNRSE_TRY(conv_halo2_plan_shape_out4(p, a0->B, a0->H, a0->W, a0->C, device_num_sms()));
    const int sub = p->sub;
    p->bias = bias4; p->scale = 1.0f;
    p->scsh = scsh;
    p->out4 = out4; p->addend4 = addend4;
    SNRSE_TRY(tma_make_act_map(&p->mapA0, a0->ptr, a0->C, a0->W, a0->H, a0->B, a0->ld, 64, HALO_W, SUB_ROWS * sub + 2));
    p->mapA1 = p->mapA0; p->mapOut = p->mapA0; p->mapRes = p->mapA0;
    const int64_t ktot = 64 * (int64_t)(9 * p->c0_chunks);
    SNRSE_TRY(tma_make_wt_map(&p->mapB, wt16, ktot, 16, 1, ktot * 16, 64, 8));
    return SNRSE_OK;
}

int conv_halo2_launch(const ConvHaloPlan* p, cudaStream_t s) {
    static bool attr_set = false;
    if (!attr_set) {
        cudaFuncAttributes fa;
        SNRSE_CUDA(cudaFuncGetAttributes(&fa, conv_halo2_kernel));
        SNRSE_CHECK_ARG(fa.sharedSizeBytes <= 768, "conv_halo2: static shared memory grew past the plan's allowance");
        SNRSE_CUDA(cudaFuncSetAttribute(conv_halo2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        227 * 1024 - (int)fa.sharedSizeBytes));
        attr_set = true;
    }
    Halo2Args g;
    g.c0_chunks = p->c0_chunks; g.c1_chunks = p->c1_chunks;
    {   // K-loop order.  Shared ring: the 3x3 chunks, then the 1x1 shortcut chunks (interleaving them there was measured
        // and did not help: the 3x3 tile that follows two shortcut tiles has only 1024 clk of MMA work to hide its load
        // behind).  Separate shortcut ring: the shortcut chunks are spread evenly behind the 3x3 chunks (c s s c s s for
        // 128 + 256 channels), so a shortcut slot has a whole 3x3 stage to reload.  The packed weights keep their
        // [taps x 3x3 channels | shortcut channels] K layout either way; the first stage is always a 3x3 chunk.
        int n = 0;
        if (p->nsc > 0) {
            int done = 0;
            for (int i = 0; i < p->c0_chunks; ++i) {
                g.seq[n++] = (unsigned char)i;
                const int upto = (int)((int64_t)(i + 1) * p->c1_chunks / p->c0_chunks);
                for (; done < upto; ++done) g.seq[n++] = (unsigned char)(0x80 | done);
            }
        } else {
            for (int i = 0; i < p->c0_chunks; ++i) g.seq[n++] = (unsigned char)i;
            for (int i = 0; i < p->c1_chunks; ++i) g.seq[n++] = (unsigned char)(0x80 | i);
        }
        for (; n < 16; ++n) g.seq[n] = 0;
    }
    g.H = p->H; g.W = p->W; g.B = p->B;
    g.sub = p->sub; g.tiles_h = p->tiles_h; g.tiles_w = p->tiles_w; g.n_tiles = p->n_tiles;
    g.N = p->N; g.nsplit = p->nsplit; g.n_total = p->n_total; g.na = p->na; g.nb = p->nb; g.nsc = p->nsc; g.acc_bufs = p->acc_bufs; g.stg_bufs = p->stg_bufs;
    g.has_res = p->res != nullptr;
    g.bias = p->bias; g.tbias = p->tbias; g.tb_stride = p->tb_stride;
    g.scale = p->scale;
    g.scsh = p->scsh; g.norm_c = p->c0_chunks * 64;
    g.ustats = p->ustats;
    g.out4 = reinterpret_cast<float4*>(p->out4); g.addend4 = reinterpret_cast<const float4*>(p->addend4);
    g.dbg = g_halo_dbg_shared;
    snrse_launch_m(2, conv_halo2_kernel, dim3(p->grid), dim3(HALO_THREADS + (p->scsh ? NORM_THREADS : 0)), p->smem_bytes, s, p->mapA0, p->mapA1, p->mapB, p->mapOut, p->mapRes, g);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}
