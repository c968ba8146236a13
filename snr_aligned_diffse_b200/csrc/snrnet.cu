// SNR estimator forward pass (reduced PESQNet) on CUDA cores, fp32.
// Replaces `SNRNet.forward` (sgmse-bbed/sgmse/backbones/snrnet.py:47-97): the STFT is split into
// 16-frame clusters; per cluster conv5x5(2->32,p2) -> maxpool 2x2 -> conv3x3(32->32,p1) -> maxpool (2,1)
// -> four (64 x k) convolutions, k = 1,2,4,8, each max-pooled over time -> 128 features; a BiLSTM(128->128)
// runs over the clusters; [mean, unbiased std, min, max] over clusters -> Linear(1024->1) -> sigmoid.
// ~1.2 MMAC per STFT frame (0.1 % of the score network): plain SIMT kernels, no tensor cores.
// Ragged batches: every kernel takes an optional clusters[B] (the valid 16-frame clusters of each item, clamped to
// [1, S]); the clusters of an item from there on are neither computed nor read, so item b gives the bits it gives when
// run alone at T16 = 16 * clusters[b].  The layouts stay dense ([B][2][256][T16] features, B*S workspace rows).
#include "kernels.h"

namespace {

struct SnrParam {
    const char* name;
    int ndim;
    int64_t dims[4];
    int64_t numel;
};
const SnrParam kParams[] = {
    {"dnn.conv5x5_1.weight", 4, {32, 2, 5, 5}, 32 * 2 * 25},          {"dnn.conv5x5_1.bias", 1, {32, 1, 1, 1}, 32},
    {"dnn.conv3x3_1.weight", 4, {32, 32, 3, 3}, 32 * 32 * 9},         {"dnn.conv3x3_1.bias", 1, {32, 1, 1, 1}, 32},
    {"dnn.convt_1.weight", 4, {32, 32, 64, 1}, 32 * 32 * 64 * 1},     {"dnn.convt_1.bias", 1, {32, 1, 1, 1}, 32},
    {"dnn.convt_2.weight", 4, {32, 32, 64, 2}, 32 * 32 * 64 * 2},     {"dnn.convt_2.bias", 1, {32, 1, 1, 1}, 32},
    {"dnn.convt_3.weight", 4, {32, 32, 64, 4}, 32 * 32 * 64 * 4},     {"dnn.convt_3.bias", 1, {32, 1, 1, 1}, 32},
    {"dnn.convt_4.weight", 4, {32, 32, 64, 8}, 32 * 32 * 64 * 8},     {"dnn.convt_4.bias", 1, {32, 1, 1, 1}, 32},
    {"dnn.blstm.weight_ih_l0", 2, {512, 128, 1, 1}, 512 * 128},       {"dnn.blstm.weight_hh_l0", 2, {512, 128, 1, 1}, 512 * 128},
    {"dnn.blstm.bias_ih_l0", 1, {512, 1, 1, 1}, 512},                 {"dnn.blstm.bias_hh_l0", 1, {512, 1, 1, 1}, 512},
    {"dnn.blstm.weight_ih_l0_reverse", 2, {512, 128, 1, 1}, 512 * 128}, {"dnn.blstm.weight_hh_l0_reverse", 2, {512, 128, 1, 1}, 512 * 128},
    {"dnn.blstm.bias_ih_l0_reverse", 1, {512, 1, 1, 1}, 512},         {"dnn.blstm.bias_hh_l0_reverse", 1, {512, 1, 1, 1}, 512},
    {"dnn.fc.weight", 2, {1, 1024, 1, 1}, 1024},                      {"dnn.fc.bias", 1, {1, 1, 1, 1}, 1},
};
constexpr int kNumParams = sizeof(kParams) / sizeof(kParams[0]);

int64_t param_offset(int i) {  // bytes, 256-aligned slots
    int64_t off = 0;
    for (int j = 0; j < i; ++j) off += (kParams[j].numel * 4 + 255) / 256 * 256;
    return off;
}
const float* P(const void* blob, int i) { return reinterpret_cast<const float*>(static_cast<const uint8_t*>(blob) + param_offset(i)); }

// Valid clusters of item b.  Clamping keeps a bad value from moving any read outside the buffers.
__device__ __forceinline__ int item_clusters(const int* __restrict__ clusters, int b, int S) {
    return clusters ? min(max(clusters[b], 1), S) : S;
}

// Bit q set: workspace row nc0 + q (cluster (nc0 + q) % S of item (nc0 + q) / S) exists and is valid.
__device__ __forceinline__ unsigned live_rows8(const int* __restrict__ clusters, int64_t nc0, int64_t ncl, int S) {
    unsigned live = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int64_t nc = nc0 + q;
        if (nc < ncl && (!clusters || (int)(nc % S) < item_clusters(clusters, (int)(nc / S), S))) live |= 1u << q;
    }
    return live;
}

__device__ __forceinline__ void cp_async4_zfill(float* smem_dst, const float* gsrc, bool valid) {
    // 4-byte asynchronous copy; !valid: nothing is read and the destination is zero-filled (src-size 0)
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc),
                 "r"(valid ? 4 : 0) : "memory");
}

// ---- conv5x5 (2->32, pad 2) + maxpool 2x2.  feat [B][2][256][T16] -> a1 [NC][32][128][8], NC = B*T16/16
// Block = one cluster x C5_TILES consecutive tiles of 16 input rows (-> 8 pooled rows each); the weights are staged once,
// the input patches are double-buffered with cp.async so that the next tile streams in while this one is computed.
// Thread = (group of 8 output channels, pooled position): the 2 x 6 x 6 input patch under its 2x2 convolution outputs
// sits in registers and every weight is ONE broadcast shared-memory load for four FMAs.  Accumulation order per output:
// bias, then c, ky, kx (as a direct loop).
constexpr int C5_TILES = 4;
__global__ void __launch_bounds__(256)
snr_conv5_pool_kernel(const float* __restrict__ feat, const float* __restrict__ w, const float* __restrict__ bias,
                      float* __restrict__ a1, int T16, const int* __restrict__ clusters) {
    pdl_sync();
    __shared__ float sw[32 * 50];
    __shared__ float sbias[32];
    __shared__ float sxb[2][2 * 20 * 20];  // two stages of the input patch: 16 freq rows (+4 halo) x 16 frames (+4 halo)
    const int nc = blockIdx.y, S = T16 / 16;
    const int b = nc / S, cl = nc % S;
    if (cl >= item_clusters(clusters, b, S)) return;   // the whole block, before its first barrier
    auto load_tile = [&](int buf, int f0) {
        for (int i = threadIdx.x; i < 2 * 20 * 20; i += 256) {
            const int c = i / 400, r = (i / 20) % 20, t = i % 20;
            const int f = f0 + r - 2, tt = t - 2;
            const bool ok = f >= 0 && f < 256 && tt >= 0 && tt < 16;
            const float* src = feat + (((int64_t)b * 2 + c) * 256 + (ok ? f : 0)) * T16 + cl * 16 + (ok ? tt : 0);
            cp_async4_zfill(&sxb[buf][i], src, ok);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    const int tile0 = blockIdx.x * C5_TILES;
    load_tile(0, tile0 * 16);
    for (int i = threadIdx.x; i < 32 * 50; i += 256) sw[i] = w[i];
    if (threadIdx.x < 32) sbias[threadIdx.x] = bias[threadIdx.x];
    const int cg = threadIdx.x >> 6, pos = threadIdx.x & 63, pr = pos >> 3, pc = pos & 7;
    for (int ti = 0; ti < C5_TILES; ++ti) {
        const int f0 = (tile0 + ti) * 16;
        if (ti + 1 < C5_TILES) {
            load_tile((ti + 1) & 1, f0 + 16);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        const float* sx = sxb[ti & 1];
        float patch[2][6][6];
#pragma unroll
        for (int c = 0; c < 2; ++c)
#pragma unroll
            for (int i = 0; i < 6; ++i)
#pragma unroll
                for (int j = 0; j < 6; ++j) patch[c][i][j] = sx[c * 400 + (2 * pr + i) * 20 + 2 * pc + j];
        for (int j = 0; j < 8; ++j) {
            const int co = cg * 8 + j;
            const float b0 = sbias[co];
            float a00 = b0, a01 = b0, a10 = b0, a11 = b0;
            const float* wc = sw + co * 50;
#pragma unroll
            for (int c = 0; c < 2; ++c)
#pragma unroll
                for (int ky = 0; ky < 5; ++ky)
#pragma unroll
                    for (int kx = 0; kx < 5; ++kx) {
                        const float wv = wc[c * 25 + ky * 5 + kx];
                        a00 = fmaf(patch[c][ky][kx], wv, a00);
                        a01 = fmaf(patch[c][ky][kx + 1], wv, a01);
                        a10 = fmaf(patch[c][ky + 1][kx], wv, a10);
                        a11 = fmaf(patch[c][ky + 1][kx + 1], wv, a11);
                    }
            a1[(((int64_t)nc * 32 + co) * 128 + (f0 / 2 + pr)) * 8 + pc] = fmaxf(fmaxf(a00, a01), fmaxf(a10, a11));
        }
        __syncthreads();   // the stage is free again before the load of the trip after next overwrites it
    }
}

// ---- conv3x3 (32->32, pad 1) + maxpool (2,1).  a1 [NC][32][128][8] -> a2 [NC][32][64][8]
// Block = one cluster x 16 conv rows x all 32 output channels.  Thread = 4 output channels x a 2x2 patch of
// conv outputs (-> 2 pooled values per channel): per input channel 16 activations + 9 weight vectors are
// loaded for 144 FMA (register tiling keeps the kernel FMA-bound instead of LDS-bound).
// A block walks C3_TILES row tiles of one cluster: the weights are staged once, the input tiles are double-buffered with
// cp.async (staging 59 KB between two barriers per 16 rows left the FMA pipe idle for about a third of a block's life).
constexpr int C3_ROWS = 16, C3_TILES = 2;
constexpr int C3_SX = 32 * 18 * 10;
constexpr int C3_SMEM = (32 * 9 * 32 + 2 * C3_SX) * 4;
__global__ void __launch_bounds__(256)
snr_conv3_pool_kernel(const float* __restrict__ a1, const float* __restrict__ w, const float* __restrict__ bias,
                      float* __restrict__ a2, int S, const int* __restrict__ clusters) {
    pdl_sync();
    extern __shared__ __align__(16) float sm3[];
    float* sw = sm3;                       // [ci][k][co]   32*9*32 floats = 36 KB
    float* sxb = sm3 + 32 * 9 * 32;        // 2 x [ci][18][10]  2 x 23 KB
    const int nc = blockIdx.y, tile0 = blockIdx.x * C3_TILES;
    if (nc % S >= item_clusters(clusters, nc / S, S)) return;   // the whole block, before its first barrier
    auto load_tile = [&](int buf, int f0) {
        float* dst = sxb + buf * C3_SX;
        for (int i = threadIdx.x; i < C3_SX; i += 256) {
            const int c = i / 180, r = (i / 10) % 18, t = i % 10;
            const int f = f0 + r - 1, tt = t - 1;
            const bool ok = f >= 0 && f < 128 && tt >= 0 && tt < 8;
            cp_async4_zfill(dst + i, a1 + (((int64_t)nc * 32 + c) * 128 + (ok ? f : 0)) * 8 + (ok ? tt : 0), ok);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    load_tile(0, tile0 * C3_ROWS);
    {   // weights pre-packed [ci][tap][co] (transform 2): a straight, conflict-free copy
        const float4* src = reinterpret_cast<const float4*>(w);
        float4* dst = reinterpret_cast<float4*>(sw);
        for (int i = threadIdx.x; i < 32 * 32 * 9 / 4; i += 256) dst[i] = __ldg(src + i);
    }
    const int cg = threadIdx.x & 7, pg = threadIdx.x >> 3;  // channel group (4 co), position group
    const int pr = pg >> 2, pc2 = pg & 3;                    // pooled row 0..7, column pair 0..3
    float bv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) bv[j] = bias[cg * 4 + j];
    for (int ti = 0; ti < C3_TILES; ++ti) {
        const int f0 = (tile0 + ti) * C3_ROWS;
        if (ti + 1 < C3_TILES) {
            load_tile((ti + 1) & 1, f0 + C3_ROWS);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        const float* sx = sxb + (ti & 1) * C3_SX;
        float acc[4][4];                                         // [co][pos: (dy,dx)]
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[j][q] = bv[j];
        for (int ci = 0; ci < 32; ++ci) {
            float xv[4][4];
#pragma unroll
            for (int r = 0; r < 4; ++r) {   // four consecutive floats at an even offset: two 8-byte loads
                const float2 lo = *reinterpret_cast<const float2*>(&sx[(ci * 18 + pr * 2 + r) * 10 + pc2 * 2]);
                const float2 hi = *reinterpret_cast<const float2*>(&sx[(ci * 18 + pr * 2 + r) * 10 + pc2 * 2 + 2]);
                xv[r][0] = lo.x; xv[r][1] = lo.y; xv[r][2] = hi.x; xv[r][3] = hi.y;
            }
#pragma unroll
            for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                for (int kx = 0; kx < 3; ++kx) {
                    const float4 wv = *reinterpret_cast<const float4*>(&sw[(ci * 9 + ky * 3 + kx) * 32 + cg * 4]);
                    const float ww[4] = {wv.x, wv.y, wv.z, wv.w};
#pragma unroll
                    for (int j = 0; j < 4; ++j)
#pragma unroll
                        for (int dy = 0; dy < 2; ++dy)
#pragma unroll
                            for (int dx = 0; dx < 2; ++dx)
                                acc[j][dy * 2 + dx] = fmaf(xv[dy + ky][dx + kx], ww[j], acc[j][dy * 2 + dx]);
                }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int dx = 0; dx < 2; ++dx)
                a2[(((int64_t)nc * 32 + cg * 4 + j) * 64 + (f0 / 2 + pr)) * 8 + pc2 * 2 + dx] =
                    fmaxf(acc[j][dx], acc[j][2 + dx]);
        __syncthreads();   // the stage is free again before a later load overwrites it
    }
}

// ---- four (64 x k) convolutions + max over time.  a2 [NC][32][64][8] -> feats [NC][128]
// Block = 8 clusters x one kernel width k; warp = cluster, lane = output channel.  Per 32-row chunk of the
// (ci,f) axis the activations [8][32][8] and weights [32][k][32 co] are staged in shared memory; a lane keeps
// the <= 8 output-frame accumulators of its channel.  A skipped cluster's stage is zero-filled instead of loaded and its
// warp stores nothing.
struct ConvtW {
    const float* w[4];
    const float* b[4];
};
__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
constexpr int CONVT_SX = 8 * 32 * 8;                       // floats of one activation stage
constexpr int CONVT_STAGE = CONVT_SX + 32 * 8 * 32;        // + the widest (k = 8) weight chunk
constexpr int CONVT_SMEM = 2 * CONVT_STAGE * 4;            // two stages, 80 KB

template <int K>   // kernel width in frames (1, 2, 4, 8): compile-time so that only the K * (9-K) useful FMAs per row are issued
__device__ __forceinline__ void snr_convt_body(const float* __restrict__ a2, const float* __restrict__ wg,
                                               const float* __restrict__ bg, float* __restrict__ feats, int ki, unsigned live,
                                               float* smem) {
    constexpr int NOUT = 9 - K;
    const int64_t nc0 = (int64_t)blockIdx.x * 8;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float acc[NOUT];
#pragma unroll
    for (int t = 0; t < NOUT; ++t) acc[t] = 0.f;
    // Two stages filled with cp.async: chunk i+1 streams in while chunk i is consumed (staging with plain loads between two
    // barriers exposed the global-memory latency 64 times per block: 287 us for the 16 x 4 s batch).
    auto load_stage = [&](int buf, int r0) {
        float* sx = smem + buf * CONVT_STAGE;
        float* sw = sx + CONVT_SX;
        for (int i = threadIdx.x; i < CONVT_SX / 4; i += 256) {     // per cluster 32 rows x 8 frames = 64 contiguous float4
            const int cl = i >> 6, q = i & 63;
            const int64_t nc = nc0 + cl;
            if ((live >> cl) & 1) cp_async16(sx + cl * 256 + q * 4, a2 + nc * 16384 + (int64_t)r0 * 8 + q * 4);
            else *reinterpret_cast<float4*>(sx + cl * 256 + q * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        // weights are pre-packed [r][dt][co]: the 32*K*32 floats of this chunk are one contiguous block
        for (int i = threadIdx.x; i < 8 * 32 * K; i += 256) cp_async16(sw + i * 4, wg + (int64_t)r0 * K * 32 + i * 4);
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    load_stage(0, 0);
    for (int it = 0; it < 64; ++it) {
        if (it + 1 < 64) {
            load_stage((it + 1) & 1, (it + 1) * 32);
            asm volatile("cp.async.wait_group 1;" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;" ::: "memory");
        }
        __syncthreads();
        const float* sx = smem + (it & 1) * CONVT_STAGE + warp * 256;
        const float* sw = smem + (it & 1) * CONVT_STAGE + CONVT_SX;
#pragma unroll 4
        for (int rr = 0; rr < 32; ++rr) {
            const float4 xa = *reinterpret_cast<const float4*>(sx + rr * 8);
            const float4 xb = *reinterpret_cast<const float4*>(sx + rr * 8 + 4);
            const float xf[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
#pragma unroll
            for (int dt = 0; dt < K; ++dt) {
                const float wv = sw[(rr * K + dt) * 32 + lane];
#pragma unroll
                for (int t = 0; t < NOUT; ++t) acc[t] = fmaf(xf[t + dt], wv, acc[t]);
            }
        }
        __syncthreads();      // everyone is done with this stage before the load issued in the next trip overwrites it
    }
    float best = -INFINITY;
#pragma unroll
    for (int t = 0; t < NOUT; ++t) best = fmaxf(best, acc[t]);
    if ((live >> warp) & 1) feats[(nc0 + warp) * 128 + ki * 32 + lane] = best + bg[lane];
}

__global__ void __launch_bounds__(256)
snr_convt_kernel(const float* __restrict__ a2, ConvtW cw, float* __restrict__ feats, int64_t ncl, int S,
                 const int* __restrict__ clusters) {
    pdl_sync();
    extern __shared__ __align__(16) float convt_smem[];
    const unsigned live = live_rows8(clusters, (int64_t)blockIdx.x * 8, ncl, S);
    if (!live) return;                               // uniform over the block, before its first barrier
    const int ki = blockIdx.y;                       // weights packed [r (2048)][dt (k)][co (32)]
    if (ki == 0) snr_convt_body<1>(a2, cw.w[0], cw.b[0], feats, 0, live, convt_smem);
    else if (ki == 1) snr_convt_body<2>(a2, cw.w[1], cw.b[1], feats, 1, live, convt_smem);
    else if (ki == 2) snr_convt_body<4>(a2, cw.w[2], cw.b[2], feats, 2, live, convt_smem);
    else snr_convt_body<8>(a2, cw.w[3], cw.b[3], feats, 3, live, convt_smem);
}

// ---- LSTM input projections for both directions: pre[dir][B*S][512] = W_ih x + b_ih + b_hh
// Block = 8 rows (clusters); thread = 4 gate rows; a weight row is read once per 8 inputs.  Skipped clusters are
// computed on zeros and not stored.
__global__ void __launch_bounds__(256)
snr_lstm_pre_kernel(const float* __restrict__ feats, const float* __restrict__ wih0, const float* __restrict__ bih0,
                    const float* __restrict__ bhh0, const float* __restrict__ wih1, const float* __restrict__ bih1,
                    const float* __restrict__ bhh1, float* __restrict__ pre, int64_t rows, int S,
                    const int* __restrict__ clusters) {
    pdl_sync();
    __shared__ float sx[8][128];
    const int64_t row0 = (int64_t)blockIdx.x * 8;
    const unsigned live = live_rows8(clusters, row0, rows, S);
    if (!live) return;                               // uniform over the block, before its barrier
    for (int i = threadIdx.x; i < 8 * 128; i += 256) {
        const int64_t row = row0 + (i >> 7);
        sx[i >> 7][i & 127] = ((live >> (i >> 7)) & 1) ? feats[row * 128 + (i & 127)] : 0.f;
    }
    __syncthreads();
    for (int o = threadIdx.x; o < 1024; o += 256) {
        const int dir = o >> 9, g = o & 511;
        const float4* wr = reinterpret_cast<const float4*>((dir ? wih1 : wih0) + (int64_t)g * 128);
        const float b0 = (dir ? bih1 : bih0)[g] + (dir ? bhh1 : bhh0)[g];
        float acc[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[q] = b0;
        for (int j = 0; j < 32; ++j) {
            const float4 wv = __ldg(wr + j);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                acc[q] = fmaf(wv.x, sx[q][4 * j], acc[q]);
                acc[q] = fmaf(wv.y, sx[q][4 * j + 1], acc[q]);
                acc[q] = fmaf(wv.z, sx[q][4 * j + 2], acc[q]);
                acc[q] = fmaf(wv.w, sx[q][4 * j + 3], acc[q]);
            }
        }
#pragma unroll
        for (int q = 0; q < 8; ++q)
            if ((live >> q) & 1) pre[((int64_t)dir * rows + row0 + q) * 512 + g] = acc[q];
    }
}

// ---- recurrence: one block per (batch item, direction); thread g owns gate row g of W_hh
// (64 weights in registers, 64 in shared memory).  Gate order i, f, g, o (torch.nn.LSTM).  The forward direction runs
// over clusters 0 .. Sb-1, the reverse one from Sb-1 down to 0 (Sb = the item's valid clusters).
__global__ void __launch_bounds__(512, 1)
snr_lstm_rec_kernel(const float* __restrict__ pre, const float* __restrict__ whh0, const float* __restrict__ whh1,
                    float* __restrict__ hout, int S, int64_t rows, const int* __restrict__ clusters) {
    pdl_sync();
    extern __shared__ float sm[];
    float* sw = sm;                  // [64][512]  second half of every W_hh row, transposed
    float* sh = sm + 64 * 512;       // [128] h
    float* sg = sh + 128;            // [512] gates
    const int b = blockIdx.x, dir = blockIdx.y, g = threadIdx.x;
    const float* wr = (dir ? whh1 : whh0) + (int64_t)g * 128;
    float wreg[64];
#pragma unroll
    for (int j = 0; j < 64; ++j) wreg[j] = wr[j];
    for (int j = 0; j < 64; ++j) sw[j * 512 + g] = wr[64 + j];
    if (g < 128) sh[g] = 0.f;
    float c = 0.f;
    const int Sb = item_clusters(clusters, b, S);
    __syncthreads();
    for (int step = 0; step < Sb; ++step) {
        const int s = dir ? Sb - 1 - step : step;
        float acc = pre[((int64_t)dir * rows + (int64_t)b * S + s) * 512 + g];
#pragma unroll
        for (int j = 0; j < 64; ++j) acc = fmaf(wreg[j], sh[j], acc);
#pragma unroll 8
        for (int j = 0; j < 64; ++j) acc = fmaf(sw[j * 512 + g], sh[64 + j], acc);
        sg[g] = acc;
        __syncthreads();
        if (g < 128) {
            const float ig = 1.f / (1.f + expf(-sg[g]));
            const float fg = 1.f / (1.f + expf(-sg[128 + g]));
            const float gg = tanhf(sg[256 + g]);
            const float og = 1.f / (1.f + expf(-sg[384 + g]));
            c = fg * c + ig * gg;
            const float h = og * tanhf(c);
            sh[g] = h;
            hout[((int64_t)b * S + s) * 256 + dir * 128 + g] = h;
        }
        __syncthreads();
    }
}

// ---- [mean, unbiased std, min, max] over the item's valid clusters -> fc -> sigmoid
__global__ void __launch_bounds__(256)
snr_head_kernel(const float* __restrict__ hout, const float* __restrict__ fcw, const float* __restrict__ fcb,
                float* __restrict__ out, int S, const int* __restrict__ clusters) {
    pdl_sync();
    __shared__ float red[8];
    const int b = blockIdx.x, j = threadIdx.x;
    const int Sb = item_clusters(clusters, b, S);
    float sum = 0.f, mn = INFINITY, mx = -INFINITY;
    for (int s = 0; s < Sb; ++s) {
        const float v = hout[((int64_t)b * S + s) * 256 + j];
        sum += v;
        mn = fminf(mn, v);
        mx = fmaxf(mx, v);
    }
    const float mean = sum / (float)Sb;
    float ss = 0.f;
    for (int s = 0; s < Sb; ++s) {
        const float d = hout[((int64_t)b * S + s) * 256 + j] - mean;
        ss = fmaf(d, d, ss);
    }
    const float sd = sqrtf(ss / (float)(Sb - 1));  // Sb == 1 -> NaN, as torch.std (snrnet.py:84)
    float acc = mean * fcw[j] + sd * fcw[256 + j] + mn * fcw[512 + j] + mx * fcw[768 + j];
    acc = warp_sum(acc);
    if ((j & 31) == 0) red[j >> 5] = acc;
    __syncthreads();
    if (j == 0) {
        float t = fcb[0];
        for (int i = 0; i < 8; ++i) t += red[i];
        out[b] = 1.f / (1.f + expf(-t));
    }
}

}  // namespace

extern "C" {

int snrse_snrnet_num_params(void) { return kNumParams; }

int snrse_snrnet_param_info(int i, char* name, int name_cap, int64_t* offset, int64_t* numel, int* transform) {
    SNRSE_CHECK_ARG(i >= 0 && i < kNumParams, "snrnet_param_info: index out of range");
    const int n = (int)strlen(kParams[i].name);
    SNRSE_CHECK_ARG(n + 1 <= name_cap, "snrnet_param_info: name buffer too small");
    memcpy(name, kParams[i].name, n + 1);
    *offset = param_offset(i);
    *numel = kParams[i].numel;
    // transform 1: [co][ci][f][dt] is stored as [r = ci*64 + f][dt][co] (co fastest): the layout snr_convt_kernel stages
    // transform 2: conv3x3 [co][ci][3][3] stored as [ci][tap][co]
    *transform = (i >= 4 && i <= 10 && (i % 2) == 0) ? 1 : (i == 2 ? 2 : 0);
    return SNRSE_OK;
}

int snrse_snrnet_param_shape(int i, int64_t* dims, int* ndim) {
    SNRSE_CHECK_ARG(i >= 0 && i < kNumParams, "snrnet_param_shape: index out of range");
    for (int j = 0; j < 4; ++j) dims[j] = kParams[i].dims[j];
    *ndim = kParams[i].ndim;
    return SNRSE_OK;
}

int64_t snrse_snrnet_weight_bytes(void) { return param_offset(kNumParams); }

// a1 [NC][32][128][8] | a2 [NC][32][64][8] | feats [NC][128] | pre [2][NC][512] | hout [NC][256]
int64_t snrse_snrnet_workspace_bytes(int B, int T16) {
    const int64_t nc = (int64_t)B * (T16 / 16);
    return nc * (32768 + 16384 + 128 + 1024 + 256) * 4;
}

int snrse_snrnet_forward_varlen(const void* weights, const float* feat, const int* clusters, float* out, int B, int T16,
                                void* workspace, void* stream) {
    SNRSE_CHECK_ARG(weights && feat && out && workspace, "snrnet_forward: null pointer");
    SNRSE_CHECK_ARG(B > 0 && T16 > 0 && T16 % 16 == 0, "snrnet_forward: T must be a positive multiple of 16");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int S = T16 / 16;
    const int64_t nc = (int64_t)B * S;
    float* a1 = static_cast<float*>(workspace);
    float* a2 = a1 + nc * 32768;
    float* feats = a2 + nc * 16384;
    float* pre = feats + nc * 128;
    float* hout = pre + nc * 1024;
    static bool attr_set = false;
    if (!attr_set) {
        SNRSE_CUDA(cudaFuncSetAttribute(snr_conv3_pool_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, C3_SMEM));
        SNRSE_CUDA(cudaFuncSetAttribute(snr_lstm_rec_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (64 * 512 + 128 + 512) * 4));
        SNRSE_CUDA(cudaFuncSetAttribute(snr_convt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CONVT_SMEM));
        attr_set = true;
    }
    snrse_launch(snr_conv5_pool_kernel, dim3(dim3(16 / C5_TILES, (unsigned)nc)), dim3(256), 0, s, feat, P(weights, 0), P(weights, 1), a1, T16, clusters);
    SNRSE_LAUNCH_CHECK();
    snrse_launch(snr_conv3_pool_kernel, dim3(dim3(128 / (C3_ROWS * C3_TILES), (unsigned)nc)), dim3(256), C3_SMEM, s, 
        a1, P(weights, 2), P(weights, 3), a2, S, clusters);
    SNRSE_LAUNCH_CHECK();
    ConvtW cw;
    for (int i = 0; i < 4; ++i) {
        cw.w[i] = P(weights, 4 + 2 * i);
        cw.b[i] = P(weights, 5 + 2 * i);
    }
    snrse_launch(snr_convt_kernel, dim3(dim3((unsigned)cdiv64(nc, 8), 4)), dim3(256), CONVT_SMEM, s, a2, cw, feats, nc, S, clusters);
    SNRSE_LAUNCH_CHECK();
    snrse_launch(snr_lstm_pre_kernel, dim3((unsigned)cdiv64(nc, 8)), dim3(256), 0, s, feats, P(weights, 12), P(weights, 14), P(weights, 15), P(weights, 16),
                                                     P(weights, 18), P(weights, 19), pre, nc, S, clusters);
    SNRSE_LAUNCH_CHECK();
    snrse_launch(snr_lstm_rec_kernel, dim3(dim3(B, 2)), dim3(512), (64 * 512 + 128 + 512) * 4, s, pre, P(weights, 13), P(weights, 17), hout, S, nc, clusters);
    SNRSE_LAUNCH_CHECK();
    snrse_launch(snr_head_kernel, dim3(B), dim3(256), 0, s, hout, P(weights, 20), P(weights, 21), out, S, clusters);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}

int snrse_snrnet_forward(const void* weights, const float* feat, float* out, int B, int T16, void* workspace,
                         void* stream) {
    return snrse_snrnet_forward_varlen(weights, feat, nullptr, out, B, T16, workspace, stream);
}

}  // extern "C"
