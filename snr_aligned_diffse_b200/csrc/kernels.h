// Host-side launcher declarations shared by the C-ABI layer (api.cu) and the NCSN++ executor (engine.cu).
// All launchers enqueue on the given stream, never allocate, never synchronise (graph-capturable).
#pragma once
#include <cuda.h>

#include "common.cuh"

// A view of an activation tensor in NHWC order: element (b,h,w,c) lives at
// ptr[((b*H + h)*W + w)*ld + c].  ld > C when the tensor is a channel slice of a concat buffer.
struct ActView {
    bf16* ptr;
    int B, H, W, C, ld;
};

// ----------------------------------------------------------------------------- conv_gemm.cu
// Implicit-GEMM convolution on tcgen05:  out[m, n] = epilogue( sum_k A[m, k] * Wt[n, k] )
//   m = output pixel (b,h,w);  k = (tap, cin) of segment 0 followed by cin of segment 1 (1x1);
//   epilogue: (+bias[n]) (+tbias[b*tb_stride + n]) (+res[m, n]) * scale  -> bf16 or f32.
struct ConvGemmPlan {
    CUtensorMap mapA0, mapA1, mapB;
    int taps0;       // 9 (3x3, pad 1) or 1
    int c0_chunks;   // Cin0 / 64
    int c1_chunks;   // Cin1 / 64 (0: no second segment)
    int B, H, W;     // output pixels
    int th_log2, tw_log2, tiles_h, tiles_w;
    int N, n_tile;   // output columns, columns per CTA (64 / 128 / 256)
    int b_batched;   // 1: operand B has one matrix per batch item (attention), 0: shared weights
    const float* bias;   // [N] or null
    const float* tbias;  // [B, tb_stride] or null
    int tb_stride;
    const bf16* res;  // residual view or null
    int res_ld;
    float scale;
    void* out;
    int out_ld;
    int out_f32;  // 0: bf16, 1: f32
    int stages;
    int a_box_bytes;  // bytes per activation TMA box (box height = min(tile rows, H))
    int smem_bytes;
    int small;        // few pixel tiles: 64-column N tiles and a deep ring
};
// a0: segment-0 input view (taps0 taps); a1: optional segment-1 input (1 tap, may be null).
// wt: [n_rows, Ktot] bf16, K-major, Ktot = (taps0*C0 + C1); for b_batched the matrix of batch b starts at
// wt + b*wt_batch_stride elements.
int conv_gemm_make_plan(ConvGemmPlan* p, const ActView* a0, int taps0, const ActView* a1, const bf16* wt, int n_rows,
                        int64_t wt_batch_stride, int b_batched, const float* bias, const float* tbias, int tb_stride,
                        const ActView* res, float scale, void* out, int out_ld, int out_f32);
// same with an explicit pitch (elements) between the rows of wt (0: dense) -- attention operands inside a fused qkv buffer
int conv_gemm_make_plan_ex(ConvGemmPlan* p, const ActView* a0, int taps0, const ActView* a1, const bf16* wt, int n_rows,
                           int64_t wt_batch_stride, int b_batched, const float* bias, const float* tbias, int tb_stride,
                           const ActView* res, float scale, void* out, int out_ld, int out_f32, int64_t wt_row_pitch);
int conv_gemm_launch(const ConvGemmPlan* p, cudaStream_t s);
// The shape-only part of conv_gemm_make_plan_ex: tile shape, N tile, small-map mode, ring depth and shared memory of a
// convolution of a B x H x W map (C0 channels, taps0 taps, C1 shortcut channels) to n_rows outputs on num_sms SMs.
// Touches no device and no tensor map; conv_gemm_make_plan_ex calls it with the device's SM count.
int conv_gemm_plan_shape(ConvGemmPlan* p, int B, int H, int W, int taps0, int C0, int C1, int n_rows, int num_sms);

// ----------------------------------------------------------------------------- conv_halo2.cu
// Plan of the persistent 2-CTA halo-reuse kernel: 3x3 convolutions with W >= 8, H >= 8, N in {128, 256}.
struct ConvHaloPlan {
    CUtensorMap mapA0, mapA1, mapB, mapOut, mapRes;   // mapOut / mapRes: 2-CTA kernel only (TMA epilogue)
    int c0_chunks, c1_chunks, B, H, W, sub, tiles_h, tiles_w, n_tiles, N, na, nb, acc_bufs, stg_bufs, grid, smem_bytes;
    int nsplit, n_total;   // 2-CTA kernel: N = n_total / nsplit output channels per cluster (nsplit 2 on small maps)
    int nsc;               // 2-CTA kernel: slots of the separate ring for the 1x1 shortcut operand (0: it shares the halo ring)
    const float* bias;
    const float* tbias;
    int tb_stride;
    const bf16* res;
    int res_ld;
    float scale;
    bf16* out;
    int out_ld;
    const float* scsh;            // GroupNorm scale / shift table of operand 0, or null
    unsigned long long* ustats;
    float* out4;                  // 2-CTA kernel, thin C -> 4 output convolution only
    const float* addend4;
};
// 2-CTA (cta_group::2) single-halo-tile version, same plan structure (conv_halo2.cu).  Its tiles need an H x W map with
// W >= 8, H >= 8; conv_halo2_make_plan also needs a 3x3 convolution with N in {128, 256}.
bool conv_halo2_fits(int H, int W);
bool conv_halo2_eligible(int H, int W, int taps0, int n_rows);
// scsh (nullable): GroupNorm scale/shift [B][2][C0] (gn_finalize_launch); when given, operand 0 is replaced by
// silu(x*scale + shift) inside the kernel (GroupNorm+SiLU+conv3x3 of ResnetBlockBigGANpp without the HBM round trip).
int conv_halo2_make_plan(ConvHaloPlan* p, const ActView* a0, const ActView* a1, const bf16* wt, int n_rows,
                         const float* bias, const float* tbias, int tb_stride, const ActView* res, float scale, bf16* out,
                         int out_ld, const float* scsh, unsigned long long* ustats);
// ustats (nullable): the epilogue also accumulates the GroupNorm sums of the result into [B][N/4][2] (zeroed by the
// caller; gn_finalize_launch source format), so the following GroupNorm needs no pass over the tensor.
int conv_halo2_launch(const ConvHaloPlan* p, cudaStream_t s);
// The shape-only parts of conv_halo2_make_plan (norm: operand normalised in flight) and conv_halo2_make_plan_out4: SUB,
// tiles, N split, accumulator buffers, ring depths, shortcut ring, persistent grid and shared memory on num_sms SMs.
// They touch no device and no tensor map; the make_plan functions call them with the device's SM count.
int conv_halo2_plan_shape(ConvHaloPlan* p, int B, int H, int W, int C0, int C1, int n_rows, int norm, int num_sms);
int conv_halo2_plan_shape_out4(ConvHaloPlan* p, int B, int H, int W, int C0, int num_sms);

// Thin 3x3 output convolution C -> 4 on the 2-CTA kernel (N = 16, weights [16][9*C] bf16 with rows 4..15 zero), fp32
// result [B,H,W,4] = conv + bias4 (+ addend4); scsh as above.  Needs W >= 8, H >= 8.
int conv_halo2_make_plan_out4(ConvHaloPlan* p, const ActView* a0, const bf16* wt16, const float* bias4, const float* addend4,
                              float* out4, const float* scsh);

// The integer fields of either convolution plan, as the debug entry points report them (snrse_conv_plan of
// include/snrse_b200_plans.h mirrors this struct); fields of the other kernel stay 0.
struct ConvPlanFields {
    int sub, nsplit, n_loc, acc_bufs, na, nb, stg_bufs, nsc;   // 2-CTA kernel (n_loc: output channels per cluster)
    int th, tw, n_tile, small, stages;                         // single-CTA implicit GEMM
    int tiles_h, tiles_w, n_tiles, grid, smem_bytes;           // both (grid: CTAs launched, GEMM: both grid dimensions)
};
inline ConvPlanFields conv_plan_fields(const ConvHaloPlan& p) {
    ConvPlanFields f{};
    f.sub = p.sub; f.nsplit = p.nsplit; f.n_loc = p.N; f.acc_bufs = p.acc_bufs;
    f.na = p.na; f.nb = p.nb; f.stg_bufs = p.stg_bufs; f.nsc = p.nsc;
    f.tiles_h = p.tiles_h; f.tiles_w = p.tiles_w; f.n_tiles = p.n_tiles; f.grid = p.grid; f.smem_bytes = p.smem_bytes;
    return f;
}
inline ConvPlanFields conv_plan_fields(const ConvGemmPlan& p) {
    ConvPlanFields f{};
    f.th = 1 << p.th_log2; f.tw = 1 << p.tw_log2; f.n_tile = p.n_tile; f.small = p.small; f.stages = p.stages;
    f.tiles_h = p.tiles_h; f.tiles_w = p.tiles_w; f.n_tiles = p.B * p.tiles_h * p.tiles_w;
    f.grid = f.n_tiles * cdiv(p.N, p.n_tile); f.smem_bytes = p.smem_bytes;
    return f;
}

// ----------------------------------------------------------------------------- conv_simt.cu
// Reference-grade direct convolution on CUDA cores (debug / cross-check path, fp32 accumulate).
int conv_simt_launch(const ActView* a0, int taps0, const ActView* a1, const bf16* wt, int N, const float* bias,
                     const float* tbias, int tb_stride, const ActView* res, float scale, bf16* out, int out_ld,
                     cudaStream_t s);
// x4: [B,H,W,4] f32 -> out bf16 view, 3x3 pad 1, w: [Cout][3][3][4] f32
int conv_in4_launch(const float* x4, const float* w, const float* bias, const ActView* out, cudaStream_t s);
// a: bf16 view (C) -> out4 [B,H,W,4] f32 = conv3x3(a) + bias (+ addend4), w: [4][3][3][C] f32
int conv_out4_launch(const ActView* a, const float* w, const float* bias, const float* addend4, float* out4,
                     cudaStream_t s);
// out = h + W[C x 4] * p4 + bias      (Combine 'sum' with a 1x1 conv on the 4-channel input pyramid)
int combine4_launch(const float* p4, const ActView* h, const float* w, const float* bias, const ActView* out,
                    cudaStream_t s);

// ----------------------------------------------------------------------------- norm.cu
// Statistics per 4-channel unit: ustats [B][U][2] (U = C/4) 64-bit fixed-point (sum, sum of squares), ACCUMULATED
// with integer atomics into a buffer the caller zeroed (gn_fixed.cuh):
//   gn_stats_launch   : stand-alone pass over x
//   gn_finalize_launch: one source (U1 = 0) or two (GroupNorm over the channel concatenation [src0 | src1]);
//                       scsh: [B][2][C] f32 (scale, shift), C = 4*(U0+U1)
int gn_stats_launch(const ActView* x, unsigned long long* ustats, cudaStream_t s);
int gn_finalize_launch(const unsigned long long* src0, int U0, const unsigned long long* src1, int U1, int B,
                       int64_t count_per_group, const float* gamma, const float* beta, float eps, float* scsh,
                       cudaStream_t s);
int gn_apply_launch(const ActView* x, const float* scsh, int silu, const ActView* out, cudaStream_t s);

// ----------------------------------------------------------------------------- fir.cu
int fir_up2_launch(const ActView* x, const ActView* out, cudaStream_t s);
int fir_down2_launch(const ActView* x, const ActView* out, cudaStream_t s);
// out_n = FIR(silu(GroupNorm(x))) and out_r = FIR(x) in one pass over x (up / down residual blocks)
int fir_dual_launch(const ActView* x, const ActView* out_n, const ActView* out_r, int up, const float* scsh, cudaStream_t s);
int fir_up2_f4_launch(const float* x, float* out, int B, int H, int W, cudaStream_t s);      // in [B,H,W,4]
int fir_down2_f4_launch(const float* x, float* out, int B, int H, int W, cudaStream_t s);    // in [B,H,W,4]
// general upfirdn2d on fp32 planes [major][in_h][in_w] (op/upfirdn2d.cpp:12-23)
int upfirdn2d_launch(const float* x, const float* kernel, float* out, int64_t major, int in_h, int in_w, int kh, int kw,
                     int up_x, int up_y, int down_x, int down_y, int pad_x0, int pad_x1, int pad_y0, int pad_y1,
                     cudaStream_t s);

// ----------------------------------------------------------------------------- attention.cu
// q,k,v: [B, n, C] bf16 views (tokens = H*W); scores: [B, n, n] f32 workspace; o: bf16 view.
// workspace: attention_workspace_bytes(B, n, C): scores f32 [B,n,n] | probabilities bf16 [B,n,n] | V^T bf16 [B,C,n].
// n % 64 == 0 and C % 64 == 0: Q K^T and P V run on the tensor cores (conv_gemm.cu, batched operand B), softmax in
// fp32 in between; otherwise (the 4 x T/64 bottleneck of short inputs) fp32 CUDA-core kernels.
int64_t attention_workspace_bytes(int B, int n, int C);
int attention_launch(const ActView* q, const ActView* k, const ActView* v, void* workspace, const ActView* o,
                     cudaStream_t s, int allow_tensor_cores = 1);

// ----------------------------------------------------------------------------- temb.cu
// t: [B]; fourier_w [nf]; w1 [4nf][2nf], b1; w2 [4nf][4nf], b2; dense_w [rows][4nf], dense_b [rows]
// scratch: B*10*nf floats (act(temb) [B][4nf], Fourier features [B][2nf], hidden [B][4nf]); tb_out: [B][rows]
int temb_launch(const float* t, int B, int nf, const float* fourier_w, const float* w1, const float* b1,
                const float* w2, const float* b2, const float* dense_w, const float* dense_b, int rows, float* scratch,
                float* tb_out, cudaStream_t s);

// ----------------------------------------------------------------------------- sampler.cu
// x, y, out: complex64 [B, F*T]; x4: [B,F,T,4] f32 = (re x, im x, re y, im y)
int pack_input_launch(const float2* x, const float2* y, float* x4, int B, int64_t n, cudaStream_t s);
// same + x64: [B,F,T,64] bf16 (hi/lo split of the 4 channels in 0..7, zeros above) for the tensor-core input convolution
int pack_input64_launch(const float2* x, const float2* y, float* x4, bf16* x64, int B, int64_t n, cudaStream_t s);
// out = alpha_b * xres + beta_b * (Wout * (p4 / t_b) + bout); mode 0: alpha=0,beta=1; 1: sebridge precond; 2: alpha=0,beta=-1
int final_launch(const float* p4, const float* t, const float* w, const float* bias, const float2* xres, float2* out,
                 int B, int64_t n, int mode, cudaStream_t s);
// out_mean = a*x + b*y + c*s ; out_x = out_mean + d*z   (per-batch coefficient arrays, any pointer may alias)
int lincomb_launch(const float2* x, const float2* y, const float2* sc, const float2* z, const float* a, const float* b,
                   const float* c, const float* d, float2* out_mean, float2* out_x, int B, int64_t n, cudaStream_t s);
int lincomb_keyed_launch(const float2* x, const float2* y, const float2* sc, const float* a, const float* b,
                         const float* c, const float* d, const unsigned long long* keys, unsigned long long seed,
                         const int* len, int tpad, float2* z_out, float2* out_mean, float2* out_x, int B, int64_t n,
                         cudaStream_t s);

// embedded Runge-Kutta helpers of the on-device ODE sampler (coef: nk host floats; K: nk stages of n complex values)
int rk_combine_launch(const float2* y, const float2* K, int nk, int64_t n, float h, const float* coef, float2* out,
                      cudaStream_t s);
int rk_partials(int64_t n);
int rk_scaled_sqnorm_launch(const float2* K, int nk, int64_t n, float h, const float* coef, const float2* y,
                            const float2* y2, float atol, float rtol, double* partial, cudaStream_t s);

// SNR -> (snapped t, norm factor): ratio[b] = noise/clean amplitude ratio, peak[b] = max|y|, t30: 30 doubles (device)
int v3_scalars_launch(const float* ratio, const float* peak, double snr_scale, float nf_const, const double* t30,
                      float* t_out, float* nf_out, int* idx_out, int B, cudaStream_t s);
// n/(s+n) sigmoid output of the SNR estimator -> n/s  (model.py:720-721)
int snr_ratio_launch(const float* g, float* ratio, int B, cudaStream_t s);

// ----------------------------------------------------------------------------- stft.cu
int stft_launch(const float* wave, const int* len, const float* scale, int scale_is_divisor, float* out, int B,
                int lstride, int tpad, int transform, float alpha, float beta, int planar, cudaStream_t s);
int spec_transform_launch(const float2* in, float2* out, int64_t n, int inverse, int transform, float alpha, float beta,
                          cudaStream_t s);
int absmax_launch(const float* wave, const int* len, int B, int lstride, float* out, cudaStream_t s);
int si_sdr_launch(const float* ref, const float* est, const int* len, int B, int lstride, double* out, cudaStream_t s);
int istft_launch(const float2* spec, const int* len, const float* scale, float* wave, float* frames_ws, int B,
                 int lstride, int tpad, int transform, float alpha, float beta, cudaStream_t s);
