/* snrse_b200.h -- C ABI of the B200-native (sm_100a) SNR-aligned diffusion speech-enhancement hot path.
 *
 * The reference (yh-jun/SNR-Aligned_diffSE) has no FFI of its own for this path except the
 * `upfirdn2d` pybind op; its boundary is the Python API of `sgmse` (SURVEY.md 8b).  This header is
 * the boundary a binding would target instead: plain pointers, sizes and a stream, int status
 * codes, no torch types.  Every function enqueues work on `stream` (a cudaStream_t passed as
 * void*), never allocates device memory, never synchronises and never reads device memory on the
 * host, so a whole enhancement pass can be captured in a CUDA graph.  All pointers are DEVICE
 * pointers unless stated otherwise.  Status: 0 = ok; otherwise see SNRSE_ERR_* and
 * snrse_last_error().  There is no CPU fallback.
 *
 * Each entry point cites the reference code it replaces (paths under sgmse-bbed/sgmse/).
 */
#ifndef SNRSE_B200_H
#define SNRSE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SNRSE_OK 0
#define SNRSE_ERR_ARG 1
#define SNRSE_ERR_CUDA 2
#define SNRSE_ERR_STATE 3
#define SNRSE_ERR_UNSUPPORTED 4

int snrse_version(void);
const char* snrse_last_error(void);       /* thread-local message of the last failing call */
int snrse_device_check(void);             /* 0 iff the current device is compute capability 10.x */
long long snrse_launch_count(void);       /* kernels launched by this library since it was loaded */
/* Programmatic dependent launch (griddepcontrol.launch_dependents / .wait in every kernel): `mask` selects the launches that
 * carry the programmatic-stream-serialization attribute, i.e. may become resident while their predecessor in the stream /
 * captured graph drains (prologue, TMEM allocation and the weight ring's first loads overlap the predecessor's tail; results
 * are unchanged).  bit0: the memory-bound / small kernels, bit1: the two tcgen05 convolution kernels, bit2: the GroupNorm
 * finalize launches alone (measured neutral).  Read at launch
 * (== graph capture) time.  Returns the previous mask; mask < 0 only queries.  Default: environment variable SNRSE_PDL when
 * set, else 2 (measured on the graphed 16 x 4 s step: 0 -> 20.13 ms, 2 -> 20.00 ms, 1 and 3 -> +0.1 ms; profiles/r02_step_ab.md). */
int snrse_set_pdl(int mask);
/* Measurement / debug entry points (per-launch-group timing, activation taps, cycle counters) are NOT part of this
 * ABI: they are declared in snrse_b200_debug.h. */

/* ---------------------------------------------------------------- signal front / back end ------
 * snrse_stft: SpecsDataModule.stft + spec_fwd + pad_spec (data_module.py:241-254,291-293;
 *   util/other.py:83-99) and the raw SNR-branch STFT + pad_spec_16 (model.py:715-719).
 *   wave [B][lstride] f32; len[b] valid samples (NULL: lstride); scale[b] optional per-utterance
 *   factor (divisor when scale_is_divisor, i.e. y / norm_factor).  n_fft 510, hop 128, periodic
 *   Hann, center/reflect.  out: complex64 [B][256][tpad] (planar=0) or f32 [B][2][256][tpad]
 *   (planar=1, re/im channels).  Frames >= 1 + len/128 are zero.  transform: 0 none,
 *   1 "exponent" beta*|X|^alpha*e^{i arg X}, 2 "log" beta*log(1+|X|)*e^{i arg X} (data_module.py:241-251). */
int snrse_stft(const float* wave, const int* len, const float* scale, int scale_is_divisor, void* out, int B,
               int lstride, int tpad, int transform, float alpha, float beta, int planar, void* stream);
/* snrse_istft: spec_back + SpecsDataModule.istft + output rescale (data_module.py:256-267,295-297;
 *   model.py:612-613,828-830).  spec complex64 [B][256][tpad]; wave[b][n] written for n < lstride
 *   (zeros for n >= len[b]); scale[b] multiplies the output.  workspace: snrse_istft_workspace_bytes. */
int64_t snrse_istft_workspace_bytes(int B, int tpad);
int snrse_istft(const void* spec, const int* len, const float* scale, float* wave, void* workspace, int B, int lstride,
                int tpad, int transform, float alpha, float beta, void* stream);
/* stand-alone spec_fwd (inverse=0) / spec_back (inverse=1) on n complex64 values (data_module.py:241-267);
 *   transform 1 "exponent" / 2 "log" as above */
int snrse_spec_transform(const void* in, void* out, int64_t n, int inverse, int transform, float alpha, float beta,
                         void* stream);
/* max|y| per utterance (model.py:715,726) */
int snrse_absmax(const float* wave, const int* len, int B, int lstride, float* out, void* stream);
/* SI-SDR in dB of est[b][0..len[b]) against ref[b] (util/other.py:71-75; B/eval.py:140-144), double accumulation */
int snrse_si_sdr(const float* ref, const float* est, const int* len, int B, int lstride, double* out, void* stream);

/* ---------------------------------------------------------------- SNR -> timestep --------------
 * calculate_snr_direct + t_30 snap + calculate_normfac_direct (model.py:22-23,627-634,726-740):
 *   ratio[b] = noise/clean; snr_scale = 10^0.25*fixed_snr; nf_const = 2.040166*sqrt(0.240253+0.759747*fixed_snr^2);
 *   t30 = the 30 float64 grid points.  Outputs t[b] (snapped), norm[b] = peak[b]*normfac, idx[b] (optional). */
int snrse_v3_scalars(const float* ratio, const float* peak, double snr_scale, float nf_const, const double* t30,
                     float* t_out, float* nf_out, int* idx_out, int B, void* stream);
int snrse_snr_ratio(const float* g, float* ratio, int B, void* stream);  /* est_gt/(1-est_gt), model.py:721 */

/* ---------------------------------------------------------------- sampler updates --------------
 * out_mean = a[b]*x + b[b]*y + c[b]*s ; out_x = out_mean + d[b]*z on complex64 [B][n].  Any of x,y,s,z,
 * out_mean,out_x may be NULL.  Covers prior sampling (sdes.py:225-232,297-304), annealed Langevin
 * (sampling/correctors.py:69-81), reverse diffusion (sampling/predictors.py:75-80; sdes.py:73-91,132-140)
 * and X_T = Y + sigma*t*Z (model.py:822-823). */
int snrse_lincomb(const void* x, const void* y, const void* s, const void* z, const float* a, const float* b,
                  const float* c, const float* d, void* out_mean, void* out_x, int B, int64_t n, void* stream);
/* snrse_lincomb_keyed: snrse_lincomb with z drawn in the kernel from a per-item key instead of read from memory, so that
 *   an utterance's noise depends on its key and the seed only, never on its row, its batch or earlier draws.  Same
 *   arithmetic as snrse_lincomb: out_x is bit-identical to snrse_lincomb(..., z = the draw written to z_out, ...).
 *   keys: uint64 [B]; n must be 256 * tpad (item b is complex64 [256][tpad], row-major); z_out (optional): the draw,
 *   complex64 [B][n].  len (optional, int32 [B]): an item whose own padded width 64*ceil((1 + len[b]/128)/64) is not
 *   tpad is written as NaN in out_mean, out_x and z_out, since enhancing it at width tpad is not enhancing it alone.
 *
 *   Keyed noise (a stable format): complex element i (0 <= i < n) of item b with key k and seed s is
 *     (x0, x1, x2, x3) = Philox4x32-10(counter = (i >> 1, 0, lo32(k), hi32(k)), key = (lo32(s), hi32(s)))
 *   (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC'11; curand's Philox4_32_10), with
 *     (xa, xb) = (x0, x1) for even i, (x2, x3) for odd i,
 *     u1 = ((xa >> 8) + 1) * 2^-24 in (0, 1],  u2 = (xb >> 8) * 2^-24 in [0, 1)   (both exact in fp32),
 *     r = sqrtf(-logf(u1)),  z = r * cospi(2 u2) + i r * sinpi(2 u2)   (accurate logf / sqrtf / sincospif).
 *   re z and im z are independent N(0, 1/2), so E|z|^2 = 1 as torch.randn_like draws on complex64; |z|^2 ~ Exp(1)
 *   truncated at 24 ln 2 (probability 6e-8 per draw).  The counter's second word is 0 here and reserved.
 *   Known answers: counter (0,0,0,0), key (0,0) -> 6627e8d5 e169c58d bc57ac4c 9b00dbd8; all ones ->
 *   408f276d 41c83b0e a20bc7c6 6d5451fd; counter (243f6a88, 85a308d3, 13198a2e, 03707344), key (a4093822, 299f31d0)
 *   -> d16cfe09 94fdcceb 5001e420 24126ea1. */
int snrse_lincomb_keyed(const void* x, const void* y, const void* s, const float* a, const float* b, const float* c,
                        const float* d, const uint64_t* keys, uint64_t seed, const int* len, int tpad, void* z_out,
                        void* out_mean, void* out_x, int B, int64_t n, void* stream);

/* Embedded Runge-Kutta helpers for the probability-flow ODE sampler kept on the device (replaces the numpy round trip
 * per RHS evaluation of `ode_sampler`, sampling/__init__.py:149-161; step control follows scipy.integrate RK45, the
 * third-party solver the reference calls at :156).  K: nk (<= 8) stage derivatives of n complex64 values each, back
 * to back; coef: nk HOST floats.
 *   snrse_rk_combine       : out = y + h * sum_j coef[j] K[j]                       (y may be NULL)
 *   snrse_rk_scaled_sqnorm : partial[i] (i < snrse_rk_partials(n), device doubles) = block sums of
 *                            |h * sum_j coef[j] K[j]|^2 / (atol + rtol * max(|y|, |y2|))^2   (y2 may be NULL) */
int snrse_rk_combine(const void* y, const void* K, int nk, int64_t n, float h, const float* coef, void* out, void* stream);
int snrse_rk_partials(int64_t n);
int snrse_rk_scaled_sqnorm(const void* K, int nk, int64_t n, float h, const float* coef, const void* y, const void* y2,
                           float atol, float rtol, double* partial, void* stream);

/* ---------------------------------------------------------------- NCSN++ score network ---------
 * Replaces NCSNpp.forward (backbones/ncsnpp.py:247-404) and the head of ScoreModel.forward
 * (model.py:481-543).  Weights: the host packs the reference state dict into one device blob
 * following the table returned by snrse_ncsnpp_param_info (kinds: 0 raw f32; 1 conv3x3 -> bf16
 * K-major [cout][k_offset + (r*3+s)*Cin + cin] with row pitch row_stride; 2 conv1x1 -> bf16
 * [cout][k_offset + cin]; 3 NIN W[in,out] -> bf16 [out][k_offset + in]; 4 conv3x3 -> f32
 * [cout][r][s][cin]; accumulate=1: add into the destination). */
int snrse_ncsnpp_create(void** handle, int nf, const int* ch_mult, int n_levels, int num_res_blocks,
                        const int* attn_resolutions, int n_attn, int image_size);
void snrse_ncsnpp_destroy(void* handle);
int snrse_ncsnpp_num_modules(void* handle);
int snrse_ncsnpp_num_params(void* handle);
int64_t snrse_ncsnpp_weight_bytes(void* handle);
int snrse_ncsnpp_param_info(void* handle, int i, char* name, int name_cap, int* kind, int64_t* offset,
                            int64_t* row_stride, int64_t* k_offset, int* accumulate);
int snrse_ncsnpp_param_shape(void* handle, int i, int64_t* dims, int* ndim); /* shape of the state-dict tensor */
int snrse_ncsnpp_set_weights(void* handle, const void* device_blob);
/* Plan for inputs [B][F][T]: returns the workspace size (or -1).  flags bit0: keep all activations
 * (debug taps, snrse_ncsnpp_read_tap); bit1: fp32 CUDA-core cross-check path (convolutions, attention and input packing
 * instead of tcgen05 / bf16 operands).  Any other bit is rejected (-1). */
int64_t snrse_ncsnpp_plan_bytes(void* handle, int B, int F, int T, int flags);
int snrse_ncsnpp_plan_bind(void* handle, int B, int F, int T, void* workspace, int64_t bytes);
/* x (state), y (noisy), out: complex64 [B][F][T]; t [B] f32.  mode 0: dnn(cat[x,y], t);
 * 1: c_skip*x + c_out*dnn (sebridge / sebridge_v3, model.py:537-541); 2: -dnn (bbed, model.py:488-489). */
int snrse_ncsnpp_forward(void* handle, int B, int F, int T, const void* x, const void* y, const float* t, void* out,
                         int mode, void* stream);

/* ---------------------------------------------------------------- single operators (NHWC bf16) --
 * conv: ddpm_conv3x3 / ddpm_conv1x1 / NIN (ncsnpp_utils/layers.py:100-124,537-555) as implicit GEMM:
 *   out[b,h,w,n] = scale*( sum_{tap,c} x0[b,h+dh,w+dw,c]*wt[n][tap*c0+c] + sum_c x1[b,h,w,c]*wt[n][taps0*c0+c]
 *                          + bias[n] + tbias[b*tb_stride+n] + res[b,h,w,n] );
 *   impl 0: tcgen05 (2-CTA halo-reuse persistent kernel when eligible), 1: CUDA cores (cross-check), 2: the
 *   single-CTA tcgen05 GEMM kernel that also serves 1x1 / NIN / attention. */
int snrse_conv_nhwc(const void* x0, int c0, int taps0, const void* x1, int c1, const void* wt, int n, const float* bias,
                    const float* tbias, int tb_stride, const void* res, float scale, void* out, int B, int H, int W,
                    int impl, void* stream);
/* GroupNorm(32, eps) (+SiLU) (ncsnpp_utils/layerspp.py:221,233,245,266) */
/* GroupNorm(32 groups, eps) + SiLU + conv3x3 (+ optional 1x1 shortcut on x1, bias, per-sample tbias, residual,
 * scale) as ONE pass: statistics kernel + convolution that normalises its operand in shared memory.  Replaces the
 * nn.GroupNorm -> SiLU -> ddpm_conv3x3 chain of ResnetBlockBigGANpp (ncsnpp_utils/layerspp.py:245-271).
 * workspace: snrse_groupnorm_workspace_bytes(B).  Needs W >= 8, H >= 8, n in {128, 256}, c0 % 128 == 0. */
int snrse_gn_silu_conv3x3_nhwc(const void* x0, int c0, const float* gamma, const float* beta, float eps, const void* x1,
                               int c1, const void* wt, int n, const float* bias, const float* tbias, int tb_stride,
                               const void* res, float scale, void* out, int B, int H, int W, void* workspace,
                               void* stream);
/* conv3x3 (as snrse_conv_nhwc, taps0 = 9) whose epilogue also accumulates the GroupNorm sums of the result:
 * ustats [B][n/4][2] int64 fixed point = (sum * 2^30, sum of squares * 2^24) per 4-channel unit (zeroed by the
 * call).  Integer accumulation: bit-identical from run to run and independent of the batch.
 * Needs W >= 8, H >= 8, n in {128, 256}. */
int snrse_conv3x3_nhwc_stats(const void* x0, int c0, const void* x1, int c1, const void* wt, int n, const float* bias,
                             const float* tbias, int tb_stride, const void* res, float scale, void* out, int B, int H,
                             int W, void* ustats, void* stream);
int64_t snrse_groupnorm_workspace_bytes(int B);
int snrse_groupnorm_nhwc(const void* x, const float* gamma, const float* beta, void* out, int B, int H, int W, int C,
                         int silu, float eps, void* workspace, void* stream);
/* upsample_2d / downsample_2d with the [1,3,3,1] FIR (ncsnpp_utils/up_or_down_sampling.py:195-257;
 * op/upfirdn2d.cpp:12-23, op/upfirdn2d_kernel.cu modes 3 and 5) */
int snrse_fir_nhwc(const void* x, void* out, int B, int H, int W, int C, int up, void* stream);
int snrse_fir_f4(const float* x, float* out, int B, int H, int W, int up, void* stream);
/* snrse_upfirdn2d: the reference's one native operator, general form -- replaces
 *   `upfirdn2d_op.upfirdn2d(input[N,H,W,1], kernel[kh,kw], up_x, up_y, down_x, down_y, pad_x0, pad_x1, pad_y0, pad_y1)`
 *   (ncsnpp_utils/op/upfirdn2d.cpp:12-23, op/upfirdn2d_kernel.cu:213-311; pure-torch statement op/upfirdn2d.py:159-200).
 *   input fp32 [major][in_h][in_w] (minor = 1 as every reference call site passes), kernel fp32 [kh][kw] (device),
 *   out fp32 [major][out_h][out_w] with out_h = (in_h*up_y + pad_y0 + pad_y1 - kh)/down_y + 1 (same for w); negative
 *   pads crop.  The caller allocates `out`; launches on `stream`; no synchronisation. */
int snrse_upfirdn2d(const float* input, const float* kernel, float* out, int64_t major, int in_h, int in_w, int kernel_h,
                    int kernel_w, int up_x, int up_y, int down_x, int down_y, int pad_x0, int pad_x1, int pad_y0, int pad_y1,
                    void* stream);
/* softmax(q k^T / sqrt(C)) v over n positions (ncsnpp_utils/layerspp.py:84-88); workspace:
 * snrse_attention_workspace_bytes(B, n, C) (fp32 scores, bf16 probabilities, V^T).  Tensor cores when n % 64 == 0. */
int64_t snrse_attention_workspace_bytes(int B, int n, int C);
int snrse_attention_nhwc(const void* q, const void* k, const void* v, void* workspace, void* out, int B, int n, int C,
                         void* stream);

/* ---------------------------------------------------------------- SNR estimator ----------------
 * SNRNet.forward (backbones/snrnet.py:47-97).  feat: f32 [B][2][256][T16] (T16 % 16 == 0);
 * out: f32 [B] = noise/(speech+noise).  weights: packed blob, see snrse_snrnet_param_info (transform 0: flat copy of
 * the state-dict tensor; 1: the (64 x k) convolution weights [co][ci][f][dt] stored as [ci*64+f][dt][co]; 2: the 3x3
 * convolution [co][ci][3][3] stored as [ci][tap][co]). */
int snrse_snrnet_num_params(void);
int snrse_snrnet_param_info(int i, char* name, int name_cap, int64_t* offset, int64_t* numel, int* transform);
int snrse_snrnet_param_shape(int i, int64_t* dims, int* ndim);
int64_t snrse_snrnet_weight_bytes(void);
int64_t snrse_snrnet_workspace_bytes(int B, int T16);
int snrse_snrnet_forward(const void* weights, const float* feat, float* out, int B, int T16, void* workspace,
                         void* stream);
/* snrse_snrnet_forward on a ragged batch: the estimate of item b is SNRNet.forward of that utterance alone, i.e. over its
 *   first clusters[b] 16-frame clusters (model.py:715-721 pads each file to its own multiple of 16 frames).
 *   clusters: int32 [B] (device), read clamped to [1, T16/16]; NULL = every item has T16/16 clusters, which is
 *   snrse_snrnet_forward.  Frames >= 16*clusters[b] of feat and the workspace rows of those clusters are never read.
 *   Item b gives the same bits as a call with that utterance alone at T16 = 16*clusters[b]; one cluster gives NaN, as
 *   the reference's unbiased std over one element.  Same feat layout and workspace size as snrse_snrnet_forward. */
int snrse_snrnet_forward_varlen(const void* weights, const float* feat, const int* clusters, float* out, int B, int T16,
                                void* workspace, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SNRSE_B200_H */
