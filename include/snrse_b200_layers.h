/* snrse_b200_layers.h -- the NCSN++ executor's launchers as entry points of libsnrse_b200.so, one per launcher.
 *
 * NOT part of the drop-in ABI (snrse_b200.h) nor of the measurement hooks (snrse_b200_debug.h): nothing in the product
 * path calls these.  Each converts its arguments and calls the internal launcher of the same name with no logic of its
 * own, so a caller runs exactly the code the executor runs, on the views the executor passes (channel slices of the
 * decoder's concatenation buffers, views into the fused qkv buffer).  tests/test_gpu_network_layers.py checks every
 * launcher through them.  Same conventions as snrse_b200.h.
 */
#ifndef SNRSE_B200_LAYERS_H
#define SNRSE_B200_LAYERS_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* snrse_view: a bf16 NHWC activation, element (b,h,w,c) at ((bf16*)ptr)[((b*H + h)*W + w)*ld + c]; ld > C and ptr
 * offset by a channel count make it a channel slice of a concatenation buffer, as the executor's views are. */
typedef struct {
    void* ptr;
    int B, H, W, C, ld;
} snrse_view;
/* out = (conv(x0) [+ 1x1 conv(x1)] + bias + tbias[b*tb_stride + n] [+ res]) * scale, wt [n][taps0*C0 + C1] bf16;
 * path 0: 2-CTA kernel (scsh: GroupNorm+SiLU of x0 in flight; ustats: GroupNorm sums of out accumulated into
 * [B][n/4][2], zeroed by the caller), 1: CUDA cores, 2: single-CTA implicit GEMM.  A shape the path does not take
 * returns SNRSE_ERR_ARG. */
int snrse_dbg_conv(const snrse_view* x0, int taps0, const snrse_view* x1, const void* wt, int n, const float* bias,
                   const float* tbias, int tb_stride, const snrse_view* res, float scale, const snrse_view* out,
                   const float* scsh, void* ustats, int path, void* stream);
/* GroupNorm in three steps: unit sums (accumulated into zeroed [B][C/4][2]), scale/shift [B][2][C] over the channel
 * concatenation of one or two sources (U1 = 0: one), count = H*W*C/32 elements per group, and y = x*scale + shift
 * (+SiLU) */
int snrse_dbg_gn_stats(const snrse_view* x, void* ustats, void* stream);
int snrse_dbg_gn_finalize(const void* src0, int U0, const void* src1, int U1, int B, int64_t count, const float* gamma,
                          const float* beta, float eps, float* scsh, void* stream);
int snrse_dbg_gn_apply(const snrse_view* x, const float* scsh, int silu, const snrse_view* out, void* stream);
/* the stand-alone single-output FIR x2 resampling (snrse_fir_nhwc's launcher; the executor does not launch it), kept as
 * the reference the dual pass is compared with, and the dual-output pass of the up / down blocks:
 * out_n = FIR(silu(x*scale + shift)), out_r = FIR(x) */
int snrse_dbg_fir(const snrse_view* x, const snrse_view* out, int up, void* stream);
int snrse_dbg_fir_dual(const snrse_view* x, const snrse_view* out_n, const snrse_view* out_r, int up, const float* scsh,
                       void* stream);
/* C -> 4 output head, out4 [B][H][W][4] f32 = conv3x3(a) + bias (+ addend4): path 0 2-CTA kernel, w bf16 [16][9C]
 * (rows 4..15 unused), scsh optional; path 1 CUDA cores, w f32 [4][3][3][C], scsh must be null */
int snrse_dbg_conv_out4(const snrse_view* a, const void* w, const float* bias, const float* addend4, float* out4,
                        const float* scsh, int path, void* stream);
/* x, y complex64 [B][n] -> x4 [B][n][4] f32 and, when x64 is non-null, the bf16 hi/lo operand [B][n][64] */
int snrse_dbg_pack_input(const void* x, const void* y, float* x4, void* x64, int B, int64_t n, void* stream);
/* input convolution on CUDA cores (x4 f32, w f32 [C][3][3][4]) and the input-pyramid combine out = h + w p4 + bias */
int snrse_dbg_conv_in4(const float* x4, const float* w, const float* bias, const snrse_view* out, void* stream);
int snrse_dbg_combine4(const float* p4, const snrse_view* h, const float* w, const float* bias, const snrse_view* out,
                       void* stream);
/* time embedding + every block's Dense_0 row, and the final head (modes as in snrse_ncsnpp_forward) */
int snrse_dbg_temb(const float* t, int B, int nf, const float* fourier_w, const float* w1, const float* b1, const float* w2,
                   const float* b2, const float* dense_w, const float* dense_b, int rows, float* scratch, float* tb_out,
                   void* stream);
int snrse_dbg_final(const float* p4, const float* t, const float* w, const float* bias, const void* xres, void* out, int B,
                    int64_t n, int mode, void* stream);
/* single-head attention over H*W tokens; workspace: snrse_attention_workspace_bytes; allow_tensor_cores 0 keeps the fp32
 * CUDA-core kernels */
int snrse_dbg_attention(const snrse_view* q, const snrse_view* k, const snrse_view* v, void* workspace, const snrse_view* o,
                        int allow_tensor_cores, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SNRSE_B200_LAYERS_H */
