/* snrse_b200_plans.h -- the convolution plans of the NCSN++ executor, as debug entry points of libsnrse_b200.so.
 *
 * NOT part of the drop-in ABI (snrse_b200.h), the measurement hooks (snrse_b200_debug.h) or the launcher entry points
 * (snrse_b200_layers.h): nothing in the product path calls these, and nothing here launches a kernel.  They list which
 * convolution plans the executor chooses (tests/test_conv_plans_cpu.py groups them into classes without a device) and
 * which plan a launcher makes for given views (tests/test_gpu_conv_plans.py checks the two agree).  Same conventions as
 * snrse_b200.h.
 */
#ifndef SNRSE_B200_PLANS_H
#define SNRSE_B200_PLANS_H

#include <stdint.h>

#include "snrse_b200_layers.h"

#ifdef __cplusplus
extern "C" {
#endif

/* integer fields of a convolution plan; those of the other kernel are 0 */
typedef struct {
    int sub, nsplit, n_loc, acc_bufs, na, nb, stg_bufs, nsc; /* 2-CTA kernel: sub-tiles, N split, output channels per
                                                              * cluster, TMEM accumulators, halo / weight ring depths,
                                                              * epilogue staging tiles, shortcut ring slots */
    int th, tw, n_tile, small, stages;                       /* single-CTA GEMM: tile, N tile, small-map mode, ring depth */
    int tiles_h, tiles_w, n_tiles, grid, smem_bytes;         /* both: tiles, CTAs launched, dynamic shared memory */
} snrse_conv_plan;
/* one convolution of the executor: the operand views (channel count, pitch ld and first channel off inside the
 * buffer), the operand combination and the plan */
typedef struct {
    int path;                       /* 0 2-CTA kernel, 1 CUDA cores, 2 single-CTA implicit GEMM (snrse_dbg_conv paths) */
    int out4;                       /* the C -> 4 output head (snrse_dbg_conv_out4); its result is fp32, ld 4 */
    int B, H, W;
    int c0, ld0, off0;              /* operand */
    int c1, ld1, off1;              /* 1x1 shortcut operand, c1 = 0: none */
    int res, ld_res, off_res;       /* identity residual (n channels) */
    int ld_out, off_out;
    int taps, n;                    /* taps of the operand (9 or 1), output channels */
    int norm, bias, tbias, tb_stride, stats, addend;   /* GroupNorm+SiLU in flight, bias, time-embedding bias with
                                                        * its row stride, epilogue GroupNorm sums, out4 pyramid addend */
    float scale;
    snrse_conv_plan plan;
} snrse_conv_row;
/* the convolutions the (B,F,T) plan with `flags` records, in order, with their plans for num_sms SMs: recorded like
 * snrse_ncsnpp_plan_bytes but not cached, no weights, no device.  *n receives the count; rows may be NULL (count only),
 * otherwise cap must hold them */
int snrse_ncsnpp_dbg_convs(void* handle, int B, int F, int T, int flags, int num_sms, snrse_conv_row* rows, int cap, int* n);
/* the plan that snrse_dbg_conv's path 0 / 2 launcher makes for these views, or, for path 0 with n = 4,
 * snrse_dbg_conv_out4's (out: the fp32 [B][H][W][4] result as a view with C = ld = 4): the launcher's own make_plan with
 * the device's SM count; nothing is launched */
int snrse_dbg_conv_plan(const snrse_view* x0, int taps0, const snrse_view* x1, const void* wt, int n, const snrse_view* res,
                        const snrse_view* out, const float* scsh, int path, snrse_conv_plan* plan);

#ifdef __cplusplus
}
#endif
#endif /* SNRSE_B200_PLANS_H */
