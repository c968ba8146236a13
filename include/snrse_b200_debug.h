/* snrse_b200_debug.h -- measurement and debugging entry points of libsnrse_b200.so.
 *
 * NOT part of the drop-in ABI (snrse_b200.h): nothing in the product path calls these.  They exist for bench.py's
 * roofline record (per-launch-group CUDA-event timing), the parity tests (per-module activation taps) and the
 * kernel-tuning tools under tools/ (cycle counters of the convolution kernels).  Same conventions as snrse_b200.h.
 */
#ifndef SNRSE_B200_DEBUG_H
#define SNRSE_B200_DEBUG_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* number of launch groups of the (B,F,T) plan == capacity needed by snrse_ncsnpp_profile_forward */
int snrse_ncsnpp_num_launch_groups(void* handle, int B, int F, int T);
/* eager forward with a CUDA event between launch groups on `stream`; SYNCHRONISES the stream and fills
 * kinds / algorithmic flops / algorithmic bytes / milliseconds per group (kind 1 = implicit-GEMM convolution) */
int snrse_ncsnpp_profile_forward(void* handle, int B, int F, int T, const void* x, const void* y, const float* t,
                                 void* out, int mode, void* stream, int cap, int* kinds, double* flops, double* bytes,
                                 float* ms, int* n_groups);
/* output of module `module_idx` (SURVEY Appendix A numbering) of the last forward of a plan bound with flag bit0
 * (keep every activation), converted to fp32 NCHW; dims receives (B, C, H, W) */
int snrse_ncsnpp_read_tap(void* handle, int B, int F, int T, int module_idx, float* out, int64_t cap_elems,
                          int64_t* dims, void* stream);
/* cycle counters of the convolution kernels: [grid][8] int64 (a / b / accumulator waits of the MMA warp, total,
 * epilogue wait / body, producer waits), filled by every later launch; NULL switches them off */
void snrse_conv_halo_set_debug(long long* dev_counters);

#ifdef __cplusplus
}
#endif
#endif /* SNRSE_B200_DEBUG_H */
