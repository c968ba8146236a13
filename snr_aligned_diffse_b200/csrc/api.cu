// C-ABI entry points for the stand-alone operators (declared in include/snrse_b200.h).
// The NCSN++ executor entry points live in engine.cu, the SNR estimator's in snrnet.cu.
#include <stdarg.h>
#include <stdlib.h>

#include <vector>

#include "kernels.h"

static thread_local char g_err[512] = "";
long long g_snrse_launches = 0;
static int pdl_default() {
    const char* e = getenv("SNRSE_PDL");
    return e ? (atoi(e) & 7) : 2;
}
int g_snrse_pdl = pdl_default();

void snrse_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static cudaStream_t S(void* s) { return static_cast<cudaStream_t>(s); }

static ActView mk_view(const void* p, int B, int H, int W, int C, int ld) {
    ActView v;
    v.ptr = const_cast<bf16*>(static_cast<const bf16*>(p));
    v.B = B; v.H = H; v.W = W; v.C = C; v.ld = ld;
    return v;
}

// GroupNorm(32, eps) statistics and scale/shift of x in a workspace of snrse_groupnorm_workspace_bytes(B): the unit sums
// [B][128][2] (zeroed here) first, then the scale/shift [B][2][C] that *scsh points to.
static int gn_scale_shift(const ActView* x, const float* gamma, const float* beta, float eps, void* workspace,
                          cudaStream_t s, float** scsh) {
    unsigned long long* ust = static_cast<unsigned long long*>(workspace);
    *scsh = reinterpret_cast<float*>(ust + (int64_t)x->B * 128 * 2);
    SNRSE_CUDA(cudaMemsetAsync(ust, 0, (size_t)x->B * (x->C / 4) * 16, s));
    SNRSE_TRY(gn_stats_launch(x, ust, s));
    return gn_finalize_launch(ust, x->C / 4, nullptr, 0, x->B, (int64_t)x->H * x->W * (x->C / 32), gamma, beta, eps,
                              *scsh, s);
}

extern "C" {

int snrse_version(void) { return 100; }
long long snrse_launch_count(void) { return g_snrse_launches; }
int snrse_set_pdl(int on) {
    const int prev = g_snrse_pdl;
    if (on >= 0) g_snrse_pdl = on & 7;
    return prev;
}
const char* snrse_last_error(void) { return g_err; }

// 0 when the current device is a Blackwell B200-class GPU (compute capability 10.x); the kernels are sm_100a-only.
int snrse_device_check(void) {
    int dev = 0;
    cudaDeviceProp prop;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess) {
        snrse_set_error("no CUDA device available: the B200 library has no CPU fallback");
        return SNRSE_ERR_CUDA;
    }
    if (prop.major != 10) {
        snrse_set_error("device %s is sm_%d%d; this library is built for sm_100a only", prop.name, prop.major, prop.minor);
        return SNRSE_ERR_UNSUPPORTED;
    }
    return SNRSE_OK;
}

int snrse_stft(const float* wave, const int* len, const float* scale, int scale_is_divisor, void* out, int B,
               int lstride, int tpad, int transform, float alpha, float beta, int planar, void* stream) {
    SNRSE_CHECK_ARG(wave && out, "stft: null pointer");
    return stft_launch(wave, len, scale, scale_is_divisor, static_cast<float*>(out), B, lstride, tpad, transform, alpha,
                       beta, planar, S(stream));
}

// the overlap-add runs in shared memory since the FFT kernels; a token workspace keeps the ABI and its callers unchanged
int64_t snrse_istft_workspace_bytes(int B, int tpad) { (void)B; (void)tpad; return 256; }

int snrse_istft(const void* spec, const int* len, const float* scale, float* wave, void* workspace, int B, int lstride,
                int tpad, int transform, float alpha, float beta, void* stream) {
    SNRSE_CHECK_ARG(spec && wave && workspace, "istft: null pointer");
    return istft_launch(static_cast<const float2*>(spec), len, scale, wave, static_cast<float*>(workspace), B, lstride,
                        tpad, transform, alpha, beta, S(stream));
}

int snrse_spec_transform(const void* in, void* out, int64_t n, int inverse, int transform, float alpha, float beta,
                         void* stream) {
    SNRSE_CHECK_ARG(in && out, "spec_transform: null pointer");
    return spec_transform_launch(static_cast<const float2*>(in), static_cast<float2*>(out), n, inverse, transform, alpha,
                                 beta, S(stream));
}

int snrse_si_sdr(const float* ref, const float* est, const int* len, int B, int lstride, double* out, void* stream) {
    return si_sdr_launch(ref, est, len, B, lstride, out, S(stream));
}

int snrse_absmax(const float* wave, const int* len, int B, int lstride, float* out, void* stream) {
    SNRSE_CHECK_ARG(wave && out, "absmax: null pointer");
    return absmax_launch(wave, len, B, lstride, out, S(stream));
}

int snrse_v3_scalars(const float* ratio, const float* peak, double snr_scale, float nf_const, const double* t30,
                     float* t_out, float* nf_out, int* idx_out, int B, void* stream) {
    SNRSE_CHECK_ARG(ratio && peak && t30 && t_out && nf_out, "v3_scalars: null pointer");
    return v3_scalars_launch(ratio, peak, snr_scale, nf_const, t30, t_out, nf_out, idx_out, B, S(stream));
}

int snrse_snr_ratio(const float* g, float* ratio, int B, void* stream) { return snr_ratio_launch(g, ratio, B, S(stream)); }

int snrse_lincomb(const void* x, const void* y, const void* sc, const void* z, const float* a, const float* b,
                  const float* c, const float* d, void* out_mean, void* out_x, int B, int64_t n, void* stream) {
    return lincomb_launch(static_cast<const float2*>(x), static_cast<const float2*>(y), static_cast<const float2*>(sc),
                          static_cast<const float2*>(z), a, b, c, d, static_cast<float2*>(out_mean),
                          static_cast<float2*>(out_x), B, n, S(stream));
}

int snrse_lincomb_keyed(const void* x, const void* y, const void* sc, const float* a, const float* b, const float* c,
                        const float* d, const uint64_t* keys, uint64_t seed, const int* len, int tpad, void* z_out,
                        void* out_mean, void* out_x, int B, int64_t n, void* stream) {
    return lincomb_keyed_launch(static_cast<const float2*>(x), static_cast<const float2*>(y),
                                static_cast<const float2*>(sc), a, b, c, d, reinterpret_cast<const unsigned long long*>(keys),
                                (unsigned long long)seed, len, tpad, static_cast<float2*>(z_out),
                                static_cast<float2*>(out_mean), static_cast<float2*>(out_x), B, n, S(stream));
}

int snrse_rk_combine(const void* y, const void* K, int nk, int64_t n, float h, const float* coef, void* out, void* stream) {
    return rk_combine_launch(static_cast<const float2*>(y), static_cast<const float2*>(K), nk, n, h, coef,
                             static_cast<float2*>(out), S(stream));
}

int snrse_rk_partials(int64_t n) { return rk_partials(n); }

int snrse_rk_scaled_sqnorm(const void* K, int nk, int64_t n, float h, const float* coef, const void* y, const void* y2,
                           float atol, float rtol, double* partial, void* stream) {
    return rk_scaled_sqnorm_launch(static_cast<const float2*>(K), nk, n, h, coef, static_cast<const float2*>(y),
                                   static_cast<const float2*>(y2), atol, rtol, partial, S(stream));
}

// ---- single-operator entry points (NHWC bf16), used by the parity tests and usable as drop-in ops
int snrse_conv_nhwc(const void* x0, int c0, int taps0, const void* x1, int c1, const void* wt, int n, const float* bias,
                    const float* tbias, int tb_stride, const void* res, float scale, void* out, int B, int H, int W,
                    int impl, void* stream) {
    SNRSE_CHECK_ARG(x0 && wt && out, "conv_nhwc: null pointer");
    ActView a0 = mk_view(x0, B, H, W, c0, c0), a1, r;
    if (x1) a1 = mk_view(x1, B, H, W, c1, c1);
    if (res) r = mk_view(res, B, H, W, n, n);
    if (impl == 1) {
        SNRSE_CHECK_ARG(n <= 256, "conv_nhwc: CUDA-core cross-check path handles N <= 256");
        return conv_simt_launch(&a0, taps0, x1 ? &a1 : nullptr, static_cast<const bf16*>(wt), n, bias, tbias, tb_stride,
                                res ? &r : nullptr, scale, static_cast<bf16*>(out), n, S(stream));
    }
    if (impl == 0 && conv_halo2_eligible(a0.H, a0.W, taps0, n)) {
        ConvHaloPlan hp;
        SNRSE_TRY(conv_halo2_make_plan(&hp, &a0, x1 ? &a1 : nullptr, static_cast<const bf16*>(wt), n, bias, tbias, tb_stride,
                                       res ? &r : nullptr, scale, static_cast<bf16*>(out), n, nullptr, nullptr));
        return conv_halo2_launch(&hp, S(stream));
    }
    ConvGemmPlan p;
    SNRSE_TRY(conv_gemm_make_plan(&p, &a0, taps0, x1 ? &a1 : nullptr, static_cast<const bf16*>(wt), n, 0, 0, bias, tbias,
                                  tb_stride, res ? &r : nullptr, scale, out, n, 0));
    return conv_gemm_launch(&p, S(stream));
}

// conv3x3 on the 2-CTA kernel that also accumulates the GroupNorm sums of its result (what the NCSN++ executor uses so
// that GroupNorm needs no pass of its own): ustats [B][n/4][2] 64-bit fixed point (sum * 2^30, sum of squares * 2^24
// per 4-channel unit), zeroed here first.
int snrse_conv3x3_nhwc_stats(const void* x0, int c0, const void* x1, int c1, const void* wt, int n, const float* bias,
                             const float* tbias, int tb_stride, const void* res, float scale, void* out, int B, int H,
                             int W, void* ustats, void* stream) {
    SNRSE_CHECK_ARG(x0 && wt && out && ustats, "conv3x3_stats: null pointer");
    ActView a0 = mk_view(x0, B, H, W, c0, c0), a1, r;
    if (x1) a1 = mk_view(x1, B, H, W, c1, c1);
    if (res) r = mk_view(res, B, H, W, n, n);
    SNRSE_CHECK_ARG(conv_halo2_eligible(a0.H, a0.W, 9, n), "conv3x3_stats: needs W >= 8, H >= 8, N in {128, 256}");
    SNRSE_CUDA(cudaMemsetAsync(ustats, 0, (size_t)B * (n / 4) * 16, S(stream)));
    ConvHaloPlan hp;
    SNRSE_TRY(conv_halo2_make_plan(&hp, &a0, x1 ? &a1 : nullptr, static_cast<const bf16*>(wt), n, bias, tbias, tb_stride,
                                   res ? &r : nullptr, scale, static_cast<bf16*>(out), n, nullptr,
                                   static_cast<unsigned long long*>(ustats)));
    return conv_halo2_launch(&hp, S(stream));
}

int64_t snrse_groupnorm_workspace_bytes(int B) { return (int64_t)B * (128 * 16 + 1024 * 4); }

int snrse_groupnorm_nhwc(const void* x, const float* gamma, const float* beta, void* out, int B, int H, int W, int C,
                         int silu, float eps, void* workspace, void* stream) {
    SNRSE_CHECK_ARG(x && gamma && beta && out && workspace, "groupnorm: null pointer");
    const ActView vx = mk_view(x, B, H, W, C, C), vo = mk_view(out, B, H, W, C, C);
    float* scsh;
    SNRSE_TRY(gn_scale_shift(&vx, gamma, beta, eps, workspace, S(stream), &scsh));
    return gn_apply_launch(&vx, scsh, silu, &vo, S(stream));
}

// GroupNorm(32, eps) + SiLU + conv3x3 (+1x1 shortcut / bias / time-embedding bias / residual, * scale) with the
// normalisation applied to the operand inside the convolution kernel: the body of ResnetBlockBigGANpp
// (ncsnpp_utils/layerspp.py:245-271) without materialising the normalised activation.
int snrse_gn_silu_conv3x3_nhwc(const void* x0, int c0, const float* gamma, const float* beta, float eps, const void* x1,
                               int c1, const void* wt, int n, const float* bias, const float* tbias, int tb_stride,
                               const void* res, float scale, void* out, int B, int H, int W, void* workspace,
                               void* stream) {
    SNRSE_CHECK_ARG(x0 && gamma && beta && wt && out && workspace, "gn_silu_conv3x3: null pointer");
    ActView a0 = mk_view(x0, B, H, W, c0, c0), a1, r;
    if (x1) a1 = mk_view(x1, B, H, W, c1, c1);
    if (res) r = mk_view(res, B, H, W, n, n);
    SNRSE_CHECK_ARG(conv_halo2_eligible(a0.H, a0.W, 9, n), "gn_silu_conv3x3: needs W >= 8, H >= 8, N in {128, 256}");
    float* scsh;
    SNRSE_TRY(gn_scale_shift(&a0, gamma, beta, eps, workspace, S(stream), &scsh));
    ConvHaloPlan hp;
    SNRSE_TRY(conv_halo2_make_plan(&hp, &a0, x1 ? &a1 : nullptr, static_cast<const bf16*>(wt), n, bias, tbias, tb_stride,
                                   res ? &r : nullptr, scale, static_cast<bf16*>(out), n, scsh, nullptr));
    return conv_halo2_launch(&hp, S(stream));
}

int snrse_fir_nhwc(const void* x, void* out, int B, int H, int W, int C, int up, void* stream) {
    SNRSE_CHECK_ARG(x && out, "fir: null pointer");
    const ActView vx = mk_view(x, B, H, W, C, C);
    const ActView vo = up ? mk_view(out, B, 2 * H, 2 * W, C, C) : mk_view(out, B, H / 2, W / 2, C, C);
    return up ? fir_up2_launch(&vx, &vo, S(stream)) : fir_down2_launch(&vx, &vo, S(stream));
}

int snrse_upfirdn2d(const float* input, const float* kernel, float* out, int64_t major, int in_h, int in_w, int kernel_h,
                    int kernel_w, int up_x, int up_y, int down_x, int down_y, int pad_x0, int pad_x1, int pad_y0, int pad_y1,
                    void* stream) {
    SNRSE_CHECK_ARG(input && kernel && out, "upfirdn2d: null pointer");
    return upfirdn2d_launch(input, kernel, out, major, in_h, in_w, kernel_h, kernel_w, up_x, up_y, down_x, down_y, pad_x0,
                            pad_x1, pad_y0, pad_y1, S(stream));
}

int snrse_fir_f4(const float* x, float* out, int B, int H, int W, int up, void* stream) {
    SNRSE_CHECK_ARG(x && out, "fir_f4: null pointer");
    return up ? fir_up2_f4_launch(x, out, B, H, W, S(stream)) : fir_down2_f4_launch(x, out, B, H, W, S(stream));
}

int64_t snrse_attention_workspace_bytes(int B, int n, int C) { return attention_workspace_bytes(B, n, C); }

int snrse_attention_nhwc(const void* q, const void* k, const void* v, void* scores, void* out, int B, int n, int C,
                         void* stream) {
    SNRSE_CHECK_ARG(q && k && v && scores && out, "attention: null pointer");
    const ActView vq = mk_view(q, B, 1, n, C, C), vk = mk_view(k, B, 1, n, C, C), vv = mk_view(v, B, 1, n, C, C),
                  vo = mk_view(out, B, 1, n, C, C);
    return attention_launch(&vq, &vk, &vv, scores, &vo, S(stream));
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// measurement hooks (include/snrse_b200_debug.h): not part of the product ABI
long long* g_halo_dbg_shared = nullptr;
// device buffer of [grid][8] cycle counters filled by subsequent conv_halo2 / conv_gemm launches (null: off)
extern "C" void snrse_conv_halo_set_debug(long long* dev_counters) { g_halo_dbg_shared = dev_counters; }

// ---- the NCSN++ executor's launchers (include/snrse_b200_layers.h), one entry point each, on caller-made views
// (channel slices of concatenation buffers, views into the fused qkv buffer).  Each converts its arguments and calls the
// kernels.h launcher of the same name, so a test runs exactly the code the executor runs.
struct snrse_view {
    void* ptr;
    int B, H, W, C, ld;
};
static_assert(sizeof(snrse_view) == sizeof(ActView), "snrse_view must mirror ActView");

static ActView AV(const snrse_view* v) { return mk_view(v->ptr, v->B, v->H, v->W, v->C, v->ld); }

extern "C" {

// path 0: 2-CTA kernel, 1: CUDA cores, 2: single-CTA implicit GEMM.  scsh / ustats: 2-CTA kernel only.
int snrse_dbg_conv(const snrse_view* x0, int taps0, const snrse_view* x1, const void* wt, int n, const float* bias,
                   const float* tbias, int tb_stride, const snrse_view* res, float scale, const snrse_view* out,
                   const float* scsh, void* ustats, int path, void* stream) {
    SNRSE_CHECK_ARG(x0 && wt && out, "dbg_conv: null pointer");
    SNRSE_CHECK_ARG(path == 0 || !(scsh || ustats), "dbg_conv: scsh / ustats need path 0");
    const ActView a0 = AV(x0), a1 = x1 ? AV(x1) : ActView{}, r = res ? AV(res) : ActView{};
    const ActView* pa1 = x1 ? &a1 : nullptr;
    const ActView* pr = res ? &r : nullptr;
    bf16* o = static_cast<bf16*>(out->ptr);
    const bf16* w = static_cast<const bf16*>(wt);
    if (path == 0) {
        ConvHaloPlan hp;
        SNRSE_TRY(conv_halo2_make_plan(&hp, &a0, pa1, w, n, bias, tbias, tb_stride, pr, scale, o, out->ld, scsh,
                                       static_cast<unsigned long long*>(ustats)));
        return conv_halo2_launch(&hp, S(stream));
    }
    if (path == 1) return conv_simt_launch(&a0, taps0, pa1, w, n, bias, tbias, tb_stride, pr, scale, o, out->ld, S(stream));
    SNRSE_CHECK_ARG(path == 2, "dbg_conv: path must be 0, 1 or 2");
    ConvGemmPlan g;
    SNRSE_TRY(conv_gemm_make_plan(&g, &a0, taps0, pa1, w, n, 0, 0, bias, tbias, tb_stride, pr, scale, o, out->ld, 0));
    return conv_gemm_launch(&g, S(stream));
}

// The plan fields snrse_dbg_conv (path 0 / 2) or, for path 0 with n = 4, snrse_dbg_conv_out4 (out: the fp32 [B][H][W][4]
// result) makes for these views, from the launcher's own make_plan with the device's SM count; nothing is launched.
int snrse_dbg_conv_plan(const snrse_view* x0, int taps0, const snrse_view* x1, const void* wt, int n, const snrse_view* res,
                        const snrse_view* out, const float* scsh, int path, void* plan) {
    SNRSE_CHECK_ARG(x0 && wt && out && plan, "dbg_conv_plan: null pointer");
    const ActView a0 = AV(x0), a1 = x1 ? AV(x1) : ActView{}, r = res ? AV(res) : ActView{};
    const bf16* w = static_cast<const bf16*>(wt);
    ConvPlanFields* f = static_cast<ConvPlanFields*>(plan);
    if (path == 0 && n == 4) {
        ConvHaloPlan hp;
        float* o4 = static_cast<float*>(out->ptr);
        SNRSE_TRY(conv_halo2_make_plan_out4(&hp, &a0, w, o4 /* a bias pointer the plan only stores */, nullptr, o4, scsh));
        *f = conv_plan_fields(hp);
        return SNRSE_OK;
    }
    if (path == 0) {
        ConvHaloPlan hp;
        SNRSE_TRY(conv_halo2_make_plan(&hp, &a0, x1 ? &a1 : nullptr, w, n, nullptr, nullptr, 0, res ? &r : nullptr, 1.0f,
                                       static_cast<bf16*>(out->ptr), out->ld, scsh, nullptr));
        *f = conv_plan_fields(hp);
        return SNRSE_OK;
    }
    SNRSE_CHECK_ARG(path == 2 && !scsh, "dbg_conv_plan: path must be 0 or 2 (scsh: path 0 only)");
    ConvGemmPlan g;
    SNRSE_TRY(conv_gemm_make_plan(&g, &a0, taps0, x1 ? &a1 : nullptr, w, n, 0, 0, nullptr, nullptr, 0, res ? &r : nullptr,
                                  1.0f, out->ptr, out->ld, 0));
    *f = conv_plan_fields(g);
    return SNRSE_OK;
}

int snrse_dbg_gn_stats(const snrse_view* x, void* ustats, void* stream) {
    const ActView vx = AV(x);
    return gn_stats_launch(&vx, static_cast<unsigned long long*>(ustats), S(stream));
}

int snrse_dbg_gn_finalize(const void* src0, int U0, const void* src1, int U1, int B, int64_t count, const float* gamma,
                          const float* beta, float eps, float* scsh, void* stream) {
    return gn_finalize_launch(static_cast<const unsigned long long*>(src0), U0, static_cast<const unsigned long long*>(src1),
                              U1, B, count, gamma, beta, eps, scsh, S(stream));
}

int snrse_dbg_gn_apply(const snrse_view* x, const float* scsh, int silu, const snrse_view* out, void* stream) {
    const ActView vx = AV(x), vo = AV(out);
    return gn_apply_launch(&vx, scsh, silu, &vo, S(stream));
}

// not launched by the executor: the stand-alone single-output FIR that the dual pass is compared with
int snrse_dbg_fir(const snrse_view* x, const snrse_view* out, int up, void* stream) {
    const ActView vx = AV(x), vo = AV(out);
    return up ? fir_up2_launch(&vx, &vo, S(stream)) : fir_down2_launch(&vx, &vo, S(stream));
}

int snrse_dbg_fir_dual(const snrse_view* x, const snrse_view* out_n, const snrse_view* out_r, int up, const float* scsh,
                       void* stream) {
    const ActView vx = AV(x), vn = AV(out_n), vr = AV(out_r);
    return fir_dual_launch(&vx, &vn, &vr, up, scsh, S(stream));
}

// path 0: 2-CTA kernel, bf16 weights [16][9C] (rows 4..15 unused); path 1: CUDA cores, fp32 weights [4][3][3][C], which
// reads an operand that is already normalised (scsh must be null)
int snrse_dbg_conv_out4(const snrse_view* a, const void* w, const float* bias, const float* addend4, float* out4,
                        const float* scsh, int path, void* stream) {
    const ActView va = AV(a);
    if (path == 0) {
        ConvHaloPlan hp;
        SNRSE_TRY(conv_halo2_make_plan_out4(&hp, &va, static_cast<const bf16*>(w), bias, addend4, out4, scsh));
        return conv_halo2_launch(&hp, S(stream));
    }
    SNRSE_CHECK_ARG(path == 1 && !scsh, "dbg_conv_out4: path 1 takes no scsh");
    return conv_out4_launch(&va, static_cast<const float*>(w), bias, addend4, out4, S(stream));
}

// x64 null: pack_input_launch, otherwise pack_input64_launch
int snrse_dbg_pack_input(const void* x, const void* y, float* x4, void* x64, int B, int64_t n, void* stream) {
    if (!x64) return pack_input_launch(static_cast<const float2*>(x), static_cast<const float2*>(y), x4, B, n, S(stream));
    return pack_input64_launch(static_cast<const float2*>(x), static_cast<const float2*>(y), x4, static_cast<bf16*>(x64), B,
                               n, S(stream));
}

int snrse_dbg_conv_in4(const float* x4, const float* w, const float* bias, const snrse_view* out, void* stream) {
    const ActView vo = AV(out);
    return conv_in4_launch(x4, w, bias, &vo, S(stream));
}

int snrse_dbg_combine4(const float* p4, const snrse_view* h, const float* w, const float* bias, const snrse_view* out,
                       void* stream) {
    const ActView vh = AV(h), vo = AV(out);
    return combine4_launch(p4, &vh, w, bias, &vo, S(stream));
}

int snrse_dbg_temb(const float* t, int B, int nf, const float* fourier_w, const float* w1, const float* b1, const float* w2,
                   const float* b2, const float* dense_w, const float* dense_b, int rows, float* scratch, float* tb_out,
                   void* stream) {
    return temb_launch(t, B, nf, fourier_w, w1, b1, w2, b2, dense_w, dense_b, rows, scratch, tb_out, S(stream));
}

int snrse_dbg_final(const float* p4, const float* t, const float* w, const float* bias, const void* xres, void* out, int B,
                    int64_t n, int mode, void* stream) {
    return final_launch(p4, t, w, bias, static_cast<const float2*>(xres), static_cast<float2*>(out), B, n, mode, S(stream));
}

int snrse_dbg_attention(const snrse_view* q, const snrse_view* k, const snrse_view* v, void* workspace, const snrse_view* o,
                        int allow_tensor_cores, void* stream) {
    const ActView vq = AV(q), vk = AV(k), vv = AV(v), vo = AV(o);
    return attention_launch(&vq, &vk, &vv, workspace, &vo, S(stream), allow_tensor_cores);
}

}  // extern "C"
