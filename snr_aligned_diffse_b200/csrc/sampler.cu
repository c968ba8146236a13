// Element-wise kernels of the sampler (a7, a8, a18 of SURVEY 8a), complex64 state [B, F*T]:
//   pack_input : dnn_input = cat([x, y]) as 4 real channels (model.py:483, ncsnpp.py:253-254)
//   final      : h / t -> 1x1 conv 4->2 -> complex (ncsnpp.py:398-403) fused with the head:
//                  mode 0  raw network output
//                  mode 1  sebridge preconditioning  c_skip*x + c_out*dnn  (model.py:537-541)
//                  mode 2  bbed score  -dnn  (model.py:488-489)
//   lincomb    : x_mean = a*x + b*y + c*s,  x' = x_mean + d*z   -- covers prior sampling
//                (sdes.py:225-232), annealed Langevin (correctors.py:69-81) and the reverse-diffusion
//                predictor (predictors.py:75-80, sdes.py:73-91,132-140) with host-computed coefficients.
//   lincomb_keyed : the same with z drawn in the kernel from a per-item key (the keyed noise of snrse_b200.h).
#include "kernels.h"

namespace {

__global__ void __launch_bounds__(256)
pack_input_kernel(const float2* __restrict__ x, const float2* __restrict__ y, float4* __restrict__ x4, int64_t total) {
    pdl_sync();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const float2 a = x[i], b = y[i];
    x4[i] = make_float4(a.x, a.y, b.x, b.y);
}

// Same, plus the tensor-core operand of the input convolution: NHWC bf16 with 64 channels per pixel, channels 0..3 =
// bf16(v), 4..7 = bf16(v - bf16(v)) (hi/lo split: the first convolution sees ~16 mantissa bits of the spectrogram,
// its weights are duplicated over both halves), 8..63 = 0.  Thread = (pixel, 16-byte chunk).
__global__ void __launch_bounds__(256)
pack_input64_kernel(const float2* __restrict__ x, const float2* __restrict__ y, float4* __restrict__ x4,
                    uint4* __restrict__ x64, int64_t total) {
    pdl_sync();
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t i = idx >> 3;
    if (i >= total) return;
    const int chunk = (int)(idx & 7);
    uint4 o = make_uint4(0, 0, 0, 0);
    if (chunk == 0) {
        const float2 a = x[i], b = y[i];
        x4[i] = make_float4(a.x, a.y, b.x, b.y);
        const float v[4] = {a.x, a.y, b.x, b.y};
        float hi[4], lo[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            hi[k] = __bfloat162float(__float2bfloat16(v[k]));
            lo[k] = v[k] - hi[k];
        }
        const float f[8] = {hi[0], hi[1], hi[2], hi[3], lo[0], lo[1], lo[2], lo[3]};
        o = pack8(f);
    }
    x64[idx] = o;
}

__global__ void __launch_bounds__(256)
final_kernel(const float4* __restrict__ p4, const float* __restrict__ t, const float* __restrict__ w,
             const float* __restrict__ bias, const float2* __restrict__ xres, float2* __restrict__ out, int64_t n,
             int mode) {
    pdl_sync();
    const int b = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float tb = t[b];
    const float4 p = p4[(int64_t)b * n + i];
    const float hx = p.x / tb, hy = p.y / tb, hz = p.z / tb, hw = p.w / tb;
    float re = bias[0] + w[0] * hx + w[1] * hy + w[2] * hz + w[3] * hw;
    float im = bias[1] + w[4] * hx + w[5] * hy + w[6] * hz + w[7] * hw;
    if (mode == 1) {
        const float eps = 0.001f, sd = 0.5f;
        const float c_skip = sd * sd / ((tb - eps) * (tb - eps) + sd * sd);
        const float c_out = (sd * (tb - eps)) / sqrtf(sd * sd + tb * tb);
        const float2 xr = xres[(int64_t)b * n + i];
        re = c_skip * xr.x + c_out * re;
        im = c_skip * xr.y + c_out * im;
    } else if (mode == 2) {
        re = -re;
        im = -im;
    }
    out[(int64_t)b * n + i] = make_float2(re, im);
}

// Noise operand of lincomb_kernel.  NoiseIn reads z from memory (snrse_lincomb); NoiseKeyed draws it from
// (key[b], seed, element index) as snrse_b200.h specifies (snrse_lincomb_keyed).
struct NoiseIn {
    const float2* z;
    __device__ bool present() const { return z != nullptr; }
    __device__ bool item_ok(int) const { return true; }
    __device__ float2 operator()(int, int64_t, int64_t o) const { return __ldg(z + o); }
};

// Philox4x32-10 (Salmon et al., SC'11; curand's Philox4_32_10)
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return c;
}

struct NoiseKeyed {
    const unsigned long long* keys;
    unsigned long long seed;
    const int* len;    // optional: item b is NaN unless its own padded width equals tpad
    int tpad;
    float2* z_out;     // optional copy of the draw
    __device__ bool present() const { return true; }
    __device__ bool item_ok(int b) const { return !len || 64 * ((1 + len[b] / 128 + 63) / 64) == tpad; }
    __device__ float2 operator()(int b, int64_t i, int64_t o) const {
        const unsigned long long k = keys[b];
        const uint4 r = philox4x32_10(make_uint4((uint32_t)(i >> 1), 0u, (uint32_t)k, (uint32_t)(k >> 32)),
                                      (uint32_t)seed, (uint32_t)(seed >> 32));
        const uint32_t xa = (i & 1) ? r.z : r.x, xb = (i & 1) ? r.w : r.y;
        const float u1 = (float)((xa >> 8) + 1u) * 0x1p-24f;     // (0, 1], exact
        const float u2 = (float)(xb >> 8) * 0x1p-24f;            // [0, 1), exact
        const float rad = sqrtf(-logf(u1));
        float sn, cs;
        sincospif(2.f * u2, &sn, &cs);
        float2 v = make_float2(rad * cs, rad * sn);
        if (!item_ok(b)) v = make_float2(__int_as_float(0x7fc00000), __int_as_float(0x7fc00000));
        if (z_out) z_out[o] = v;
        return v;
    }
};

template <class Noise>
__global__ void __launch_bounds__(256)
lincomb_kernel(const float2* __restrict__ x, const float2* __restrict__ y, const float2* __restrict__ sc, Noise z,
               const float* __restrict__ a, const float* __restrict__ bq, const float* __restrict__ c,
               const float* __restrict__ d, float2* out_mean, float2* out_x, int64_t n) {
    pdl_sync();
    const int b = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t o = (int64_t)b * n + i;
    float re = 0.f, im = 0.f;
    if (x) { const float2 v = x[o]; const float k = a[b]; re = k * v.x; im = k * v.y; }
    if (y) { const float2 v = y[o]; const float k = bq[b]; re = fmaf(k, v.x, re); im = fmaf(k, v.y, im); }
    if (sc) { const float2 v = sc[o]; const float k = c[b]; re = fmaf(k, v.x, re); im = fmaf(k, v.y, im); }
    float2 zv = make_float2(0.f, 0.f);
    if (z.present()) zv = z(b, i, o);     // before the first store: NoiseIn's z must not wait for out_mean
    if (!z.item_ok(b)) re = im = __int_as_float(0x7fc00000);
    if (out_mean) out_mean[o] = make_float2(re, im);
    if (z.present()) { const float k = d[b]; re = fmaf(k, zv.x, re); im = fmaf(k, zv.y, im); }
    if (out_x) out_x[o] = make_float2(re, im);
}

// model.py:726-740 / 811-817 on device (no host sync): t_raw = ratio / (10^0.25 fixed_snr); snap to the
// nearest of the 30 float64 grid points (first minimum, like numpy argmin); normfac evaluated in
// float32 exactly as the reference's tensor arithmetic does.
__global__ void v3_scalars_kernel(const float* __restrict__ ratio, const float* __restrict__ peak, double snr_scale,
                                  float nf_const, const double* __restrict__ t30, float* __restrict__ t_out,
                                  float* __restrict__ nf_out, int* __restrict__ idx_out, int B) {
    pdl_sync();
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float t_raw = ratio[b] / (float)snr_scale;
    int best = 0;
    double bd = fabs(t30[0] - (double)t_raw);
    for (int i = 1; i < 30; ++i) {
        const double d = fabs(t30[i] - (double)t_raw);
        if (d < bd) {
            bd = d;
            best = i;
        }
    }
    const double t = t30[best];
    const float est = (float)(snr_scale * t);
    const float nf = nf_const / sqrtf(1.0f + est * est);
    t_out[b] = (float)t;
    nf_out[b] = peak[b] * nf;
    if (idx_out) idx_out[b] = best;
}

__global__ void snr_ratio_kernel(const float* __restrict__ g, float* __restrict__ ratio, int B) {
    pdl_sync();
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < B) ratio[b] = g[b] / (1.0f - g[b]);
}

// ---- embedded Runge-Kutta (Dormand-Prince 5(4)) helpers for the on-device probability-flow ODE sampler, replacing
// scipy.integrate.solve_ivp's numpy round trip per RHS evaluation (sampling/__init__.py:149-161).
struct RKCoef {
    float v[8];
};

// out = y + h * sum_{j<nk} c[j] * K[j]   (K: nk stage derivatives, n complex values each, back to back)
__global__ void __launch_bounds__(256)
rk_combine_kernel(const float2* __restrict__ y, const float2* __restrict__ K, int nk, float h, RKCoef c,
                  float2* __restrict__ out, int64_t n) {
    pdl_sync();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float re = 0.f, im = 0.f;
    for (int j = 0; j < nk; ++j) {
        if (c.v[j] == 0.f) continue;
        const float2 k = K[(int64_t)j * n + i];
        re = fmaf(c.v[j], k.x, re);
        im = fmaf(c.v[j], k.y, im);
    }
    float2 v = make_float2(h * re, h * im);
    if (y) { const float2 b = y[i]; v.x += b.x; v.y += b.y; }
    out[i] = v;
}

// partial[block] = sum over the block's elements of |h * sum_j c[j] K[j]|^2 / (atol + rtol * max(|y|, |y2|))^2 in
// double; fixed grid + fixed reduction tree, so the sum (and with it every accept / reject decision) is reproducible.
__global__ void __launch_bounds__(256)
rk_scaled_sqnorm_kernel(const float2* __restrict__ K, int nk, float h, RKCoef c, const float2* __restrict__ y,
                        const float2* __restrict__ y2, float atol, float rtol, double* __restrict__ partial, int64_t n) {
    pdl_sync();
    __shared__ double sm[8];
    double acc = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float re = 0.f, im = 0.f;
        for (int j = 0; j < nk; ++j) {
            if (c.v[j] == 0.f) continue;
            const float2 k = K[(int64_t)j * n + i];
            re = fmaf(c.v[j], k.x, re);
            im = fmaf(c.v[j], k.y, im);
        }
        re *= h;
        im *= h;
        const float2 a = y[i];
        float mag = sqrtf(a.x * a.x + a.y * a.y);
        if (y2) { const float2 b = y2[i]; mag = fmaxf(mag, sqrtf(b.x * b.x + b.y * b.y)); }
        const double sc = (double)atol + (double)rtol * (double)mag;
        acc += ((double)re * re + (double)im * im) / (sc * sc);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += sm[w];
        partial[blockIdx.x] = t;
    }
}

}  // namespace

int rk_combine_launch(const float2* y, const float2* K, int nk, int64_t n, float h, const float* coef, float2* out,
                      cudaStream_t s) {
    SNRSE_CHECK_ARG(K && out && coef && nk >= 1 && nk <= 8 && n > 0, "rk_combine: bad arguments (1..8 stages)");
    RKCoef c;
    for (int j = 0; j < 8; ++j) c.v[j] = j < nk ? coef[j] : 0.f;
    snrse_launch(rk_combine_kernel, dim3((unsigned)cdiv64(n, 256)), dim3(256), 0, s, y, K, nk, h, c, out, n);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}

int rk_partials(int64_t n) { return (int)(cdiv64(n, 256 * 8) < 1024 ? (cdiv64(n, 256 * 8) > 0 ? cdiv64(n, 256 * 8) : 1) : 1024); }

int rk_scaled_sqnorm_launch(const float2* K, int nk, int64_t n, float h, const float* coef, const float2* y,
                            const float2* y2, float atol, float rtol, double* partial, cudaStream_t s) {
    SNRSE_CHECK_ARG(K && y && coef && partial && nk >= 1 && nk <= 8 && n > 0, "rk_scaled_sqnorm: bad arguments");
    RKCoef c;
    for (int j = 0; j < 8; ++j) c.v[j] = j < nk ? coef[j] : 0.f;
    snrse_launch(rk_scaled_sqnorm_kernel, dim3(rk_partials(n)), dim3(256), 0, s, K, nk, h, c, y, y2, atol, rtol, partial, n);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}


int v3_scalars_launch(const float* ratio, const float* peak, double snr_scale, float nf_const, const double* t30,
                      float* t_out, float* nf_out, int* idx_out, int B, cudaStream_t s) {
    snrse_launch(v3_scalars_kernel, dim3(cdiv(B, 128)), dim3(128), 0, s, ratio, peak, snr_scale, nf_const, t30, t_out, nf_out, idx_out, B);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}

int snr_ratio_launch(const float* g, float* ratio, int B, cudaStream_t s) {
    snrse_launch(snr_ratio_kernel, dim3(cdiv(B, 128)), dim3(128), 0, s, g, ratio, B);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}

int pack_input_launch(const float2* x, const float2* y, float* x4, int B, int64_t n, cudaStream_t s) {
    const int64_t total = (int64_t)B * n;
    snrse_launch(pack_input_kernel, dim3((unsigned)cdiv64(total, 256)), dim3(256), 0, s, x, y, reinterpret_cast<float4*>(x4), total);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}

int pack_input64_launch(const float2* x, const float2* y, float* x4, bf16* x64, int B, int64_t n, cudaStream_t s) {
    const int64_t total = (int64_t)B * n;
    snrse_launch(pack_input64_kernel, dim3((unsigned)cdiv64(total * 8, 256)), dim3(256), 0, s, x, y, reinterpret_cast<float4*>(x4),
                                                                        reinterpret_cast<uint4*>(x64), total);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}

int final_launch(const float* p4, const float* t, const float* w, const float* bias, const float2* xres, float2* out,
                 int B, int64_t n, int mode, cudaStream_t s) {
    SNRSE_CHECK_ARG(mode >= 0 && mode <= 2, "final: bad mode %d", mode);
    SNRSE_CHECK_ARG(mode != 1 || xres, "final: mode 1 needs the residual state");
    dim3 grid((unsigned)cdiv64(n, 256), B);
    snrse_launch(final_kernel, dim3(grid), dim3(256), 0, s, reinterpret_cast<const float4*>(p4), t, w, bias, xres, out, n, mode);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}

int lincomb_launch(const float2* x, const float2* y, const float2* sc, const float2* z, const float* a, const float* b,
                   const float* c, const float* d, float2* out_mean, float2* out_x, int B, int64_t n, cudaStream_t s) {
    dim3 grid((unsigned)cdiv64(n, 256), B);
    snrse_launch(lincomb_kernel<NoiseIn>, dim3(grid), dim3(256), 0, s, x, y, sc, NoiseIn{z}, a, b, c, d, out_mean, out_x, n);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}

int lincomb_keyed_launch(const float2* x, const float2* y, const float2* sc, const float* a, const float* b,
                         const float* c, const float* d, const unsigned long long* keys, unsigned long long seed,
                         const int* len, int tpad, float2* z_out, float2* out_mean, float2* out_x, int B, int64_t n,
                         cudaStream_t s) {
    SNRSE_CHECK_ARG(keys && d, "lincomb_keyed: null keys or noise coefficient");
    SNRSE_CHECK_ARG(tpad >= 1 && n == 256 * (int64_t)tpad, "lincomb_keyed: n = %lld is not 256 x tpad (tpad %d)",
                    (long long)n, tpad);
    dim3 grid((unsigned)cdiv64(n, 256), B);
    snrse_launch(lincomb_kernel<NoiseKeyed>, dim3(grid), dim3(256), 0, s, x, y, sc, NoiseKeyed{keys, seed, len, tpad, z_out},
                 a, b, c, d, out_mean, out_x, n);
    SNRSE_LAUNCH_CHECK();
    return SNRSE_OK;
}
