"""Thin torch-tensor wrappers over the stand-alone C-ABI operators (device memory + streams only).

Every function enqueues on the current CUDA stream and returns torch tensors that own the output
memory.  No computation happens in Python/PyTorch here.
"""
import math
from ctypes import byref, c_int, c_int64, c_void_p, create_string_buffer

import numpy as np
import torch

from . import _lib

N_FFT, HOP, N_BINS = 510, 128, 256

# model.py:22-23 (float64)
T_30 = (0.001 ** (1 / 7) + (np.arange(1, 31) - 1) / (30 - 1) * (1 ** (1 / 7) - 0.001 ** (1 / 7))) ** 7


def n_frames(length):
    return 1 + length // HOP


def padded_frames(length, multiple=64):
    nf = n_frames(length)
    return multiple * ((nf + multiple - 1) // multiple)


def _lib_dev():
    lib = _lib.load()
    _lib.require_device()
    return lib


def stft(wave, lengths=None, scale=None, scale_is_divisor=True, tpad=None, transform=True, alpha=0.5, beta=0.15,
         planar=False, pad_multiple=64):
    """wave [B, L] f32 cuda -> complex64 [B, 256, Tpad] (or f32 [B, 2, 256, Tpad] if planar)."""
    lib = _lib_dev()
    assert wave.is_cuda and wave.dtype == torch.float32 and wave.dim() == 2
    wave = wave.contiguous()
    B, L = wave.shape
    if tpad is None:
        tpad = padded_frames(L, pad_multiple)
    if planar:
        out = torch.empty(B, 2, N_BINS, tpad, dtype=torch.float32, device=wave.device)
    else:
        out = torch.empty(B, N_BINS, tpad, dtype=torch.complex64, device=wave.device)
    _lib.check(lib.snrse_stft(_lib.ptr(wave), _lib.ptr(lengths), _lib.ptr(scale), int(scale_is_divisor), _lib.ptr(out),
                              B, L, tpad, int(transform), alpha, beta, int(planar), _lib.stream_ptr()), "stft")
    return out


def istft(spec, length, lengths=None, scale=None, transform=True, alpha=0.5, beta=0.15):
    """spec complex64 [B, 256, Tpad] cuda -> wave [B, length] f32."""
    lib = _lib_dev()
    assert spec.is_cuda and spec.dtype == torch.complex64 and spec.dim() == 3 and spec.shape[1] == N_BINS
    spec = spec.contiguous()
    B, _, tpad = spec.shape
    ws = torch.empty(int(lib.snrse_istft_workspace_bytes(B, tpad)), dtype=torch.uint8, device=spec.device)
    wave = torch.empty(B, length, dtype=torch.float32, device=spec.device)
    _lib.check(lib.snrse_istft(_lib.ptr(spec), _lib.ptr(lengths), _lib.ptr(scale), _lib.ptr(wave), _lib.ptr(ws), B,
                               length, tpad, int(transform), alpha, beta, _lib.stream_ptr()), "istft")
    return wave


def si_sdr(ref, est, lengths=None):
    """SI-SDR (dB, float64 [B]) of est [B, L] against ref [B, L] over the first lengths[b] samples, on the device."""
    lib = _lib_dev()
    assert ref.is_cuda and est.is_cuda and ref.shape == est.shape and ref.dim() == 2
    ref, est = ref.to(torch.float32).contiguous(), est.to(torch.float32).contiguous()
    out = torch.empty(ref.shape[0], dtype=torch.float64, device=ref.device)
    _lib.check(lib.snrse_si_sdr(_lib.ptr(ref), _lib.ptr(est), _lib.ptr(lengths), ref.shape[0], ref.shape[1], _lib.ptr(out),
                                _lib.stream_ptr()), "si_sdr")
    return out


def absmax(wave, lengths=None):
    lib = _lib_dev()
    wave = wave.contiguous()
    out = torch.empty(wave.shape[0], dtype=torch.float32, device=wave.device)
    _lib.check(lib.snrse_absmax(_lib.ptr(wave), _lib.ptr(lengths), wave.shape[0], wave.shape[1], _lib.ptr(out),
                                _lib.stream_ptr()), "absmax")
    return out


_t30_cache = {}


def v3_scalars(ratio, peak, fixed_snr):
    """ratio = noise/clean [B], peak = max|y| [B] (cuda f32) -> (t [B], norm_factor [B], index [B])."""
    lib = _lib_dev()
    dev = ratio.device
    if dev not in _t30_cache:
        _t30_cache[dev] = torch.from_numpy(T_30.copy()).to(dev)
    B = ratio.numel()
    t = torch.empty(B, dtype=torch.float32, device=dev)
    nf = torch.empty(B, dtype=torch.float32, device=dev)
    idx = torch.empty(B, dtype=torch.int32, device=dev)
    snr_scale = 10 ** 0.25 * fixed_snr
    nf_const = float(np.float32(2.040166 * (0.240253 + 0.759747 * fixed_snr ** 2) ** 0.5))
    _lib.check(lib.snrse_v3_scalars(_lib.ptr(ratio.contiguous()), _lib.ptr(peak.contiguous()), snr_scale, nf_const,
                                    _lib.ptr(_t30_cache[dev]), _lib.ptr(t), _lib.ptr(nf), _lib.ptr(idx), B,
                                    _lib.stream_ptr()), "v3_scalars")
    return t, nf, idx


def _lincomb_operands(name, ops_):
    """Validated operands of lincomb / lincomb_keyed: (first operand, B, {key: tensor}, {key: coefficient})."""
    present = [(k, t, co) for k, (t, co) in ops_.items() if t is not None]
    if not present:
        raise ValueError(f"{name}: no operand given")
    ref = present[0][1]
    B = ref.shape[0]
    tensors, coefs = {}, {}
    for k, t, co in present:
        if not (torch.is_tensor(t) and t.is_cuda and t.dtype == torch.complex64):
            raise ValueError(f"{name}: operand {k} must be a CUDA complex64 tensor (got "
                             f"{getattr(t, 'dtype', type(t))} on {getattr(t, 'device', 'host')})")
        if t.shape != ref.shape or t.device != ref.device:
            raise ValueError(f"{name}: operand {k} has shape {tuple(t.shape)} on {t.device}, expected "
                             f"{tuple(ref.shape)} on {ref.device} (operands must match exactly; no broadcasting)")
        if co is None or not (torch.is_tensor(co) and co.is_cuda and co.dtype == torch.float32 and co.numel() == B):
            raise ValueError(f"{name}: coefficient of {k} must be a CUDA float32 vector with {B} elements")
        tensors[k], coefs[k] = t.contiguous(), co.contiguous()
    return ref, B, tensors, coefs


def lincomb(x=None, y=None, s=None, z=None, a=None, b=None, c=None, d=None, want_mean=True, want_x=True):
    """out_mean = a x + b y + c s; out_x = out_mean + d z  on complex64 [B, ...] tensors; a..d are [B] float32
    coefficient vectors (one per operand present).  Every sampler state update is built on this call, so operands are
    validated here: all on one CUDA device, complex64, identical shapes (the reference's elementwise ops would raise a
    broadcast error on a mismatch), made contiguous before their raw pointers are handed to the kernel."""
    lib = _lib_dev()
    ref, B, tensors, coefs = _lincomb_operands("lincomb", {"x": (x, a), "y": (y, b), "s": (s, c), "z": (z, d)})
    n = ref.numel() // B
    shape = ref.shape
    out_mean = torch.empty(shape, dtype=torch.complex64, device=ref.device) if want_mean else None
    out_x = torch.empty(shape, dtype=torch.complex64, device=ref.device) if want_x else None
    g = lambda d_, k: d_.get(k)  # noqa: E731
    _lib.check(lib.snrse_lincomb(_lib.ptr(g(tensors, "x")), _lib.ptr(g(tensors, "y")), _lib.ptr(g(tensors, "s")),
                                 _lib.ptr(g(tensors, "z")), _lib.ptr(g(coefs, "x")), _lib.ptr(g(coefs, "y")),
                                 _lib.ptr(g(coefs, "s")), _lib.ptr(g(coefs, "z")), _lib.ptr(out_mean), _lib.ptr(out_x), B, n,
                                 _lib.stream_ptr()), "lincomb")
    return out_mean, out_x


def key_tensor(keys, B=None):
    """Per-item 64-bit noise keys as an int64 tensor (the kernel reads its bits as uint64).  keys: a sequence of Python
    ints in [-2^63, 2^64) (values >= 2^63 wrap to their two's complement) or an integer tensor, host or device."""
    if torch.is_tensor(keys):
        if keys.dtype not in (torch.int64, torch.int32, torch.int16, torch.int8, torch.uint8):
            raise ValueError(f"keys must be an integer tensor (got {keys.dtype})")
        kt = keys.reshape(-1).to(torch.int64)
    else:
        vals = [int(k) for k in keys]
        if any(not -(1 << 63) <= k < (1 << 64) for k in vals):
            raise ValueError("keys must lie in [-2^63, 2^64)")
        kt = torch.tensor([k - (1 << 64) if k >= (1 << 63) else k for k in vals], dtype=torch.int64)
    if B is not None and kt.numel() != B:
        raise ValueError(f"keys: expected {B} keys, got {kt.numel()}")
    return kt


def lincomb_keyed(x=None, y=None, s=None, a=None, b=None, c=None, d=None, keys=None, seed=0, lengths=None,
                  want_mean=True, want_x=True, want_z=False):
    """`lincomb` with z drawn in the kernel from the keyed noise of include/snrse_b200.h: item b's draw depends on
    (keys[b], seed, element index) only.  Operands complex64 [B, ..., 256, Tpad]; d: [B] float32 coefficient of the
    draw; keys: int64 [B] (CUDA, read as uint64; see `key_tensor`); seed: int in [0, 2^64); lengths: optional CUDA int32
    [B], items whose own padded width is not Tpad come out NaN.  Returns (out_mean, out_x, z)."""
    lib = _lib_dev()
    ref, B, tensors, coefs = _lincomb_operands("lincomb_keyed", {"x": (x, a), "y": (y, b), "s": (s, c)})
    if ref.dim() < 3 or ref.shape[-2] != N_BINS or ref.numel() // B != N_BINS * ref.shape[-1]:
        raise ValueError(f"lincomb_keyed: operands must be [B, ..., {N_BINS}, Tpad] (got {tuple(ref.shape)})")
    if d is None or not (torch.is_tensor(d) and d.is_cuda and d.dtype == torch.float32 and d.numel() == B):
        raise ValueError(f"lincomb_keyed: coefficient of z must be a CUDA float32 vector with {B} elements")
    if not (torch.is_tensor(keys) and keys.is_cuda and keys.dtype == torch.int64 and keys.numel() == B
            and keys.device == ref.device):
        raise ValueError(f"lincomb_keyed: keys must be a CUDA int64 vector with {B} elements on {ref.device}")
    if lengths is not None and not (torch.is_tensor(lengths) and lengths.is_cuda and lengths.dtype == torch.int32
                                    and lengths.numel() == B):
        raise ValueError(f"lincomb_keyed: lengths must be a CUDA int32 vector with {B} elements")
    seed = int(seed)
    if not 0 <= seed < (1 << 64):
        raise ValueError(f"lincomb_keyed: seed must lie in [0, 2^64) (got {seed})")
    tpad = ref.shape[-1]
    n = ref.numel() // B
    shape = ref.shape
    new = lambda on: torch.empty(shape, dtype=torch.complex64, device=ref.device) if on else None  # noqa: E731
    out_mean, out_x, z = new(want_mean), new(want_x), new(want_z)
    g = lambda d_, k: d_.get(k)  # noqa: E731
    _lib.check(lib.snrse_lincomb_keyed(_lib.ptr(g(tensors, "x")), _lib.ptr(g(tensors, "y")), _lib.ptr(g(tensors, "s")),
                                       _lib.ptr(g(coefs, "x")), _lib.ptr(g(coefs, "y")), _lib.ptr(g(coefs, "s")),
                                       _lib.ptr(d.contiguous()), _lib.ptr(keys.contiguous()), seed,
                                       _lib.ptr(None if lengths is None else lengths.contiguous()), tpad, _lib.ptr(z),
                                       _lib.ptr(out_mean), _lib.ptr(out_x), B, n, _lib.stream_ptr()), "lincomb_keyed")
    return out_mean, out_x, z


def rk_combine(y, K, coef, h):
    """y + h * sum_j coef[j] * K[j]; K complex64 [nk, ...] (stages), y complex64 [...] or None."""
    import ctypes
    lib = _lib_dev()
    nk = len(coef)
    n = K[0].numel()
    out = torch.empty_like(K[0])
    c = (ctypes.c_float * nk)(*[float(v) for v in coef])
    _lib.check(lib.snrse_rk_combine(_lib.ptr(y), _lib.ptr(K), nk, n, float(h), c, _lib.ptr(out), _lib.stream_ptr()),
               "rk_combine")
    return out


def rk_scaled_norm(K, coef, h, y, y2, atol, rtol):
    """RMS of (h * sum_j coef[j] K[j]) / (atol + rtol * max(|y|, |y2|)) over all complex elements (host float).
    One device->host read of <= 1024 block sums, added on the host in a fixed order."""
    import ctypes
    import math
    lib = _lib_dev()
    nk = len(coef)
    n = K[0].numel()
    part = torch.empty(int(lib.snrse_rk_partials(n)), dtype=torch.float64, device=K.device)
    c = (ctypes.c_float * nk)(*[float(v) for v in coef])
    _lib.check(lib.snrse_rk_scaled_sqnorm(_lib.ptr(K), nk, n, float(h), c, _lib.ptr(y), _lib.ptr(y2), float(atol),
                                          float(rtol), _lib.ptr(part), _lib.stream_ptr()), "rk_scaled_sqnorm")
    return math.sqrt(math.fsum(part.cpu().tolist()) / n)


# ------------------------------------------------------------------------------ single NHWC operators
def conv_nhwc(x0, wt, taps0, x1=None, bias=None, tbias=None, res=None, scale=1.0, impl=0):
    """x0 [B,H,W,C0] bf16, wt [N, taps0*C0 (+C1)] bf16 K-major -> [B,H,W,N] bf16."""
    lib = _lib_dev()
    B, H, W, C0 = x0.shape
    N = wt.shape[0]
    out = torch.empty(B, H, W, N, dtype=torch.bfloat16, device=x0.device)
    _lib.check(lib.snrse_conv_nhwc(_lib.ptr(x0), C0, taps0, _lib.ptr(x1), 0 if x1 is None else x1.shape[-1],
                                   _lib.ptr(wt), N, _lib.ptr(bias), _lib.ptr(tbias),
                                   0 if tbias is None else tbias.shape[-1], _lib.ptr(res), scale, _lib.ptr(out), B, H, W,
                                   impl, _lib.stream_ptr()), "conv_nhwc")
    return out


def groupnorm_nhwc(x, gamma, beta, silu=True, eps=1e-6):
    lib = _lib_dev()
    B, H, W, C = x.shape
    out = torch.empty_like(x)
    ws = torch.empty(int(lib.snrse_groupnorm_workspace_bytes(B)), dtype=torch.uint8, device=x.device)
    _lib.check(lib.snrse_groupnorm_nhwc(_lib.ptr(x), _lib.ptr(gamma), _lib.ptr(beta), _lib.ptr(out), B, H, W, C,
                                        int(silu), eps, _lib.ptr(ws), _lib.stream_ptr()), "groupnorm")
    return out


def gn_silu_conv3x3_nhwc(x0, gamma, beta, wt, x1=None, bias=None, tbias=None, res=None, scale=1.0, eps=1e-6):
    """conv3x3(silu(GroupNorm32(x0))) (+ 1x1 shortcut on x1, bias, tbias, residual, * scale) in one pass."""
    lib = _lib_dev()
    B, H, W, C0 = x0.shape
    N = wt.shape[0]
    out = torch.empty(B, H, W, N, dtype=torch.bfloat16, device=x0.device)
    ws = torch.empty(int(lib.snrse_groupnorm_workspace_bytes(B)), dtype=torch.uint8, device=x0.device)
    _lib.check(lib.snrse_gn_silu_conv3x3_nhwc(_lib.ptr(x0), C0, _lib.ptr(gamma), _lib.ptr(beta), eps, _lib.ptr(x1),
                                              0 if x1 is None else x1.shape[-1], _lib.ptr(wt), N, _lib.ptr(bias),
                                              _lib.ptr(tbias), 0 if tbias is None else tbias.shape[-1], _lib.ptr(res),
                                              scale, _lib.ptr(out), B, H, W, _lib.ptr(ws), _lib.stream_ptr()),
               "gn_silu_conv3x3")
    return out


def conv3x3_nhwc_stats(x0, wt, x1=None, bias=None, tbias=None, res=None, scale=1.0):
    """conv3x3 on the 2-CTA kernel; also returns the per-unit (4 channels) sums / sums of squares of the result as
    [B, N/4, 2] float64 (decoded from the kernel's 64-bit fixed-point accumulators) and the raw int64 tensor."""
    lib = _lib_dev()
    B, H, W, C0 = x0.shape
    N = wt.shape[0]
    out = torch.empty(B, H, W, N, dtype=torch.bfloat16, device=x0.device)
    ust = torch.empty(B, N // 4, 2, dtype=torch.int64, device=x0.device)
    _lib.check(lib.snrse_conv3x3_nhwc_stats(_lib.ptr(x0), C0, _lib.ptr(x1), 0 if x1 is None else x1.shape[-1],
                                            _lib.ptr(wt), N, _lib.ptr(bias), _lib.ptr(tbias),
                                            0 if tbias is None else tbias.shape[-1], _lib.ptr(res), scale, _lib.ptr(out),
                                            B, H, W, _lib.ptr(ust), _lib.stream_ptr()), "conv3x3_stats")
    dec = ust.double() * torch.tensor([2.0 ** -30, 2.0 ** -20], dtype=torch.float64, device=x0.device)   # gn_fixed.cuh scales
    return out, dec, ust


def fir_nhwc(x, up):
    lib = _lib_dev()
    B, H, W, C = x.shape
    if x.dtype == torch.bfloat16:
        out = torch.empty((B, 2 * H, 2 * W, C) if up else (B, H // 2, W // 2, C), dtype=x.dtype, device=x.device)
        _lib.check(lib.snrse_fir_nhwc(_lib.ptr(x), _lib.ptr(out), B, H, W, C, int(up), _lib.stream_ptr()), "fir")
    else:
        assert C == 4 and x.dtype == torch.float32
        out = torch.empty((B, 2 * H, 2 * W, 4) if up else (B, H // 2, W // 2, 4), dtype=x.dtype, device=x.device)
        _lib.check(lib.snrse_fir_f4(_lib.ptr(x), _lib.ptr(out), B, H, W, int(up), _lib.stream_ptr()), "fir_f4")
    return out


def upfirdn2d(input, kernel, up=(1, 1), down=(1, 1), pad=(0, 0, 0, 0)):
    """General upfirdn2d (op/upfirdn2d.cpp:12-23): input [N, C, H, W], kernel [kh, kw], up / down = (x, y),
    pad = (x0, x1, y0, y1) -> [N, C, out_h, out_w] in the input's dtype and on the input's device."""
    lib = _lib_dev()
    if input.dim() != 4 or kernel.dim() != 2:
        raise RuntimeError("upfirdn2d: input must be [N, C, H, W] and kernel [kh, kw]")
    dev, dt = input.device, input.dtype
    x = input.to("cuda", torch.float32).contiguous()
    k = kernel.to("cuda", torch.float32).contiguous()
    N, C, H, W = x.shape
    kh, kw = k.shape
    (ux, uy), (dx, dy), (px0, px1, py0, py1) = up, down, pad
    if min(ux, uy, dx, dy) < 1:
        raise RuntimeError("upfirdn2d: up / down factors must be >= 1")
    oh = (H * uy + py0 + py1 - kh) // dy + 1
    ow = (W * ux + px0 + px1 - kw) // dx + 1
    if N * C == 0 or H * uy + py0 + py1 < kh or W * ux + px0 + px1 < kw:
        raise RuntimeError("upfirdn2d: padded input smaller than the kernel")
    out = torch.empty(N, C, oh, ow, dtype=torch.float32, device=x.device)
    _lib.check(lib.snrse_upfirdn2d(_lib.ptr(x), _lib.ptr(k), _lib.ptr(out), N * C, H, W, kh, kw, ux, uy, dx, dy, px0, px1,
                                   py0, py1, _lib.stream_ptr()), "upfirdn2d")
    return out.to(dev, dt)


def attention_nhwc(q, k, v):
    """q,k,v [B, n, C] bf16 -> [B, n, C] bf16."""
    lib = _lib_dev()
    B, n, C = q.shape
    scores = torch.empty(int(lib.snrse_attention_workspace_bytes(B, n, C)), dtype=torch.uint8, device=q.device)
    out = torch.empty_like(q)
    _lib.check(lib.snrse_attention_nhwc(_lib.ptr(q), _lib.ptr(k), _lib.ptr(v), _lib.ptr(scores), _lib.ptr(out), B, n, C,
                                        _lib.stream_ptr()), "attention")
    return out


# ------------------------------------------------------------------------------ SNR estimator
class SNRNetEngine:
    """Packed SNRNet weights on one GPU + forward (backbones/snrnet.py:47-97)."""

    def __init__(self):
        self.lib = _lib.load()
        self.blob = None

    def param_table(self):
        out = []
        name = create_string_buffer(256)
        off, numel, tr = c_int64(), c_int64(), c_int()
        for i in range(self.lib.snrse_snrnet_num_params()):
            _lib.check(self.lib.snrse_snrnet_param_info(i, name, 256, byref(off), byref(numel), byref(tr)), "snrnet_param_info")
            dims, nd = (c_int64 * 4)(), c_int()
            _lib.check(self.lib.snrse_snrnet_param_shape(i, dims, byref(nd)), "snrnet_param_shape")
            out.append(dict(name=name.value.decode(), offset=off.value, numel=numel.value, transform=tr.value,
                            shape=tuple(int(dims[j]) for j in range(nd.value))))
        return out

    def param_shapes(self):
        return {p["name"]: p["shape"] for p in self.param_table()}

    def load_state_dict(self, sd, device="cuda"):
        _lib.require_device()
        blob = torch.zeros(int(self.lib.snrse_snrnet_weight_bytes()), dtype=torch.uint8)
        f32 = blob.view(torch.float32)
        for p in self.param_table():
            w = sd[p["name"]].detach().to("cpu", torch.float32)
            if p["transform"] == 1:   # (64 x k) convolutions: [co][ci][f][dt] -> [ci*64 + f][dt][co]
                co, ci, f, k = w.shape
                w = w.reshape(co, ci * f, k).permute(1, 2, 0).contiguous()
            elif p["transform"] == 2:   # conv3x3: [co][ci][3][3] -> [ci][tap][co]
                co, ci = w.shape[0], w.shape[1]
                w = w.reshape(co, ci, 9).permute(1, 2, 0).contiguous()
            w = w.reshape(-1)
            assert w.numel() == p["numel"], p["name"]
            f32[p["offset"] // 4: p["offset"] // 4 + w.numel()].copy_(w)
        self.blob = blob.to(device)
        return self

    def forward(self, feat, clusters=None):
        """feat f32 [B,2,256,T16] cuda -> [B] = noise/(speech+noise).  clusters: optional int32 [B] cuda, the valid
        16-frame clusters of each item (read clamped to [1, T16/16]); item b is then estimated over its first
        clusters[b] clusters only, as if it had been run alone at T16 = 16 * clusters[b]."""
        assert self.blob is not None and feat.is_cuda and feat.dtype == torch.float32
        feat = feat.contiguous()
        B, _, _, T16 = feat.shape
        if clusters is not None and not (torch.is_tensor(clusters) and clusters.device == feat.device
                                         and clusters.dtype == torch.int32 and clusters.numel() == B):
            raise ValueError(f"snrnet forward: clusters must be an int32 tensor of {B} elements on {feat.device}")
        clusters = None if clusters is None else clusters.contiguous()
        ws = torch.empty(int(self.lib.snrse_snrnet_workspace_bytes(B, T16)), dtype=torch.uint8, device=feat.device)
        out = torch.empty(B, dtype=torch.float32, device=feat.device)
        if clusters is None:
            _lib.check(self.lib.snrse_snrnet_forward(_lib.ptr(self.blob), _lib.ptr(feat), _lib.ptr(out), B, T16,
                                                     _lib.ptr(ws), _lib.stream_ptr()), "snrnet_forward")
        else:
            _lib.check(self.lib.snrse_snrnet_forward_varlen(_lib.ptr(self.blob), _lib.ptr(feat),
                                                            _lib.ptr(clusters), _lib.ptr(out), B, T16,
                                                            _lib.ptr(ws), _lib.stream_ptr()), "snrnet_forward_varlen")
        return out

    def noise_over_clean(self, g):
        out = torch.empty_like(g)
        _lib.check(self.lib.snrse_snr_ratio(_lib.ptr(g), _lib.ptr(out), g.numel(), _lib.stream_ptr()), "snr_ratio")
        return out
