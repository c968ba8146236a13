"""Every launcher of the NCSN++ executor, called through the snrse_dbg_* entry points on the views the executor passes
(run with -m gpu on a B200).

The executor rarely hands a kernel a dense tensor: skip tensors live in channel slices of the decoder's concatenation
buffers (ld > C, pointer offset by the slice's first channel), GroupNorm over cat([h, skip]) is finalised from two
statistics sources, and attention reads q, k and v inside one fused qkv buffer (ld = 3C).  These tests run each
launcher on such views and check

  A. slices: the result on a slice is bit-identical to the same launcher on dense copies, every channel outside the
     written slice still holds a bf16 NaN sentinel, and the sentinel in the neighbours of an input slice (which any
     over-read would pull in as NaN) never reaches the output;
  B. the two-source GroupNorm finalize: the same scale/shift bits as one source over a dense copy of the
     concatenation, and the normalised result against fp64 group_norm;
  C. the thin layers (input packing, input convolution, input pyramid, output head, time embedding, final head)
     against float64 references computed from exactly the operands the kernel reads.  Bounds are stated per test in
     terms of A = the same expression evaluated on absolute values (sum |w||x| + |bias| + ...).  Where the result is
     stored in bf16, the 2^-8 |ref| term is the unit roundoff of that rounding itself, so those checks sit just below
     err/bound = 1 by construction; the A term bounds the accumulation;
  D. one decoder residual block composed from the launchers in the executor's order, against the fp64 oracle.
"""
import ctypes
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ncsnpp as o_ncsnpp

pytestmark = pytest.mark.gpu

DEV = "cuda"
SENT = 0x7FD5            # bf16 quiet NaN with a payload no kernel produces: marks channels nobody may write
F64 = torch.float64


# ----------------------------------------------------------------------------------------------- bindings
class View(ctypes.Structure):
    """snrse_view (include/snrse_b200_layers.h)."""
    _fields_ = [("ptr", ctypes.c_void_p), ("B", ctypes.c_int), ("H", ctypes.c_int), ("W", ctypes.c_int),
                ("C", ctypes.c_int), ("ld", ctypes.c_int)]


@pytest.fixture(scope="module")
def lib():
    from snr_aligned_diffse_b200 import _lib
    lib = _lib.load()
    _lib.require_device()
    return lib


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _ref(v):
    return None if v is None else ctypes.byref(v)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _check(lib, status, what):
    assert status == 0, f"{what}: {lib.snrse_last_error().decode(errors='replace')}"


def dense(t):
    """snrse_view of a contiguous bf16 [B, H, W, C] tensor."""
    assert t.is_contiguous() and t.dtype == torch.bfloat16 and t.dim() == 4
    B, H, W, C = t.shape
    return View(t.data_ptr(), B, H, W, C, C)


class Slice:
    """Channels [coff, coff + C) of a bf16 parent buffer [B, H, W, coff + C + after]: a channel slice of a concatenation
    buffer as the executor's views are.  Every channel outside the slice holds the NaN sentinel."""

    def __init__(self, B, H, W, C, coff=64, after=64, data=None):
        self.parent = torch.empty(B, H, W, coff + C + after, dtype=torch.bfloat16, device=DEV)
        self.parent.view(torch.int16).fill_(SENT)
        self.coff, self.C = coff, C
        if data is not None:
            self.t.copy_(data)

    @property
    def t(self):
        return self.parent[..., self.coff:self.coff + self.C]

    def view(self):
        B, H, W, ld = self.parent.shape
        return View(self.parent.data_ptr() + 2 * self.coff, B, H, W, self.C, ld)

    def intact(self):
        bits = self.parent.view(torch.int16)
        return bool((bits[..., :self.coff] == SENT).all()) and bool((bits[..., self.coff + self.C:] == SENT).all())


def conv(lib, x0, wt, n, taps=9, x1=None, bias=None, tbias=None, tb_stride=0, res=None, scale=1.0, out=None, scsh=None,
         ustats=None, path=0):
    _check(lib, lib.snrse_dbg_conv(_ref(x0), taps, _ref(x1), _ptr(wt), n, _ptr(bias), _ptr(tbias), tb_stride, _ref(res),
                                   scale, _ref(out), _ptr(scsh), _ptr(ustats), path, _stream()), f"dbg_conv path {path}")


def gn_stats(lib, x, B, C):
    ust = torch.zeros(B, C // 4, 2, dtype=torch.int64, device=DEV)
    _check(lib, lib.snrse_dbg_gn_stats(_ref(x), _ptr(ust), _stream()), "dbg_gn_stats")
    return ust


def gn_finalize(lib, src0, src1, B, count, gamma, beta, eps=1e-6):
    U0, U1 = src0.shape[1], 0 if src1 is None else src1.shape[1]
    scsh = torch.empty(B, 2, 4 * (U0 + U1), dtype=torch.float32, device=DEV)
    _check(lib, lib.snrse_dbg_gn_finalize(_ptr(src0), U0, _ptr(src1), U1, B, count, _ptr(gamma), _ptr(beta), eps,
                                          _ptr(scsh), _stream()), "dbg_gn_finalize")
    return scsh


def gn_apply(lib, x, scsh, silu, out):
    _check(lib, lib.snrse_dbg_gn_apply(_ref(x), _ptr(scsh), int(silu), _ref(out), _stream()), "dbg_gn_apply")


def fir(lib, x, out, up):
    _check(lib, lib.snrse_dbg_fir(_ref(x), _ref(out), int(up), _stream()), "dbg_fir")


def fir_dual(lib, x, out_n, out_r, up, scsh):
    _check(lib, lib.snrse_dbg_fir_dual(_ref(x), _ref(out_n), _ref(out_r), int(up), _ptr(scsh), _stream()), "dbg_fir_dual")


def fir_f4(lib, x, up):
    B, H, W, _ = x.shape
    out = torch.empty((B, 2 * H, 2 * W, 4) if up else (B, H // 2, W // 2, 4), dtype=torch.float32, device=DEV)
    _check(lib, lib.snrse_fir_f4(_ptr(x), _ptr(out), B, H, W, int(up), _stream()), "fir_f4")
    return out


def conv_out4(lib, a, w, bias, addend4, scsh, path, B, H, W):
    out4 = torch.empty(B, H, W, 4, dtype=torch.float32, device=DEV)
    _check(lib, lib.snrse_dbg_conv_out4(_ref(a), _ptr(w), _ptr(bias), _ptr(addend4), _ptr(out4), _ptr(scsh), path,
                                        _stream()), f"dbg_conv_out4 path {path}")
    return out4


def bits(t):
    return t.contiguous().view(torch.int16 if t.element_size() == 2 else torch.int32)


def same_bits(a, b):
    return torch.equal(bits(a), bits(b))


def within(err, bound, what):
    """err <= bound everywhere; prints the worst err / bound ratio (the margin of the bound)."""
    ratio = float((err / bound).max())
    print(f"{what}: max err/bound = {ratio:.3g}")
    assert ratio <= 1.0, f"{what}: max err/bound = {ratio:.3g}"


def bf16(g, *shape, scale=1.0, shift=0.0):
    return (torch.randn(*shape, generator=g) * scale + shift).to(torch.bfloat16).to(DEV)


def pack_w3(w):  # [Cout, Cin, 3, 3] -> [Cout, 9 * Cin] (tap-major, cin inner)
    return w.permute(0, 2, 3, 1).reshape(w.shape[0], -1).contiguous()


def conv_ref(x, w, bias=None, pad=1):
    """fp64 convolution of an NHWC operand with [Cout, Cin, k, k] weights -> NHWC."""
    y = F.conv2d(x.to(DEV, F64).permute(0, 3, 1, 2), w.to(DEV, F64), None if bias is None else bias.to(DEV, F64),
                 padding=pad)
    return y.permute(0, 2, 3, 1)


def gn_params(g, C):
    return (torch.rand(C, generator=g) + 0.5).to(DEV), (torch.randn(C, generator=g) * 0.2).to(DEV)


# ----------------------------------------------------------------------------------------------- A. slices
# B, H, W, Cin, Cout, taps: the edge shapes of test_gpu_parity.CONV_CASES
SLICE_CONV_CASES = [
    (2, 32, 64, 128, 128, 9),
    (1, 24, 40, 128, 256, 9),      # ragged tiles (H % 16 != 0, W % 16 != 0)
    (2, 8, 16, 512, 256, 9),       # H = 8: one sub-tile
    (2, 40, 12, 128, 128, 9),      # W % 8 != 0
    (3, 72, 20, 128, 256, 9),      # odd tile count: the peer CTA of the last pair runs an all-padding tile
    (1, 4, 3, 512, 256, 9),        # below the 2-CTA kernel's tiles
    (3, 4, 1, 256, 256, 1),
]


@pytest.mark.parametrize("path", [0, 1, 2], ids=["halo2", "cudacore", "gemm"])
@pytest.mark.parametrize("case", SLICE_CONV_CASES)
def test_conv_on_slices_equals_dense(lib, case, path):
    """Input, shortcut, residual and output as channel slices (offset > 0, ld > C) == the same launcher on dense copies,
    bit for bit, with and without shortcut, residual, time-embedding bias, in-flight GroupNorm and epilogue sums."""
    B, H, W, Ci, Co, taps = case
    if path == 0 and not (taps == 9 and H >= 8 and W >= 8):
        pytest.skip("the 2-CTA kernel needs a 3x3 convolution on an H, W >= 8 map")
    g = torch.Generator().manual_seed(sum(case) + path)
    Cs = 128
    x, xs = bf16(g, B, H, W, Ci, scale=1.3, shift=0.2), bf16(g, B, H, W, Cs)
    res = bf16(g, B, H, W, Co)
    w = (torch.randn(Co, taps * Ci + Cs, generator=g) / math.sqrt(taps * Ci + Cs)).to(torch.bfloat16).to(DEV)
    w0 = w[:, :taps * Ci].contiguous()
    bias = (torch.randn(Co, generator=g) * 0.1).to(DEV)
    tb_stride = Co + 40                            # a block's rows inside the concatenated Dense_0 output
    tball = (torch.randn(B, tb_stride, generator=g) * 0.2).to(DEV)
    tb = tball[:, 24:]
    gamma, beta = gn_params(g, Ci)
    scsh = gn_finalize(lib, gn_stats(lib, dense(x), B, Ci), None, B, H * W * Ci // 32, gamma, beta)
    variants = {"plain": dict(wt=w0),
                "shortcut+tbias": dict(wt=w, x1=xs, tbias=tb, tb_stride=tb_stride),
                "residual+tbias+scale": dict(wt=w0, res=res, tbias=tb, tb_stride=tb_stride, scale=0.7)}
    if path == 0:
        variants["gn-in-flight+shortcut+stats"] = dict(wt=w, x1=xs, scsh=scsh, stats=True, scale=0.7)
        variants["residual+stats"] = dict(wt=w0, res=res, stats=True)
    for name, v in variants.items():
        kw = dict(n=Co, taps=taps, bias=bias, tbias=v.get("tbias"), tb_stride=v.get("tb_stride", 0),
                  scale=v.get("scale", 1.0), scsh=v.get("scsh"), path=path)
        sx, sxs, sres = Slice(B, H, W, Ci, data=x), Slice(B, H, W, Cs, coff=128, after=0, data=xs), \
            Slice(B, H, W, Co, coff=256, after=8, data=res)
        sout = Slice(B, H, W, Co, coff=128, after=64)
        ust_s = torch.zeros(B, Co // 4, 2, dtype=torch.int64, device=DEV) if v.get("stats") else None
        ust_d = torch.zeros_like(ust_s) if v.get("stats") else None
        conv(lib, sx.view(), v["wt"], x1=sxs.view() if "x1" in v else None, res=sres.view() if "res" in v else None,
             out=sout.view(), ustats=ust_s, **kw)
        dout = torch.empty(B, H, W, Co, dtype=torch.bfloat16, device=DEV)
        conv(lib, dense(x), v["wt"], x1=dense(xs) if "x1" in v else None, res=dense(res) if "res" in v else None,
             out=dense(dout), ustats=ust_d, **kw)
        assert torch.isfinite(dout.float()).all(), name
        assert same_bits(sout.t, dout), name
        assert sout.intact() and sx.intact() and sxs.intact() and sres.intact(), name
        if ust_s is not None:
            assert torch.equal(ust_s, ust_d), name


@pytest.mark.parametrize("C", [128, 256, 384, 512])
def test_groupnorm_and_fir_on_slices_equal_dense(lib, C):
    """gn_stats, gn_apply (with and without SiLU), the FIR pass and the dual-output FIR pass on slices == on dense copies,
    bit for bit; nothing outside the written slices changes."""
    g = torch.Generator().manual_seed(C)
    B, H, W = 2, 16, 24
    x = bf16(g, B, H, W, C, scale=1.5, shift=0.3)
    gamma, beta = gn_params(g, C)
    sx = Slice(B, H, W, C, coff=128, after=128, data=x)
    ust = gn_stats(lib, sx.view(), B, C)
    assert torch.equal(ust, gn_stats(lib, dense(x), B, C))
    scsh = gn_finalize(lib, ust, None, B, H * W * C // 32, gamma, beta)
    for silu in (0, 1):
        so = Slice(B, H, W, C, coff=64, after=128)
        gn_apply(lib, sx.view(), scsh, silu, so.view())
        do = torch.empty_like(x)
        gn_apply(lib, dense(x), scsh, silu, dense(do))
        assert same_bits(so.t, do) and so.intact(), silu
    sh = so                                           # silu(GroupNorm(x)) as a channel slice
    for up in (1, 0):
        oh, ow = (2 * H, 2 * W) if up else (H // 2, W // 2)
        sn, sr = Slice(B, oh, ow, C, coff=64, after=0), Slice(B, oh, ow, C, coff=C, after=64)
        fir_dual(lib, sx.view(), sn.view(), sr.view(), up, scsh)
        dn, dr = (torch.empty(B, oh, ow, C, dtype=torch.bfloat16, device=DEV) for _ in range(2))
        fir_dual(lib, dense(x), dense(dn), dense(dr), up, scsh)
        assert torch.isfinite(dn.float()).all() and torch.isfinite(dr.float()).all()
        assert same_bits(sn.t, dn) and same_bits(sr.t, dr) and sn.intact() and sr.intact(), up
        for src, dual in ((sx, dr), (sh, dn)):
            so = Slice(B, oh, ow, C, coff=64, after=64)
            fir(lib, src.view(), so.view(), up)
            do = torch.empty(B, oh, ow, C, dtype=torch.bfloat16, device=DEV)
            fir(lib, dense(src.t.contiguous()), dense(do), up)
            assert same_bits(so.t, do) and so.intact(), (up, src is sx)
            assert same_bits(so.t, dual), (up, src is sx)   # dual pass == single passes
    assert sx.intact() and sh.intact()


@pytest.mark.parametrize("shape", [(2, 128, 16, 24), (1, 256, 8, 8), (3, 384, 6, 10)])
@pytest.mark.parametrize("up", [True, False])
def test_fir_dual_equals_groupnorm_and_two_fir_passes(lib, shape, up):
    """The dual-output FIR pass of the up / down residual blocks (rows staged in shared memory raw and normalised) ==
    GroupNorm pass + FIR pass for the normalised branch and FIR pass of x for the raw branch, bit for bit."""
    B, C, H, W = shape
    g = torch.Generator().manual_seed(C + H + int(up))
    x = bf16(g, B, H, W, C, scale=1.5, shift=0.3)
    gamma, beta = gn_params(g, C)
    scsh = gn_finalize(lib, gn_stats(lib, dense(x), B, C), None, B, H * W * C // 32, gamma, beta)
    oh, ow = (2 * H, 2 * W) if up else (H // 2, W // 2)
    out_n, out_r, want_n, want_r = (torch.empty(B, oh, ow, C, dtype=torch.bfloat16, device=DEV) for _ in range(4))
    fir_dual(lib, dense(x), dense(out_n), dense(out_r), up, scsh)
    h = torch.empty_like(x)
    gn_apply(lib, dense(x), scsh, 1, dense(h))
    fir(lib, dense(h), dense(want_n), up)
    fir(lib, dense(x), dense(want_r), up)
    assert torch.isfinite(want_n.float()).all() and torch.isfinite(want_r.float()).all()
    assert same_bits(out_n, want_n) and same_bits(out_r, want_r)


@pytest.mark.parametrize("H,W", [(4, 1), (16, 4), (16, 32)], ids=["n4-cudacore", "n64", "n512"])
def test_attention_on_fused_qkv_views(lib, H, W):
    """q, k, v as ld = 3C views of one fused qkv buffer (as the NIN_0..2 convolution writes it), output into a slice ==
    ops.attention_nhwc on dense copies, bit for bit.  n = 4 runs the fp32 CUDA-core kernels, n % 64 == 0 the tensor
    cores (row-pitched operand B of the implicit GEMM)."""
    from snr_aligned_diffse_b200 import ops
    g = torch.Generator().manual_seed(H * W)
    B, C = 2, 256
    n = H * W
    qkv = bf16(g, B, H, W, 3 * C)
    ws = torch.empty(int(lib.snrse_attention_workspace_bytes(B, n, C)), dtype=torch.uint8, device=DEV)
    q, k, v = (View(qkv.data_ptr() + 2 * j * C, B, H, W, C, 3 * C) for j in range(3))
    so = Slice(B, H, W, C, coff=128, after=64)
    _check(lib, lib.snrse_dbg_attention(_ref(q), _ref(k), _ref(v), _ptr(ws), _ref(so.view()), 1, _stream()), "attention")
    flat = qkv.reshape(B, n, 3 * C)
    want = ops.attention_nhwc(*(flat[..., j * C:(j + 1) * C].contiguous() for j in range(3)))
    assert torch.isfinite(want.float()).all()
    assert same_bits(so.t.reshape(B, n, C), want) and so.intact()


# ----------------------------------------------------------------------------------------------- B. concat GroupNorm
@pytest.mark.parametrize("ch,cs", [(128, 128), (256, 128), (256, 256)])
def test_concat_groupnorm_from_two_sources(lib, ch, cs):
    """GroupNorm over cat([h, skip]) finalised from the statistics of the two slices (at 256 + 128 channels group 21
    spans both sources): the same scale/shift bits as one source over a dense copy of the concatenation, and the
    normalised result matches fp64 group_norm(cat), also when h's statistics come from the 2-CTA convolution's
    epilogue."""
    g = torch.Generator().manual_seed(ch + 3 * cs)
    B, H, W = 2, 32, 64
    ci = ch + cs
    gamma, beta = gn_params(g, ci)
    cnt = H * W * ci // 32

    def halves(cat):
        return View(cat.data_ptr(), B, H, W, ch, ci), View(cat.data_ptr() + 2 * ch, B, H, W, cs, ci)

    # (1) values k/16, |k| <= 64: every partial sum is exact in fp32 whatever the thread layout of the statistics pass
    # (which depends on C), so the two-source result must equal the dense one bit for bit
    cat = (torch.randint(-64, 65, (B, H, W, ci), generator=g) / 16).to(torch.bfloat16).to(DEV)
    vh, vs = halves(cat)
    u0, u1, ud = gn_stats(lib, vh, B, ch), gn_stats(lib, vs, B, cs), gn_stats(lib, dense(cat), B, ci)
    assert torch.equal(torch.cat([u0, u1], 1), ud)
    assert same_bits(gn_finalize(lib, u0, u1, B, cnt, gamma, beta), gn_finalize(lib, ud, None, B, cnt, gamma, beta))

    # (2) general values, both sources from the statistics pass, and (3) h written by the 2-CTA convolution into its
    # slice of the concatenation buffer, its statistics gathered by the epilogue
    def check_normalised(cat, u0, u1, what):
        scsh = gn_finalize(lib, u0, u1, B, cnt, gamma, beta)
        out = torch.empty_like(cat)
        gn_apply(lib, dense(cat), scsh, 1, dense(out))
        ref = F.silu(F.group_norm(cat.to(F64).permute(0, 3, 1, 2), 32, gamma.to(F64), beta.to(F64), eps=1e-6))
        ref = ref.permute(0, 2, 3, 1)
        within((out.to(F64) - ref).abs(), 2 ** -7 * ref.abs() + 2e-3, what)

    cat = bf16(g, B, H, W, ci, scale=1.7, shift=0.4)
    vh, vs = halves(cat)
    check_normalised(cat, gn_stats(lib, vh, B, ch), gn_stats(lib, vs, B, cs), f"concat GN {ch}+{cs}")
    xin = bf16(g, B, H, W, 128)
    w = (torch.randn(ch, 9 * 128, generator=g) / math.sqrt(9 * 128)).to(torch.bfloat16).to(DEV)
    bias = (torch.randn(ch, generator=g) * 0.3).to(DEV)
    u0 = torch.zeros(B, ch // 4, 2, dtype=torch.int64, device=DEV)
    conv(lib, dense(xin), w, ch, bias=bias, out=vh, ustats=u0, path=0)
    check_normalised(cat, u0, gn_stats(lib, vs, B, cs), f"concat GN {ch}+{cs}, h from the conv epilogue")


# ----------------------------------------------------------------------------------------------- C. thin layers
def _bf16_rne_bits(a):
    """float32 ndarray -> bf16 bits, round to nearest even (finite inputs)."""
    b = a.view(np.uint32).astype(np.uint64)
    return ((b + 0x7FFF + ((b >> 16) & 1)) >> 16).astype(np.uint16)


def _complex_input(g, B, n):
    """complex64 [B, n] spanning six decades, with exact zeros and bf16 rounding ties."""
    v = torch.randn(B, n, 2, generator=g) * 10.0 ** (torch.rand(B, n, 2, generator=g) * 6 - 4)
    v.view(-1)[::97] = 0.0
    tie = v.view(-1)[5::89]
    tie.copy_((tie.view(torch.int32) & ~0xFFFF | 0x8000).view(torch.float32))     # exactly half way between bf16s
    return torch.view_as_complex(v).to(DEV)


def pack_input(lib, x, y, with64):
    B, n = x.shape
    x4 = torch.empty(B, n, 4, dtype=torch.float32, device=DEV)
    x64 = None
    if with64:
        x64 = torch.empty(B, n, 64, dtype=torch.bfloat16, device=DEV)
        x64.view(torch.int16).fill_(SENT)
    _check(lib, lib.snrse_dbg_pack_input(_ptr(x), _ptr(y), _ptr(x4), _ptr(x64), B, n, _stream()), "pack_input")
    return x4, x64


def test_pack_input64_hi_lo_split(lib):
    """x4 = (re x, im x, re y, im y) exactly; the 64-channel operand holds bf16(v) (round to nearest even) in channels
    0..3, bf16(v - hi) in 4..7 and exact zeros in 8..63."""
    g = torch.Generator().manual_seed(1)
    B, n = 2, 256 * 64 + 40
    x, y = _complex_input(g, B, n), _complex_input(g, B, n)
    x4, x64 = pack_input(lib, x, y, True)
    want = torch.stack([x.real, x.imag, y.real, y.imag], -1)
    assert same_bits(x4, want)
    assert same_bits(pack_input(lib, x, y, False)[0], want)
    v = want.cpu().numpy()
    hb = _bf16_rne_bits(v)
    lo = v - (hb.astype(np.uint32) << 16).view(np.float32)          # exact in fp32
    got = x64.view(torch.int16).cpu().numpy().view(np.uint16)
    assert np.array_equal(got[..., 0:4], hb)
    assert np.array_equal(got[..., 4:8], _bf16_rne_bits(lo))
    assert not got[..., 8:].any()


@pytest.mark.parametrize("B,H,W", [(2, 256, 64), (1, 256, 512), (2, 8, 40)])
def test_input_convolution(lib, B, H, W):
    """4 -> 128 input convolution: the 2-CTA kernel on the 64-channel hi/lo operand with PK_CONV3_K_BF16_HILO64 weights,
    and conv_in4 on the fp32 input, both writing a channel slice."""
    g = torch.Generator().manual_seed(H + W)
    Co = 128
    x, y = (torch.view_as_complex(torch.randn(B, H * W, 2, generator=g) * 0.7).to(DEV) for _ in range(2))
    x4, x64 = pack_input(lib, x, y, True)
    x4, x64 = x4.reshape(B, H, W, 4), x64.reshape(B, H, W, 64)
    w = torch.randn(Co, 4, 3, 3, generator=g) * 0.3
    bias = (torch.randn(Co, generator=g) * 0.1).to(DEV)
    wb = w.to(torch.bfloat16)
    taps = wb.permute(0, 2, 3, 1).reshape(Co, 9, 4)
    wt = torch.zeros(Co, 9, 64, dtype=torch.bfloat16)
    wt[:, :, 0:4], wt[:, :, 4:8] = taps, taps                        # [cout][(r*3+s)*64 + c] = w[cout][c % 4][r][s]
    wt = wt.reshape(Co, 9 * 64).to(DEV)
    s0 = Slice(B, H, W, Co, coff=128, after=0)
    conv(lib, dense(x64), wt, Co, bias=bias, out=s0.view(), path=0)
    d0 = torch.empty(B, H, W, Co, dtype=torch.bfloat16, device=DEV)
    conv(lib, dense(x64), wt, Co, bias=bias, out=dense(d0), path=0)
    assert same_bits(s0.t, d0) and s0.intact()
    hl = x64[..., 0:4].to(F64) + x64[..., 4:8].to(F64)
    got = s0.t.to(F64)
    ref = conv_ref(hl, wb, bias)
    A = conv_ref(hl.abs(), wb.abs()) + bias.to(F64).abs()
    within((got - ref).abs(), 2 ** -8 * ref.abs() + 2 ** -16 * A, f"input conv hi/lo {H}x{W} vs bf16 weights")
    ref32 = conv_ref(x4, w, bias)                                     # what the bf16 weights cost
    A32 = conv_ref(x4.abs(), w.abs()) + bias.to(F64).abs()
    within((got - ref32).abs(), 2 ** -8 * ref32.abs() + 2 ** -8 * A32, f"input conv hi/lo {H}x{W} vs fp32 weights")
    w32 = w.permute(0, 2, 3, 1).contiguous().to(DEV)                  # [cout][r][s][cin]
    s1 = Slice(B, H, W, Co, coff=64, after=64)
    _check(lib, lib.snrse_dbg_conv_in4(_ptr(x4), _ptr(w32), _ptr(bias), _ref(s1.view()), _stream()), "conv_in4")
    d1 = torch.empty(B, H, W, Co, dtype=torch.bfloat16, device=DEV)
    _check(lib, lib.snrse_dbg_conv_in4(_ptr(x4), _ptr(w32), _ptr(bias), _ref(dense(d1)), _stream()), "conv_in4")
    assert same_bits(s1.t, d1) and s1.intact()
    within((s1.t.to(F64) - ref32).abs(), 2 ** -8 * ref32.abs() + 2 ** -20 * A32, f"conv_in4 {H}x{W}")


@pytest.mark.parametrize("T", [64, 512])
def test_input_pyramid(lib, T):
    """fir_down2_f4 then combine4 into an output slice at every level 1..6 (down to 4 x 1 for T = 64)."""
    g = torch.Generator().manual_seed(T)
    B, Fq = 2, 256
    p = torch.randn(B, Fq, T, 4, generator=g).to(DEV)
    for lv in range(1, 7):
        H, W = Fq >> lv, T >> lv
        C = 128 if lv <= 2 else 256
        q = fir_f4(lib, p, up=False)
        assert q.shape == (B, H, W, 4)
        nchw = p.to(F64).permute(0, 3, 1, 2)
        ref = o_ncsnpp.fir_downsample_2d(nchw).permute(0, 2, 3, 1)
        A = o_ncsnpp.fir_downsample_2d(nchw.abs()).permute(0, 2, 3, 1)
        within((q.to(F64) - ref).abs(), 2 ** -20 * A, f"fir_down2_f4 level {lv} T={T}")
        h = bf16(g, B, H, W, C)
        w = (torch.randn(C, 4, generator=g) * 0.5).to(DEV)
        bias = (torch.randn(C, generator=g) * 0.1).to(DEV)
        sh, so = Slice(B, H, W, C, coff=C, after=0, data=h), Slice(B, H, W, C, coff=64, after=64)
        _check(lib, lib.snrse_dbg_combine4(_ptr(q), _ref(sh.view()), _ptr(w), _ptr(bias), _ref(so.view()), _stream()),
               "combine4")
        do = torch.empty_like(h)
        _check(lib, lib.snrse_dbg_combine4(_ptr(q), _ref(dense(h)), _ptr(w), _ptr(bias), _ref(dense(do)), _stream()),
               "combine4")
        assert same_bits(so.t, do) and so.intact() and sh.intact()
        q64, w64 = q.to(F64), w.to(F64)
        ref = h.to(F64) + q64 @ w64.T + bias.to(F64)
        A = h.to(F64).abs() + q64.abs() @ w64.abs().T + bias.to(F64).abs()
        within((so.t.to(F64) - ref).abs(), 2 ** -8 * ref.abs() + 2 ** -20 * A, f"combine4 level {lv} T={T}")
        p = q


HEAD_MAPS = [(8, 8), (8, 16), (16, 12), (24, 40), (256, 64), (32, 944), (4, 8), (8, 4), (4, 1)]


@pytest.mark.parametrize("H,W", HEAD_MAPS)
def test_output_head(lib, H, W):
    """C -> 4 output head, out4 = conv3x3(silu(GroupNorm(x))) + bias + fir_up2_f4(prev pyramid level), on the 2-CTA
    kernel (16-row weight tile, in-flight GroupNorm) where the map fits its tiles and on CUDA cores everywhere."""
    g = torch.Generator().manual_seed(H * 1000 + W)
    B = 2
    C = 128 if (H, W) == (256, 64) else 256
    x = bf16(g, B, H, W, C, scale=1.3, shift=0.2)
    gamma, beta = gn_params(g, C)
    sx = Slice(B, H, W, C, coff=128, after=64, data=x)
    scsh = gn_finalize(lib, gn_stats(lib, sx.view(), B, C), None, B, H * W * C // 32, gamma, beta)
    sa = Slice(B, H, W, C, coff=64, after=64)
    gn_apply(lib, sx.view(), scsh, 1, sa.view())
    a = sa.t.contiguous()
    addend = None
    if H % 2 == 0 and W % 2 == 0:
        addend = fir_f4(lib, torch.randn(B, H // 2, W // 2, 4, generator=g).to(DEV), up=True)
    w = torch.randn(4, C, 3, 3, generator=g) / math.sqrt(9 * C)
    bias = (torch.randn(4, generator=g) * 0.1).to(DEV)
    add64 = 0.0 if addend is None else addend.to(F64)
    add_abs = 0.0 if addend is None else addend.to(F64).abs()
    w32 = w.permute(0, 2, 3, 1).contiguous().to(DEV)                  # [4][3][3][C]
    o1 = conv_out4(lib, sa.view(), w32, bias, addend, None, 1, B, H, W)
    ref1 = conv_ref(a, w, bias) + add64
    A1 = conv_ref(a.abs(), w.abs()) + bias.to(F64).abs() + add_abs
    within((o1.to(F64) - ref1).abs(), 2 ** -20 * A1, f"conv_out4 (CUDA cores) {H}x{W}")
    assert sa.intact() and sx.intact()
    if H < 8 or W < 8:
        return
    wb = w.to(torch.bfloat16)
    w16 = torch.zeros(16, 9 * C, dtype=torch.bfloat16)
    w16[:4] = pack_w3(wb)
    w16_big = w16.clone()
    w16_big[4:] = (torch.randn(12, 9 * C, generator=g) * 1e3).to(torch.bfloat16)   # rows 4..15 must never reach out4
    w16, w16_big = w16.to(DEV), w16_big.to(DEV)
    fused = conv_out4(lib, sx.view(), w16_big, bias, addend, scsh, 0, B, H, W)
    plain = conv_out4(lib, sa.view(), w16_big, bias, addend, None, 0, B, H, W)
    zero_rows = conv_out4(lib, dense(a), w16, bias, addend, None, 0, B, H, W)
    assert same_bits(fused, plain) and same_bits(plain, zero_rows)
    ref0 = conv_ref(a, wb, bias) + add64
    A0 = conv_ref(a.abs(), wb.abs()) + bias.to(F64).abs() + add_abs
    within((fused.to(F64) - ref0).abs(), 2 ** -16 * A0, f"out4 (2-CTA) {H}x{W}")
    within((fused.to(F64) - o1.to(F64)).abs(), 2 ** -8 * A1, f"out4 2-CTA vs CUDA cores {H}x{W}")


def _fourier_ref(t32, fw32):
    """Candidate fp32 projections log(t) * W * 2 * pi (the reference's operation order), one per logf result within
    1 ulp of the correctly rounded log: the library's logf is accurate to 1 ulp, not correctly rounded."""
    l0 = np.float32(np.log(np.float64(t32)))
    cands = [l0, np.nextafter(l0, np.float32(-np.inf)), np.nextafter(l0, np.float32(np.inf))] if l0 != 0 else [l0]
    return [((np.float32(lg) * fw32) * np.float32(2)) * np.float32(math.pi) for lg in cands]


def test_time_embedding(lib):
    """Gaussian Fourier features of log t (within 2 ulp of fp64 sin / cos of the fp32 projection), the two SiLU
    layers and every block's Dense_0 row (fp64 from the same projection), rows not a multiple of 8."""
    g = torch.Generator().manual_seed(2)
    nf, rows = 128, 1004
    d = 4 * nf
    t = torch.tensor([1e-3, 0.03, 0.5, 1.0], dtype=torch.float32)
    B = t.numel()
    fw = torch.randn(nf, generator=g) * 16
    w1, b1 = torch.randn(d, 2 * nf, generator=g) / math.sqrt(2 * nf), torch.randn(d, generator=g) * 0.1
    w2, b2 = torch.randn(d, d, generator=g) / math.sqrt(d), torch.randn(d, generator=g) * 0.1
    dw, db = torch.randn(rows, d, generator=g) / math.sqrt(d), torch.randn(rows, generator=g) * 0.1
    scratch = torch.empty(B * 10 * nf, dtype=torch.float32, device=DEV)
    tb = torch.empty(B, rows, dtype=torch.float32, device=DEV)
    dv = [v.to(DEV) for v in (t, fw, w1, b1, w2, b2, dw, db)]
    _check(lib, lib.snrse_dbg_temb(_ptr(dv[0]), B, nf, *(_ptr(v) for v in dv[1:7]), _ptr(dv[7]), rows, _ptr(scratch),
                                   _ptr(tb), _stream()), "temb")
    emb = scratch[B * d:B * d + B * 2 * nf].reshape(B, 2 * nf).cpu().numpy().astype(np.float64)
    fw32 = fw.numpy()
    projs = []
    for b in range(B):
        ok = None
        for proj in _fourier_ref(t[b].numpy(), fw32):
            p64 = proj.astype(np.float64)
            want = np.concatenate([np.sin(p64), np.cos(p64)])
            ulp = np.spacing(np.abs(want).astype(np.float32)).astype(np.float64)
            if (np.abs(emb[b] - want) <= 2 * ulp).all():
                ok = p64
                break
        assert ok is not None, f"Fourier features of t={float(t[b])} are not sin/cos of log(t) * W * 2 pi"
        projs.append(ok)
    assert (emb[-1, :nf] == 0).all() and (emb[-1, nf:] == 1).all()   # t = 1: log t = 0
    p = torch.from_numpy(np.stack(projs))
    e = torch.cat([torch.sin(p), torch.cos(p)], 1)
    h1 = F.silu(e @ w1.to(F64).T + b1.to(F64))
    act = F.silu(h1 @ w2.to(F64).T + b2.to(F64))
    ref = act @ dw.to(F64).T + db.to(F64)
    A = act.abs() @ dw.to(F64).abs().T + db.to(F64).abs()
    within((tb.cpu().to(F64) - ref).abs(), 2 ** -18 * A, "temb Dense_0 rows")


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_final_head(lib, mode):
    """h / t, 1x1 conv 4 -> 2 and the preconditioning of mode 1 (sebridge) / the sign of mode 2; at t = 0.001
    (c_out = 0, c_skip = 1) mode 1 returns x exactly."""
    g = torch.Generator().manual_seed(mode)
    B, n = 4, 256 * 64 + 37
    t = torch.tensor([0.001, 0.03, 0.5, 1.0], dtype=torch.float32)
    p4 = torch.randn(B, n, 4, generator=g) * 3
    w, bias = torch.randn(8, generator=g) * 0.5, torch.randn(2, generator=g) * 0.1
    xr = torch.view_as_complex(torch.randn(B, n, 2, generator=g))
    out = torch.empty(B, n, dtype=torch.complex64, device=DEV)
    dv = [v.to(DEV) for v in (p4, t, w, bias, xr)]
    _check(lib, lib.snrse_dbg_final(*(_ptr(v) for v in dv), _ptr(out), B, n, mode, _stream()), "final")
    got = torch.view_as_real(out).cpu().to(F64)
    t64 = t.to(F64)[:, None]
    h = p4.to(F64) / t64[..., None]
    wm = w.to(F64).reshape(2, 4)
    net = h @ wm.T + bias.to(F64)
    A = h.abs() @ wm.abs().T + bias.to(F64).abs()
    if mode == 1:
        eps, sd = float(np.float32(0.001)), 0.5
        c_skip = sd ** 2 / ((t64 - eps) ** 2 + sd ** 2)
        c_out = sd * (t64 - eps) / torch.sqrt(sd ** 2 + t64 ** 2)
        x64 = torch.view_as_real(xr).to(F64)
        net = c_skip[..., None] * x64 + c_out[..., None] * net
        A = c_skip[..., None] * x64.abs() + c_out[..., None].abs() * A
        assert same_bits(out[0].view(torch.float32), xr[0].to(DEV).view(torch.float32))
    elif mode == 2:
        net = -net
    within((got - net).abs(), 2 ** -20 * A, f"final mode {mode}")


# ----------------------------------------------------------------------------------------------- D. decoder block
@pytest.mark.parametrize("B,H,W,path", [(2, 32, 64, 0), (2, 8, 4, 2)], ids=["halo2", "gemm"])
def test_decoder_block_composed_from_launchers(lib, B, H, W, path):
    """A decoder ResnetBlockBigGANpp over cat([h (256), skip (128)]) -> 128, recorded as the executor records it:
    two-source GroupNorm_0, Conv_0 (in flight on the 2-CTA kernel, after a GroupNorm pass on the GEMM path) + Dense_0
    bias from the time embedding, GroupNorm_1 from the epilogue sums (a statistics pass on the GEMM path), Conv_1 with
    the 1x1 Conv_2 shortcut over the concatenation, written into the first slice of the next concatenation buffer.
    Against oracle.ncsnpp.resblock in fp64 with the bf16-rounded convolution weights."""
    g = torch.Generator().manual_seed(H + path)
    ch, cs, co, nf = 256, 128, 128, 128
    ci, d = ch + cs, 4 * nf
    r = lambda *s, k=1.0: torch.randn(*s, generator=g) * k          # noqa: E731
    sd = {"all_modules.0.W": r(nf, k=16), "all_modules.1.weight": r(d, 2 * nf, k=(2 * nf) ** -0.5),
          "all_modules.1.bias": r(d, k=0.1), "all_modules.2.weight": r(d, d, k=d ** -0.5), "all_modules.2.bias": r(d, k=0.1),
          "p.GroupNorm_0.weight": torch.rand(ci, generator=g) + 0.5, "p.GroupNorm_0.bias": r(ci, k=0.2),
          "p.Conv_0.weight": r(co, ci, 3, 3, k=(9 * ci) ** -0.5).to(torch.bfloat16).float(), "p.Conv_0.bias": r(co, k=0.1),
          "p.Dense_0.weight": r(co, d, k=d ** -0.5), "p.Dense_0.bias": r(co, k=0.1),
          "p.GroupNorm_1.weight": torch.rand(co, generator=g) + 0.5, "p.GroupNorm_1.bias": r(co, k=0.2),
          "p.Conv_1.weight": r(co, co, 3, 3, k=(9 * co) ** -0.5).to(torch.bfloat16).float(), "p.Conv_1.bias": r(co, k=0.1),
          "p.Conv_2.weight": r(co, ci, 1, 1, k=ci ** -0.5).to(torch.bfloat16).float(), "p.Conv_2.bias": r(co, k=0.1)}
    t = torch.tensor([0.3, 0.05])
    td = t.to(DEV)
    gd = {k: v.to(DEV) for k, v in sd.items()}
    cat = bf16(g, B, H, W, ci, scale=1.2, shift=0.1)
    # time embedding: this block's Dense_0 rows only
    scratch = torch.empty(B * 10 * nf, dtype=torch.float32, device=DEV)
    tb = torch.empty(B, co, dtype=torch.float32, device=DEV)
    _check(lib, lib.snrse_dbg_temb(_ptr(td), B, nf, _ptr(gd["all_modules.0.W"]), _ptr(gd["all_modules.1.weight"]),
                                   _ptr(gd["all_modules.1.bias"]), _ptr(gd["all_modules.2.weight"]),
                                   _ptr(gd["all_modules.2.bias"]), _ptr(gd["p.Dense_0.weight"]), _ptr(gd["p.Dense_0.bias"]),
                                   co, _ptr(scratch), _ptr(tb), _stream()), "temb")
    # GroupNorm_0 over the concatenation, from the statistics of its two slices
    vh, vs = View(cat.data_ptr(), B, H, W, ch, ci), View(cat.data_ptr() + 2 * ch, B, H, W, cs, ci)
    scsh0 = gn_finalize(lib, gn_stats(lib, vh, B, ch), gn_stats(lib, vs, B, cs), B, H * W * ci // 32,
                        gd["p.GroupNorm_0.weight"], gd["p.GroupNorm_0.bias"])
    w0 = pack_w3(sd["p.Conv_0.weight"]).to(torch.bfloat16).to(DEV)
    h1 = torch.empty(B, H, W, co, dtype=torch.bfloat16, device=DEV)
    if path == 0:
        ust = torch.zeros(B, co // 4, 2, dtype=torch.int64, device=DEV)
        conv(lib, dense(cat), w0, co, bias=gd["p.Conv_0.bias"], tbias=tb, tb_stride=co, out=dense(h1), scsh=scsh0,
             ustats=ust, path=0)
    else:
        a0 = torch.empty_like(cat)
        gn_apply(lib, dense(cat), scsh0, 1, dense(a0))
        conv(lib, dense(a0), w0, co, bias=gd["p.Conv_0.bias"], tbias=tb, tb_stride=co, out=dense(h1), path=2)
        ust = gn_stats(lib, dense(h1), B, co)
    scsh1 = gn_finalize(lib, ust, None, B, H * W * co // 32, gd["p.GroupNorm_1.weight"], gd["p.GroupNorm_1.bias"])
    w1 = torch.cat([pack_w3(sd["p.Conv_1.weight"]), sd["p.Conv_2.weight"].reshape(co, ci)], 1).to(torch.bfloat16).to(DEV)
    b12 = gd["p.Conv_1.bias"] + gd["p.Conv_2.bias"]
    nxt = Slice(B, H, W, co, coff=0, after=128)     # the block's output is the first half of the next concatenation
    if path == 0:
        conv(lib, dense(h1), w1, co, x1=dense(cat), bias=b12, scale=1 / math.sqrt(2), out=nxt.view(), scsh=scsh1, path=0)
    else:
        a1 = torch.empty_like(h1)
        gn_apply(lib, dense(h1), scsh1, 1, dense(a1))
        conv(lib, dense(a1), w1, co, x1=dense(cat), bias=b12, scale=1 / math.sqrt(2), out=nxt.view(), path=2)
    assert nxt.intact()
    sd64 = {k: v.to(F64) for k, v in gd.items()}
    temb = o_ncsnpp.time_embedding(sd64, "", td.to(F64))
    ref = o_ncsnpp.resblock(sd64, "p.", {"up": 0, "down": 0}, cat.to(F64).permute(0, 3, 1, 2), temb).permute(0, 2, 3, 1)
    got = nxt.t.to(F64)
    # four bf16 roundings on the way (the normalised operands of both convolutions, h1, the output) each add ~1.6e-3
    # rms relative error; a wrong tile, group or slice moves the result by far more than the 4e-3 bound
    rel = float((got - ref).norm() / ref.norm())
    print(f"decoder block {B}x{H}x{W} path {path}: rel L2 {rel:.3g} (bound 4e-3)")
    assert rel <= 4e-3
    within((got - ref).abs(), 2 ** -6 * ref.abs() + 3e-2 * ref.abs().mean(), f"decoder block {B}x{H}x{W} path {path}")
