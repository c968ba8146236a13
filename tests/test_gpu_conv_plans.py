"""Every convolution plan the NCSN++ executor can choose, run once on its cheapest instance against fp64 (-m gpu, B200).

tests/test_conv_plans_cpu.py enumerates the executor's convolutions over B = 1..64 x Tpad = 64..7552 and groups them into
classes (plan fields, persistent / uneven walk, odd tile count, ragged edges, operand combination).  Here the enumeration
is repeated with the device's SM count and the cheapest instance (fewest MACs) of every class runs through the
launcher the executor calls (snrse_dbg_conv path 0 / 2, snrse_dbg_conv_out4) on views with the dumped pitch and channel
offset, with the dumped operand combination: GroupNorm + SiLU in flight from a real scale/shift table, 1x1 shortcut,
residual, time-embedding bias with the executor's row stride, epilogue statistics.  For every instance:

  plan       the fields the launcher's own make_plan chooses for these views equal the dump's;
  fp64       the result against a float64 convolution of exactly the operands the kernel reads, within
               2^-8 |ref|                                  rounding of the bf16 store (absent for the fp32 out4 head)
             + (1 + 2^-6) * [ (K/16 + 8) 2^-22 A           fp32 accumulation: one tcgen05.mma per 16 K values adds
                                                            its exact products with an error below 2 ulp (2^-22) of
                                                            the largest partial sum, |partial| <= A; the + 8 covers the
                                                            epilogue's fp32 adds / multiplies
                              + 2^-8 A_a                    in-flight normalisation: bf16 rounding of silu(t)
                              + 2^-10.9 A_h ]               tanh.approx.f32 (max relative error 2^-10.987, PTX ISA)
                                                            in silu(t) = h + h tanh(h), h = t / 2, plus fp32 rounding
                                                            of h; the (1 + 2^-6) covers second-order products
             A = the same expression on absolute values, A_a = sum |w| |silu(t)|, A_h = sum |w| |t| / 2, both times
             scale; K = 9 C0 + C1 (3x3) or C0 + C1 (1x1);
  stats      the epilogue's GroupNorm sums against fp64 sums of the stored output, within the bounds of
             test_gpu_parity.test_conv_epilogue_groupnorm_partials (its sqrt(n) written as sqrt(sum y^2), equal at
             unit rms);
  batch      the last image of the instance run alone at B = 1 (usually another class: no persistent walk, SUB 1,
             N split) gives the same bits and the same statistics.  The network's batch invariance rests on this:
             the K order of every plan depends on the layer only (test_gpu_parity.test_shortcut_ring_batch_invariance).
  sentinel   no channel outside the written slice changes, no neighbour channel of an input slice reaches the output.
"""
import ctypes
import math
import time

import pytest
import torch
import torch.nn.functional as F

from test_conv_plans_cpu import PATH_NAMES, class_key, enumerate_classes
from test_gpu_network_layers import Slice, View, _check, _ptr, _ref, conv, conv_out4, gn_finalize, gn_stats
from snr_aligned_diffse_b200.engine import CONV_PLAN_FIELDS

pytestmark = pytest.mark.gpu

DEV = "cuda"
F64 = torch.float64
TB_ROW = 40                 # this layer's first row inside the executor's time-embedding bias block


@pytest.fixture(scope="module")
def lib():
    from snr_aligned_diffse_b200 import _lib
    lib = _lib.load()
    _lib.require_device()
    return lib


@pytest.fixture(scope="module")
def classes():
    from snr_aligned_diffse_b200.engine import NCSNppEngine
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return enumerate_classes(NCSNppEngine(), sms)


def _rand(g, *shape, scale=1.0, shift=0.0):
    return torch.randn(*shape, generator=g, device=DEV) * scale + shift


def _plan(lib, r, x0, x1, wt, res, out, scsh):
    p = (ctypes.c_int * len(CONV_PLAN_FIELDS))()
    _check(lib, lib.snrse_dbg_conv_plan(_ref(x0), int(r["taps"]), _ref(x1), _ptr(wt), 4 if r["out4"] else int(r["n"]),
                                        _ref(res), _ref(out), _ptr(scsh), int(r["path"]), ctypes.byref(p)), "dbg_conv_plan")
    return dict(zip(CONV_PLAN_FIELDS, list(p)))


class Instance:
    """The operands of one dumped convolution, dense; run() places them in views with the dumped pitch and offset."""

    def __init__(self, lib, r, seed):
        self.lib, self.r = lib, r
        g = torch.Generator(device=DEV).manual_seed(seed)
        B, H, W = int(r["B"]), int(r["H"]), int(r["W"])
        c0, c1, n, taps = int(r["c0"]), int(r["c1"]), int(r["n"]), int(r["taps"])
        self.B, self.H, self.W, self.c0, self.c1, self.n, self.taps = B, H, W, c0, c1, n, taps
        self.x = _rand(g, B, H, W, c0, scale=1.3, shift=0.2).to(torch.bfloat16)
        self.x1 = _rand(g, B, H, W, c1).to(torch.bfloat16) if c1 else None
        self.res = _rand(g, B, H, W, n).to(torch.bfloat16) if r["res"] else None
        k = taps * c0 + c1
        self.w0 = (_rand(g, n, c0, 3 if taps == 9 else 1, 3 if taps == 9 else 1) / math.sqrt(k)).to(torch.bfloat16)
        self.w1 = (_rand(g, n, c1, 1, 1) / math.sqrt(k)).to(torch.bfloat16) if c1 else None
        packed = self.w0.permute(0, 2, 3, 1).reshape(n, taps * c0)
        if r["out4"]:
            # rows 4..15 of the 16-row weight tile are large: they must never reach the result
            self.wt = torch.cat([packed, (_rand(g, 12, 9 * c0) * 1e3).to(torch.bfloat16)]).contiguous()
        else:
            self.wt = torch.cat([packed] + ([self.w1.reshape(n, c1)] if c1 else []), 1).contiguous()
        self.bias = _rand(g, n, scale=0.5) if r["bias"] else None
        self.tball = _rand(g, B, int(r["tb_stride"]), scale=0.3) if r["tbias"] else None
        self.addend = _rand(g, B, H, W, 4) if r["addend"] else None
        self.scale = float(r["scale"])
        self.scsh = None
        if r["norm"]:
            gamma, beta = torch.rand(c0, generator=g, device=DEV) + 0.5, _rand(g, c0, scale=0.2)
            sx = Slice(B, H, W, c0, coff=int(r["off0"]), after=int(r["ld0"]) - int(r["off0"]) - c0, data=self.x)
            self.scsh = gn_finalize(self.lib, gn_stats(self.lib, sx.view(), B, c0), None, B, H * W * c0 // 32, gamma, beta)

    def run(self, b0=0):
        """Launch on images b0..B-1 in views shaped like the dump's; returns (output, statistics, plan fields)."""
        r, lib, s = self.r, self.lib, slice(b0, None)
        B, H, W, n = self.B - b0, self.H, self.W, self.n

        def sl(t, C, off, ld):
            return Slice(B, H, W, C, coff=off, after=ld - off - C, data=t[s])

        sx = sl(self.x, self.c0, int(r["off0"]), int(r["ld0"]))
        sx1 = sl(self.x1, self.c1, int(r["off1"]), int(r["ld1"])) if self.x1 is not None else None
        sres = sl(self.res, n, int(r["off_res"]), int(r["ld_res"])) if self.res is not None else None
        scsh = self.scsh[s].contiguous() if self.scsh is not None else None
        tb = self.tball[s][:, TB_ROW:] if self.tball is not None else None
        ins = [v for v in (sx, sx1, sres) if v is not None]
        if r["out4"]:
            out4 = torch.empty(B, H, W, 4, dtype=torch.float32, device=DEV)
            plan = _plan(lib, r, sx.view(), None, self.wt, None, View(out4.data_ptr(), B, H, W, 4, 4), scsh)
            addend = self.addend[s].contiguous() if self.addend is not None else None
            out = conv_out4(lib, sx.view(), self.wt, self.bias, addend, scsh, 0, B, H, W)
            assert all(v.intact() for v in ins)
            return out, None, plan
        sout = Slice(B, H, W, n, coff=int(r["off_out"]), after=int(r["ld_out"]) - int(r["off_out"]) - n)
        ust = torch.zeros(B, n // 4, 2, dtype=torch.int64, device=DEV) if r["stats"] else None
        view = lambda v: None if v is None else v.view()    # noqa: E731
        plan = _plan(lib, r, sx.view(), view(sx1), self.wt, view(sres), sout.view(), scsh)
        conv(lib, sx.view(), self.wt, n, taps=self.taps, x1=view(sx1), bias=self.bias, tbias=tb,
             tb_stride=int(r["tb_stride"]), res=view(sres), scale=self.scale, out=sout.view(), scsh=scsh, ustats=ust,
             path=int(r["path"]))
        assert sout.intact() and all(v.intact() for v in ins)
        return sout.t.contiguous(), ust, plan

    def reference(self):
        """(ref, A, A_a, A_h) in float64, NHWC, from exactly the operands the kernel reads."""
        nchw = lambda t: t.to(F64).permute(0, 3, 1, 2)      # noqa: E731
        pad = 1 if self.taps == 9 else 0
        nrow = 4 if self.r["out4"] else self.n
        w0 = self.w0[:nrow].to(F64)
        a = nchw(self.x)
        a_h = None
        if self.scsh is not None:
            sc, sh = (self.scsh[:, i, :, None, None].to(F64) for i in (0, 1))
            t = a * sc + sh
            a = t * torch.sigmoid(t)
            a_h = F.conv2d(t.abs() * 0.5, w0.abs(), padding=pad)
            del t
        ref = F.conv2d(a, w0, padding=pad)
        A_a = F.conv2d(a.abs(), w0.abs(), padding=pad)
        del a
        A = A_a.clone()
        if self.x1 is not None:
            x1, w1 = nchw(self.x1), self.w1.to(F64)
            ref += F.conv2d(x1, w1)
            A += F.conv2d(x1.abs(), w1.abs())
            del x1
        add = []
        if self.bias is not None:
            add.append(self.bias.to(F64)[None, :, None, None])
        if self.tball is not None:
            add.append(self.tball[:, TB_ROW:TB_ROW + nrow].to(F64)[:, :, None, None])
        if self.res is not None:
            add.append(nchw(self.res))
        if self.addend is not None:
            add.append(nchw(self.addend))
        for v in add:
            ref += v
            A += v.abs()
        out = [v * self.scale if v is not None else None for v in (ref, A, A_a, a_h)]
        return [v.permute(0, 2, 3, 1) if v is not None else None for v in out]


def check_fp64(inst, out):
    ref, A, A_a, A_h = inst.reference()
    steps = (inst.taps * inst.c0 + inst.c1) / 16
    e = (steps + 8) * 2.0 ** -22 * A
    if A_h is not None:
        e += 2.0 ** -8 * A_a + 2.0 ** -10.9 * A_h
    bound = (1 + 2.0 ** -6) * e
    if not inst.r["out4"]:
        bound += 2.0 ** -8 * ref.abs()
    err = (out.to(F64) - ref).abs()
    assert bool((bound > 0).all())
    return float((err / bound).max())


def check_stats(inst, out, ust):
    o = out.to(F64).reshape(inst.B, inst.H * inst.W, inst.n // 4, 4)
    want_s, want_q = o.sum((1, 3)), (o * o).sum((1, 3))
    st = ust.to(F64) * torch.tensor([2.0 ** -30, 2.0 ** -20], dtype=F64, device=DEV)
    ok_s = (st[..., 0] - want_s).abs() <= 2 ** -8 * want_q.sqrt() * 2.0 + 2 ** -9 * want_s.abs()
    ok_q = (st[..., 1] - want_q).abs() <= 2 ** -7 * want_q
    return bool(ok_s.all()) and bool(ok_q.all())


def bitwise(a, b):
    return torch.equal(a.contiguous().view(torch.int16 if a.element_size() == 2 else torch.int32),
                       b.contiguous().view(torch.int16 if b.element_size() == 2 else torch.int32))


@pytest.mark.parametrize("path", ["2-CTA", "2-CTA out4", "GEMM"], ids=["halo2", "halo2-out4", "gemm"])
def test_every_plan_class_against_fp64(lib, classes, path):
    """The cheapest instance of every class of this path: plan agreement, fp64 bound, epilogue statistics, batch
    invariance and slice sentinels.  Prints the class count, the worst err/bound and the wall time."""
    t0 = time.time()
    todo = sorted((v[0], k, v) for k, v in classes.items() if PATH_NAMES[k[0], k[1]] == path)
    failures, worst = [], (0.0, None)
    for i, (m, k, (_, B, T, r)) in enumerate(todo):
        what = f"{path} B={B} T={T} {int(r['H'])}x{int(r['W'])} {k}"
        try:
            assert class_key(r) == k
            inst = Instance(lib, r, seed=i)
            out, ust, plan = inst.run()
            want = {f: int(r[f]) for f in CONV_PLAN_FIELDS}
            assert plan == want, f"plan {plan} != dump {want}"
            assert torch.isfinite(out.float()).all(), "non-finite output"
            ratio = check_fp64(inst, out)
            if ratio > worst[0]:
                worst = (ratio, what)
            assert ratio <= 1.0, f"max err/bound = {ratio:.3g}"
            if ust is not None:
                assert check_stats(inst, out, ust), "epilogue statistics"
            if B > 1:
                alone, ust1, _ = inst.run(b0=B - 1)
                assert bitwise(alone[0], out[-1]), "the last image alone differs from the batch"
                if ust is not None:
                    assert torch.equal(ust1[0], ust[-1]), "the last image's statistics alone differ from the batch"
            del inst, out, ust
        except AssertionError as ex:
            failures.append(f"{what}: {ex}")
    torch.cuda.synchronize()
    print(f"{path}: {len(todo)} classes, worst err/bound {worst[0]:.3g} ({worst[1]}), {time.time() - t0:.1f} s")
    for f in failures:
        print("FAIL", f)
    assert not failures, f"{len(failures)} of {len(todo)} classes failed; first: {failures[0]}"
