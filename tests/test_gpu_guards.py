"""Out-of-bounds WRITE detection with guard bands (compute-sanitizer is closed on this GPU pool: "find a bad access
with bounds checks and asserts of your own, small cases, and a comparison with the CPU reference").

Every device buffer the host layer hands to the C ABI is allocated with `torch.empty` / `torch.empty_like`
(`ops.py`, `engine.py`, `pipeline.py`).  These tests replace both with an allocator that surrounds each buffer with
64 KB of 0xA5 bytes on either side, run the kernels on ragged / odd shapes (tile edges, partial frames, lengths that
are not multiples of anything), and then check every guard byte.  A kernel that stores even one byte before or after
a buffer it was given (an output, the network's activation arena, the attention / iSTFT / GroupNorm workspaces)
fails here.  Results are compared with the oracle in the other test files; this file only checks the guards.
"""
import numpy as np
import pytest
import torch

from oracle.topology import NCSNppConfig, param_specs, snrnet_param_specs
from snr_aligned_diffse_b200.synth import synth_state_dict, synth_waves

pytestmark = pytest.mark.gpu
PAD = 65536


class GuardedAllocator:
    def __init__(self):
        self._empty, self._empty_like = torch.empty, torch.empty_like
        self.live = []

    def empty(self, *size, dtype=None, device=None, **kw):
        if len(size) == 1 and isinstance(size[0], (tuple, list, torch.Size)):
            size = tuple(size[0])
        dev = torch.device(device) if device is not None else None
        if dev is None or dev.type != "cuda" or kw.get("pin_memory"):
            if dtype is not None:
                kw["dtype"] = dtype
            if device is not None:
                kw["device"] = device
            return self._empty(*size, **kw)
        dtype = dtype or torch.get_default_dtype()
        item = self._empty((), dtype=dtype).element_size()
        n = int(np.prod(size)) * item if len(size) else item
        raw = self._empty(n + 2 * PAD, dtype=torch.uint8, device=dev)
        raw.fill_(0xA5)
        self.live.append((raw, n))
        return raw[PAD:PAD + n].view(dtype).view(*size)

    def empty_like(self, x, **kw):
        if not x.is_cuda:
            return self._empty_like(x, **kw)
        return self.empty(*x.shape, dtype=kw.get("dtype", x.dtype), device=x.device)

    def check(self):
        torch.cuda.synchronize()
        assert self.live, "no guarded allocation happened"
        for raw, n in self.live:
            lo, hi = raw[:PAD], raw[PAD + n:]
            assert bool((lo == 0xA5).all()) and bool((hi == 0xA5).all()), f"guard band of a {n}-byte buffer was overwritten"
        return len(self.live)


@pytest.fixture
def guard(monkeypatch):
    g = GuardedAllocator()
    monkeypatch.setattr(torch, "empty", g.empty)
    monkeypatch.setattr(torch, "empty_like", g.empty_like)
    return g


@pytest.fixture(scope="module")
def v3():
    from snr_aligned_diffse_b200.sgmse import model as sg_model
    from snr_aligned_diffse_b200.sgmse.model import ScoreModel
    from snr_aligned_diffse_b200.sgmse.snr_estimator import SNRModel
    est = SNRModel(base_dir="")
    est._error_loading_ema = True
    est.load_state_dict(synth_state_dict(snrnet_param_specs(), seed=1))
    est.eval(no_ema=True)
    sg_model.set_snr_model(est)
    m = ScoreModel.from_state_dict(synth_state_dict(param_specs(NCSNppConfig()), seed=0), backbone="ncsnpp", sde="ouve",
                                   model_type="sebridge_v3", snr_conditioned="true", fixed_snr=0.17783, theta=1.5,
                                   sigma_min=0.05, sigma_max=1.0, base_dir="")
    return m.eval(no_ema=True)


@pytest.mark.parametrize("L,lengths", [(9000, [9000, 5001, 131]), (24577, [24577]), (8191, [8191, 8190])])
def test_enhance_batch_ragged_stays_inside_its_buffers(v3, guard, L, lengths):
    """Full sebridge_v3 pass (absmax, both STFTs, SNRNet, scalars, noise injection, NCSN++ with its activation arena,
    iSTFT) on ragged batches: Tpad 128 / 256 / 64 buckets, last frames partial, one utterance shorter than a frame pad."""
    v3.dnn.engine._ws.clear()                      # the arena for this shape is allocated under the guard
    y = synth_waves(len(lengths), L, seed=3)
    out = v3.enhance_batch(y, lengths=torch.tensor(lengths, dtype=torch.int32), oracle=False)
    assert guard.check() >= 8
    assert torch.isfinite(out).all()
    v3.dnn.engine._ws.clear()


def test_operators_on_odd_shapes_stay_inside_their_buffers(guard):
    from snr_aligned_diffse_b200 import ops
    g = torch.Generator().manual_seed(0)
    dev = "cuda"
    x = (torch.randn(2, 24, 40, 128, generator=g) * 0.5).to(torch.bfloat16).to(dev)          # ragged 16x8 tile edges
    wt = (torch.randn(256, 9 * 128, generator=g) * 0.03).to(torch.bfloat16).to(dev)
    for impl in (0, 2, 1):
        ops.conv_nhwc(x, wt, 9, bias=torch.zeros(256, device=dev), impl=impl)
    gam, bet = torch.ones(128, device=dev), torch.zeros(128, device=dev)
    ops.groupnorm_nhwc(x, gam, bet)
    ops.gn_silu_conv3x3_nhwc(x, gam, bet, wt[:128].contiguous())
    ops.fir_nhwc(x, True)
    ops.fir_nhwc(x, False)
    for n in (200, 128, 12):                                                                 # CUDA-core and tensor-core paths
        q = torch.randn(2, n, 256, generator=g).to(torch.bfloat16).to(dev)
        ops.attention_nhwc(q, q, q)
    w = torch.randn(3, 5003, generator=g).to(dev)
    S = ops.stft(w, lengths=torch.tensor([5003, 4000, 77], dtype=torch.int32, device=dev))
    ops.istft(S, 5003, lengths=torch.tensor([5003, 4000, 77], dtype=torch.int32, device=dev))
    ops.stft(w, planar=True, transform=False, pad_multiple=16)
    ops.absmax(w)
    ops.si_sdr(w, w * 0.9 + 0.01)
    assert guard.check() >= 13


def test_pc_loop_stays_inside_its_buffers(guard):
    from snr_aligned_diffse_b200.sgmse.model import ScoreModel
    m = ScoreModel.from_state_dict(synth_state_dict(param_specs(NCSNppConfig()), seed=0), backbone="ncsnpp", sde="ouve",
                                   model_type="bbed", snr_conditioned="false", theta=1.5, sigma_min=0.05, sigma_max=0.5,
                                   base_dir="").eval(no_ema=True)
    g = torch.Generator().manual_seed(1)
    Y = torch.view_as_complex(torch.randn(1, 1, 256, 64, 2, generator=g) * 0.05).cuda()
    out, nfe = m.get_pc_sampler("reverse_diffusion", "ald", Y, N=2, corrector_steps=1, snr=0.5, graph=False)()
    assert nfe == 4 and guard.check() >= 6
