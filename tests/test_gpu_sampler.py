"""GPU tests of the sampler variants against fixtures produced by the UNMODIFIED reference (oracle/make_golden.py
sections 6c-6e; VERDICT r01 item 7): Langevin corrector in the PC loop (correctors.py:38-57), Euler-Maruyama predictor
step (predictors.py:41-52) and the BBED loop at T_sampling = 0.5 (sdes.py:240-307).  Every random tensor is supplied
explicitly in the order the reference calls `torch.randn_like`.

Tolerance: bf16 network vs the fp32 reference, 4 network evaluations chained -> rel-L2 <= 6e-2 on the final state
(as for the OUVE fixture in test_gpu_api.py); a single predictor step -> 2e-2 on the drift-dominated state.
"""
import os

import numpy as np
import pytest
import torch

from oracle.topology import NCSNppConfig, param_specs
from snr_aligned_diffse_b200.synth import synth_state_dict

pytestmark = pytest.mark.gpu


def _c(a):
    return torch.from_numpy(np.ascontiguousarray(a))


def rel_l2(a, b):
    a, b = torch.view_as_real(a).double().flatten(), torch.view_as_real(b).double().flatten()
    return float((a - b).norm() / b.norm())


@pytest.fixture(scope="module")
def sd():
    return synth_state_dict(param_specs(NCSNppConfig()), seed=0)


def _model(sd, sde, **kw):
    from snr_aligned_diffse_b200.sgmse.model import ScoreModel
    return ScoreModel.from_state_dict(sd, backbone="ncsnpp", sde=sde, model_type="bbed", snr_conditioned="false",
                                      base_dir="", **kw).eval(no_ema=True)


def _feed(monkeypatch, noises):
    feed = iter([n.cuda() for n in noises])
    monkeypatch.setattr(torch, "randn_like", lambda x, *a, **k: next(feed).to(x.dtype))


def test_langevin_corrector_loop_matches_reference_fixture(sd, golden_dir, monkeypatch):
    z = np.load(os.path.join(golden_dir, "pc_langevin.npz"))
    bb = _model(sd, "ouve", theta=1.5, sigma_min=0.05, sigma_max=0.5)
    _feed(monkeypatch, _c(z["noises"]))
    out, nfe = bb.get_pc_sampler("reverse_diffusion", "langevin", _c(z["Y"]).cuda(), N=2, corrector_steps=1, snr=0.5)()
    assert nfe == int(z["nfe"]) == 4
    assert rel_l2(out.cpu(), _c(z["out"])) <= 6e-2


def test_euler_maruyama_step_matches_reference_fixture(sd, golden_dir, monkeypatch):
    from snr_aligned_diffse_b200.sgmse.sampling.predictors import PredictorRegistry
    z = np.load(os.path.join(golden_dir, "em_step.npz"))
    bb = _model(sd, "ouve", theta=1.5, sigma_min=0.05, sigma_max=0.5)
    sde = bb.sde.copy()
    sde.N = 30
    em = PredictorRegistry.get_by_name("euler_maruyama")(sde, bb, probability_flow=False)
    _feed(monkeypatch, [_c(z["z"])])
    x_new, x_mean = em.update_fn(_c(z["x"]).cuda(), _c(z["t"]).cuda(), _c(z["Y"]).cuda())
    assert rel_l2(x_new.cpu(), _c(z["x_new"])) <= 2e-2 and rel_l2(x_mean.cpu(), _c(z["x_mean"])) <= 2e-2
    # through pc_sampler the reference raises TypeError (the predictor receives a 4th positional argument)
    assert str(z["in_loop"]) == "TypeError"
    monkeypatch.undo()                                        # the loop draws its own prior noise
    with pytest.raises(TypeError):
        bb.get_pc_sampler("euler_maruyama", "none", _c(z["Y"]).cuda(), N=2)()


@pytest.mark.parametrize("graph", [False, True], ids=["eager", "graph"])
def test_bbed_loop_matches_reference_fixture(sd, golden_dir, monkeypatch, graph):
    z = np.load(os.path.join(golden_dir, "pc_bbed.npz"))
    bbed = _model(sd, "bbed", T_sampling=0.5, k=2.6, theta=0.52, sigma_min=0.05, sigma_max=0.5)
    noises = _c(z["noises"])
    if graph:
        # captured loop: noise comes from torch's CUDA generator inside the graph, so feed the fixture's draws by
        # patching randn_like during capture with static buffers that are refilled before the replay
        bufs = [torch.empty_like(noises[0], device="cuda") for _ in range(len(noises) - 1)]
        feed = iter([noises[0].cuda()] + bufs[:2] + bufs)      # prior draw, eager warm-up of step 0, the captured steps
        order = []

        def fake(x, *a, **k):
            t = next(feed)
            order.append(t)
            return t
        monkeypatch.setattr(torch, "randn_like", fake)
        for b, n in zip(bufs, noises[1:]):
            b.copy_(n)
    else:
        _feed(monkeypatch, noises)
    sampler = bbed.get_pc_sampler("reverse_diffusion", "ald", _c(z["Y"]).cuda(), N=2, corrector_steps=1, snr=0.5,
                                  graph=graph)
    out, nfe = sampler()
    torch.cuda.synchronize()
    assert nfe == int(z["nfe"]) == 4 and out.dtype == torch.complex64
    assert rel_l2(out.cpu(), _c(z["out"])) <= 6e-2


def test_whole_loop_graph_is_default_when_shapes_repeat(sd):
    """get_pc_sampler() without a `graph` argument: the first call of a (shape, settings) combination runs the host
    loop, the second captures the WHOLE N-step loop as one CUDA graph and later calls replay it; with the generator
    re-seeded the three agree bit for bit."""
    m = _model(sd, "ouve", theta=1.5, sigma_min=0.05, sigma_max=0.5)
    g = torch.Generator().manual_seed(3)
    Y = torch.view_as_complex(torch.randn(2, 1, 256, 64, 2, generator=g) * 0.05).cuda()
    outs = []
    for call in range(3):
        torch.manual_seed(5)
        torch.cuda.manual_seed_all(5)
        out, nfe = m.get_pc_sampler("reverse_diffusion", "ald", Y, N=3, corrector_steps=1, snr=0.5)()
        assert nfe == 6
        outs.append(out.clone())
    loops = [v for k, v in m._pc_graph_cache.items() if k[0] != "seen"]
    assert len(loops) == 1 and len(loops[0].graphs) == 1            # one graph holds all three steps
    assert torch.equal(torch.view_as_real(outs[0]), torch.view_as_real(outs[1]))
    assert torch.equal(torch.view_as_real(outs[1]), torch.view_as_real(outs[2]))


def test_lincomb_rejects_mismatched_operands_and_accepts_strided_ones():
    """ops.lincomb / sdes.axpby (every sampler state update): a Y_prior whose shape differs from Y raises ValueError
    (the reference's elementwise arithmetic raises a broadcast error there) instead of reading past the end of a buffer;
    a non-contiguous operand (e.g. a transposed STFT view) gives the same values as its contiguous copy."""
    from snr_aligned_diffse_b200.sgmse.sdes import OUVESDE, axpby
    g = torch.Generator().manual_seed(9)
    Y = torch.view_as_complex(torch.randn(2, 1, 256, 64, 2, generator=g)).cuda()
    short = Y[..., :32].contiguous()
    with pytest.raises(ValueError):
        axpby(x=Y, a=1.0, y=short, b=1.0)
    with pytest.raises(ValueError):
        axpby(x=Y, a=1.0, y=Y.to(torch.complex128), b=1.0)
    with pytest.raises(ValueError):
        axpby(x=Y, a=torch.ones(3, device="cuda"), y=Y, b=1.0)
    strided = torch.view_as_complex(torch.randn(2, 1, 64, 256, 2, generator=g)).cuda().transpose(2, 3)
    assert not strided.is_contiguous()
    a = axpby(x=Y, a=0.5, y=strided, b=2.0)
    b = axpby(x=Y, a=0.5, y=strided.contiguous(), b=2.0)
    assert a.is_contiguous() and torch.equal(torch.view_as_real(a), torch.view_as_real(b))
    ref = 0.5 * Y + 2.0 * strided
    assert (a - ref).abs().max() <= 1e-6 * ref.abs().max()
    sde = OUVESDE(1.5, 0.05, 0.5, N=2)
    x0, _ = sde.prior_sampling(strided.shape, strided)          # state built from a strided Y is a plain contiguous tensor
    assert x0.is_contiguous() and x0.shape == strided.shape
