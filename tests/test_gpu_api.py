"""GPU tests of the reference-facing API (`sgmse` mirror) against the golden fixtures / the CPU oracle.

Tolerances: scalars (t, index) exact, norm factor 1e-6 relative; enhanced waveform in bf16 vs the fp32
reference: rel-L2 <= 2e-2 on the spectrogram, SI-SDR >= 30 dB and max-abs error <= 4 % of the waveform peak (measured
1.6e-2 / 33.7 dB / 2.6 %, profiles/r01_parity.md; SURVEY 7 measured 30.7 dB / 2-4 % for a bf16 run of the reference
itself on such random weights); 4-NFE PC sampler: rel-L2 <= 6e-2.
"""
import os

import numpy as np
import pytest
import torch

from oracle import frontend, sampler as o_sampler, snrnet as o_snrnet
from oracle.topology import NCSNppConfig, param_specs, snrnet_param_specs
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


@pytest.fixture(scope="module")
def v3(sd):
    from snr_aligned_diffse_b200.sgmse.model import ScoreModel
    m = ScoreModel.from_state_dict(sd, backbone="ncsnpp", sde="ouve", model_type="sebridge_v3", snr_conditioned="true",
                                   fixed_snr=0.17783, theta=1.5, sigma_min=0.05, sigma_max=1.0, base_dir="")
    return m.eval(no_ema=True)


@pytest.fixture(scope="module")
def snr_sd():
    return synth_state_dict(snrnet_param_specs(), seed=1)


@pytest.fixture(scope="module")
def estimator(snr_sd):
    from snr_aligned_diffse_b200.sgmse import model as sg_model
    from snr_aligned_diffse_b200.sgmse.snr_estimator import SNRModel
    est = SNRModel(base_dir="")
    est._error_loading_ema = True
    est.load_state_dict(snr_sd)
    est.eval(no_ema=True)
    sg_model.set_snr_model(est)
    return est


def test_enhance_v3_matches_reference_fixture(v3, golden_dir):
    z = np.load(os.path.join(golden_dir, "enhance_v3.npz"))
    y, Z = _c(z["y"]), _c(z["Z"])
    x_hat = v3.enhance(y, y, oracle=True, clean_rms=1.0, noise_rms=float(z["ratio"]), noise=Z)
    ref = z["x_hat"]
    assert isinstance(x_hat, np.ndarray) and x_hat.dtype == np.float32 and x_hat.shape == ref.shape   # eval.py:140
    assert o_sampler.si_sdr(ref.astype(np.float64), x_hat.astype(np.float64)) >= 30.0
    assert np.abs(x_hat - ref).max() <= 0.04 * np.abs(ref).max()
    out, aux = v3.enhance_batch(y, oracle=True, noise_over_clean=[float(z["ratio"])], noise=Z, return_aux=True)
    assert float(aux["t"][0]) == np.float32(z["t"])                                   # snapped timestep: exact
    assert abs(float(aux["norm_factor"][0]) / float(z["norm_factor"]) - 1) <= 1e-6
    assert rel_l2(aux["sample"].cpu(), _c(z["sample"])[:, 0]) <= 2e-2
    xh, nfe, rtf = v3.enhance(y, y, oracle=True, clean_rms=1.0, noise_rms=float(z["ratio"]), noise=Z, timeit=True)
    assert nfe == 1 and rtf > 0 and np.array_equal(xh, x_hat)


def test_enhance_batch_ragged_lengths(v3, sd):
    g = torch.Generator().manual_seed(21)
    lens = [8100, 7300]                                      # both pad to Tpad = 64
    y = torch.zeros(2, max(lens))
    for b, L in enumerate(lens):
        y[b, :L] = torch.randn(L, generator=g) * 0.05 + 0.1 * torch.sin(torch.arange(L) * (0.03 + 0.01 * b))
    Z = torch.view_as_complex(torch.randn(2, 1, 256, 64, 2, generator=g) * 0.5 ** 0.5)
    ratios = [0.2, 0.6]
    out = v3.enhance_batch(y, lengths=torch.tensor(lens), oracle=True, noise_over_clean=ratios, noise=Z).cpu()
    for b, L in enumerate(lens):
        ref = o_sampler.enhance_v3(sd, y[b:b + 1, :L], Z[b:b + 1], ratios[b], 0.17783, sigma_max=1.0)["x_hat"]
        assert o_sampler.si_sdr(ref.double().numpy(), out[b, :L].double().numpy()) >= 30.0
        assert torch.count_nonzero(out[b, L:]) == 0


def test_estimator_in_the_loop(v3, estimator, snr_sd):
    g = torch.Generator().manual_seed(33)
    y = torch.randn(2, 8000, generator=g) * torch.tensor([[0.02], [0.3]]) + 0.1 * torch.sin(torch.arange(8000) * 0.05)[None]
    out, aux = v3.enhance_batch(y, oracle=False, return_aux=True)
    for b in range(2):
        ref_ratio = float(o_snrnet.estimate_noise_over_clean(snr_sd, y[b:b + 1])[0, 0])
        assert abs(float(aux["ratio"][b]) / ref_ratio - 1) <= 1e-4
        idx, t, nf = o_sampler.v3_scalars(ref_ratio, 0.17783, float(y[b].abs().max()))
        assert int(aux["t_index"][b]) == idx and float(aux["t"][b]) == np.float32(t)
    assert torch.isfinite(out).all()


def test_pc_sampler_matches_reference_fixture(sd, golden_dir, monkeypatch):
    from snr_aligned_diffse_b200.sgmse.model import ScoreModel
    z = np.load(os.path.join(golden_dir, "pc_ouve.npz"))
    bb = ScoreModel.from_state_dict(sd, backbone="ncsnpp", sde="ouve", model_type="bbed", snr_conditioned="false",
                                    theta=1.5, sigma_min=0.05, sigma_max=0.5, base_dir="").eval(no_ema=True)
    feed = iter([n.cuda() for n in _c(z["noises"])])
    monkeypatch.setattr(torch, "randn_like", lambda x, *a, **k: next(feed).to(x.dtype))
    sampler = bb.get_pc_sampler("reverse_diffusion", "ald", _c(z["Y"]).cuda(), N=2, corrector_steps=1, snr=0.5)
    out, nfe = sampler()
    assert nfe == int(z["nfe"]) == 4
    assert rel_l2(out.cpu(), _c(z["out"])) <= 6e-2
    with pytest.raises(NotImplementedError):
        bb.get_pc_sampler("reverse_diffusion", "ald", _c(z["Y"]).cuda(), N=2, intermediate=True)


def test_forward_contract(v3):
    x = torch.view_as_complex(torch.randn(1, 1, 256, 64, 2))
    with pytest.raises(IndexError):                          # the reference's t.squeeze(3) on a [B] tensor (model.py:540)
        v3(x, torch.ones(1), x)
    out = v3(x, torch.full((1, 1, 1, 1), 0.3), x)           # host tensors in -> host tensor out
    assert out.shape == (1, 1, 256, 64) and out.dtype == torch.complex64 and not out.is_cuda


def test_data_module_transforms(v3):
    g = torch.Generator().manual_seed(4)
    w = torch.randn(2, 5000, generator=g) * 0.2
    S = v3._stft(w)
    ref = frontend.stft(w)
    assert S.shape == ref.shape and (S - ref).abs().max() <= 2e-5 * ref.abs().max()
    F_ = v3._forward_transform(ref)
    assert (F_ - frontend.spec_fwd(ref)).abs().max() <= 1e-6
    assert (v3._backward_transform(F_) - ref).abs().max() <= 1e-4 * ref.abs().max()
    back = v3.to_audio(F_, 5000)
    assert back.shape == w.shape and (back - w)[:, :5000 - 300].abs().max() <= 1e-4
    from snr_aligned_diffse_b200.sgmse.util.other import pad_spec, pad_spec_16
    assert pad_spec(F_[:, None]).shape[-1] == 64 and pad_spec_16(F_[:, None]).shape[-1] == 48


def test_cuda_graph_replay_is_bit_identical(v3):
    g = torch.Generator().manual_seed(8)
    y = (torch.randn(2, 8000, generator=g) * 0.1).cuda()
    Z = torch.view_as_complex(torch.randn(2, 1, 256, 64, 2, generator=g) * 0.5 ** 0.5).cuda()
    ratio = torch.tensor([0.3, 0.5]).cuda()
    eager = v3.enhance_batch(y, oracle=True, noise_over_clean=ratio, noise=Z).clone()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            out = v3.enhance_batch(y, oracle=True, noise_over_clean=ratio, noise=Z)
        graph.replay()
        s.synchronize()
        first = out.clone()
        y.mul_(0.5)                                          # new input in the static buffer -> new result
        graph.replay()
        s.synchronize()
    assert torch.equal(first, eager)
    assert not torch.equal(out, first) and torch.isfinite(out).all()


def test_sweep_matches_single_utterance_calls(v3, sd):
    """sweep.enhance_sweep (LPT shard + equal-Tpad batches + ragged lengths) returns, for every utterance, exactly
    what a call with that utterance alone returns: results do not depend on batching or on the rank count."""
    from snr_aligned_diffse_b200.sweep import enhance_sweep
    g = torch.Generator().manual_seed(11)
    lens = [5000, 9000, 8100, 16500, 8000, 5100, 23000]
    waves = [torch.randn(n, generator=g) * 0.05 + 0.1 * torch.sin(torch.arange(n) * 0.03) for n in lens]

    def fn(y, n):
        # explicit, per-utterance noise so that batches and single calls see the same draw
        tpad = (y.shape[1] + 1) // 128
        Z = torch.stack([torch.view_as_complex(torch.randn(1, 256, tpad, 2, generator=torch.Generator().manual_seed(int(k)))
                                               * 0.5 ** 0.5) for k in n.tolist()])
        return v3.enhance_batch(y, lengths=n, oracle=True, noise_over_clean=[0.3] * y.shape[0], noise=Z)

    merged = {}
    for world, tf in ((1, None), (2, None), (1, 300), (2, 160)):      # tf: frame-budget batching (larger batches of short utterances)
        for rank in range(world):
            r = enhance_sweep(fn, waves, rank=rank, world=world, max_batch=3 if tf is None else 1, device="cuda", keep_audio=True,
                              references=waves, target_frames=tf)
            for i, a in r["audio"].items():
                if i in merged:
                    assert torch.equal(merged[i], a), i          # same bits whatever the sharding
                merged[i] = a
            # the SI-SDR column (computed on the device) == util/other.py:71-75 on the returned audio
            for i, q in zip(r["ids"], r["si_sdr"]):
                ref = o_sampler.si_sdr(waves[i].double().numpy(), r["audio"][i].double().numpy())
                assert abs(q - ref) <= 1e-6 * max(1.0, abs(ref)), (i, q, ref)
    assert sorted(merged) == list(range(len(lens)))
    for i, w in enumerate(waves):
        tpad = 64 * (-(-(1 + lens[i] // 128) // 64))
        y = torch.zeros(1, 128 * tpad - 1)
        y[0, :lens[i]] = w
        alone = fn(y.cuda(), torch.tensor([lens[i]], dtype=torch.int32, device="cuda"))[0, :lens[i]].cpu()
        assert torch.equal(alone, merged[i]), i


def test_graphed_enhancer_pipeline_matches_eager(v3):
    """GraphedEnhancer (CUDA graph + copies overlapped on a second stream): every batch pushed through the host-buffer
    API comes back bit-identical to an eager enhance_batch call on the same input and noise draw."""
    from snr_aligned_diffse_b200.pipeline import GraphedEnhancer
    B, L = 2, 8100
    g = torch.Generator().manual_seed(21)
    Z = torch.view_as_complex(torch.randn(B, 1, 256, 64, 2, generator=g) * 0.5 ** 0.5).cuda()
    pipe = GraphedEnhancer(v3, B, L, "cuda", oracle=True, noise_over_clean=[0.4, 0.2], noise=Z).capture()
    ins = [(torch.randn(B, L, generator=g) * 0.05 + 0.1 * torch.sin(torch.arange(L) * (0.02 + 0.01 * k))).pin_memory()
           for k in range(4)]
    outs = [torch.empty(B, L).pin_memory() for _ in range(4)]
    for a, o in zip(ins, outs):
        pipe.enhance_host(a, o)
    pipe.flush()
    torch.cuda.synchronize()
    for a, o in zip(ins, outs):
        ref = v3.enhance_batch(a.cuda(), oracle=True, noise_over_clean=[0.4, 0.2], noise=Z).cpu()
        assert torch.equal(o, ref)


def test_graphed_enhancers_with_own_generators_are_reproducible_when_replays_overlap(v3, sd):
    """Two GraphedEnhancers drawing their noise from their own generators, replayed alternately on their two streams (as
    bench.py runs them): every replay draws fresh noise, and each enhancer returns exactly what an enhancer with an
    equally seeded generator returns when it is replayed alone."""
    from snr_aligned_diffse_b200.pipeline import GraphedEnhancer
    from snr_aligned_diffse_b200.sgmse.model import ScoreModel
    B, L, n = 2, 8100, 3
    y = (torch.randn(B, L, generator=torch.Generator().manual_seed(23)) * 0.05).cuda()
    # a second model: enhancers whose replays overlap need their own network workspace
    models = (v3, ScoreModel.from_state_dict(sd, backbone="ncsnpp", sde="ouve", model_type="sebridge_v3",
                                             snr_conditioned="true", fixed_snr=0.17783, theta=1.5, sigma_min=0.05,
                                             sigma_max=1.0, base_dir="").eval(no_ema=True))

    def make(k):
        p = GraphedEnhancer(models[k], B, L, "cuda", oracle=True, noise_over_clean=[0.4, 0.2],
                            generator=torch.Generator(device="cuda").manual_seed(k + 1))
        p.y_dev.copy_(y)
        torch.cuda.synchronize()
        return p.capture()

    def replays(pipes, count):
        outs = [[] for _ in pipes]
        for i in range(count * len(pipes)):
            p = pipes[i % len(pipes)]
            with torch.cuda.stream(p.stream):
                outs[i % len(pipes)].append(p.replay().clone())
        torch.cuda.synchronize()
        return outs

    overlapped = replays([make(0), make(1)], n)
    alone = [replays([make(k)], n)[0] for k in (0, 1)]
    for k in range(2):
        assert all(torch.equal(a, b) for a, b in zip(overlapped[k], alone[k])), k
        assert not torch.equal(overlapped[k][0], overlapped[k][1]) and torch.isfinite(overlapped[k][0]).all()
    assert not torch.equal(overlapped[0][0], overlapped[1][0])


def test_snr_sweep_batch_equals_per_snr_calls(v3):
    """deep_eval.py's nine-SNR loop as one batch == nine separate enhance() calls (same noise draws), bit for bit."""
    g = torch.Generator().manual_seed(31)
    L = 9000
    x = (0.1 * torch.sin(torch.arange(L) * 0.04) * (1 + 0.5 * torch.sin(torch.arange(L) * 0.001)))[None]
    n0 = torch.randn(1, L, generator=g) * 0.05
    snrs = list(range(0, 41, 5))
    Z = torch.view_as_complex(torch.randn(len(snrs), 1, 256, 128, 2, generator=g) * 0.5 ** 0.5)
    sweep = v3.enhance_snr_sweep(x, n0, snrs, oracle=True, noise_draws=Z)
    assert len(sweep) == 9 and all(o.shape == (L,) for o in sweep)
    for k, s in enumerate(snrs):
        y = x + n0 * 10 ** (-s / 20)
        one = v3.enhance(x, y, oracle=True, clean_rms=1, noise_rms=10 ** ((-s + 5) / 20), noise=Z[k:k + 1])
        assert np.array_equal(one, sweep[k]), s


def test_on_device_rk45_follows_scipy():
    """Device-resident Dormand-Prince integrator (sampling/ode.py) against scipy.integrate.solve_ivp(RK45), the
    solver the reference's ode_sampler calls: same accepted-step sequence (equal nfev) and the same end state within
    the float32 state rounding, on a stiff-ish complex linear ODE integrated backwards in time like the sampler."""
    from scipy import integrate
    from snr_aligned_diffse_b200.sgmse.sampling.ode import rk45_integrate
    g = torch.Generator().manual_seed(3)
    y0 = torch.view_as_complex(torch.randn(2, 1, 16, 8, 2, generator=g))
    lam = torch.view_as_complex(torch.stack([torch.rand(2, 1, 16, 8, generator=g) * 3 + 0.5,
                                             torch.randn(2, 1, 16, 8, generator=g) * 4], -1))
    lam_d, lam_n = lam.cuda(), lam.numpy().reshape(-1).astype(np.complex128)

    def f_dev(t, y):
        return lam_d * y * (0.5 + t) + (1.0 - t)

    def f_np(t, y):
        return lam_n * y * (0.5 + t) + (1.0 - t)

    for rtol, atol in ((1e-5, 1e-5), (1e-3, 1e-6)):
        res = rk45_integrate(f_dev, 1.0, y0.cuda(), 0.03, rtol=rtol, atol=atol)
        sol = integrate.solve_ivp(f_np, (1.0, 0.03), y0.numpy().reshape(-1).astype(np.complex128), rtol=rtol, atol=atol,
                                  method="RK45")
        ref = torch.from_numpy(sol.y[:, -1]).reshape(y0.shape)
        assert res.status == 0 and res.t == 0.03
        assert abs(res.nfev - sol.nfev) <= 6, (res.nfev, sol.nfev)       # at most one borderline accept/reject apart
        assert (res.y.cpu() - ref).abs().max() <= 20 * rtol * float(ref.abs().max())
    again = rk45_integrate(f_dev, 1.0, y0.cuda(), 0.03, rtol=1e-5, atol=1e-5)
    first = rk45_integrate(f_dev, 1.0, y0.cuda(), 0.03, rtol=1e-5, atol=1e-5)
    assert again.nfev == first.nfev and torch.equal(torch.view_as_real(again.y), torch.view_as_real(first.y))


def test_ode_sampler_on_device_matches_host_round_trip():
    """get_ode_sampler(on_device=True) == the reference-style scipy loop on the same prior draw (analytic score)."""
    from snr_aligned_diffse_b200.sgmse import sampling
    from snr_aligned_diffse_b200.sgmse.sdes import OUVESDE
    sde = OUVESDE(theta=1.5, sigma_min=0.05, sigma_max=0.5, N=30)
    g = torch.Generator().manual_seed(8)
    Y = torch.view_as_complex(torch.randn(2, 1, 256, 64, 2, generator=g) * 0.3).cuda()

    def score_fn(x, t, y):                        # score of N(y, std(t)^2): -(x - y) / std^2
        std = sde._std(t).reshape(-1, 1, 1, 1).to(x.device)
        return -(x - y) / std ** 2

    outs = []
    for on_dev in (False, True):
        torch.manual_seed(11)
        sample, nfe = sampling.get_ode_sampler(sde, score_fn, Y, rtol=1e-4, atol=1e-4, eps=0.03, on_device=on_dev)()
        assert sample.shape == Y.shape and sample.dtype == torch.complex64
        outs.append((sample, nfe))
    assert abs(outs[0][1] - outs[1][1]) <= 6
    assert rel_l2(outs[1][0].cpu(), outs[0][0].cpu()) <= 1e-3
    with pytest.raises(NotImplementedError):
        sampling.get_ode_sampler(sde, score_fn, Y, method="RK23", on_device=True)()


def test_si_sdr_on_device_matches_reference_formula():
    from snr_aligned_diffse_b200 import ops
    from snr_aligned_diffse_b200.sgmse.util.other import si_sdr as si_sdr_numpy
    g = torch.Generator().manual_seed(2)
    s = torch.randn(3, 40000, generator=g)
    e = s * torch.tensor([[0.7], [1.3], [1.0]]) + torch.randn(3, 40000, generator=g) * torch.tensor([[0.5], [1e-3], [0.05]])
    lens = torch.tensor([40000, 12345, 257], dtype=torch.int32)
    got = ops.si_sdr(s.cuda(), e.cuda(), lens.cuda()).cpu()
    for b in range(3):
        L = int(lens[b])
        ref = si_sdr_numpy(s[b, :L].double().numpy(), e[b, :L].double().numpy())
        assert abs(float(got[b]) - ref) <= 1e-9 * max(1.0, abs(ref))
    assert torch.equal(ops.si_sdr(s.cuda(), e.cuda(), lens.cuda()).cpu(), got)      # fixed reduction tree: reproducible


@pytest.mark.parametrize("sde_name", ["ouve", "bbed"])
def test_pc_sampler_graph_replay_equals_eager_loop(sd, sde_name):
    """get_pc_sampler(graph=True): the reverse loop replayed from one CUDA graph returns the same bits as the
    eager host loop when both see the same noise draws (the generator is re-seeded before each run; eager and captured
    `randn_like` calls consume the same Philox sequence), and a second run with a new seed differs (fresh noise per
    replay).  BBED exercises the host-tagged time vector (no device->host read of t inside the loop)."""
    from snr_aligned_diffse_b200.sgmse.model import ScoreModel
    kw = dict(theta=1.5, sigma_min=0.05, sigma_max=0.5) if sde_name == "ouve" else dict(theta=0.08, k=2.6, T_sampling=0.5)
    m = ScoreModel.from_state_dict(sd, backbone="ncsnpp", sde=sde_name, model_type="bbed", snr_conditioned="false",
                                   base_dir="", **kw).eval(no_ema=True)
    g = torch.Generator().manual_seed(31)
    Y = torch.view_as_complex(torch.randn(2, 1, 256, 64, 2, generator=g) * 0.05).cuda()
    outs = {}
    for mode in ("eager", "graph", "graph_again"):
        torch.manual_seed(77)
        torch.cuda.manual_seed_all(77)
        s = m.get_pc_sampler("reverse_diffusion", "ald", Y, N=2, corrector_steps=1, snr=0.5, graph=(mode != "eager"))
        out, nfe = s()
        assert nfe == 4 and torch.isfinite(torch.view_as_real(out)).all(), mode
        outs[mode] = out.clone()
    assert len(m._pc_graph_cache) == 1                      # the second sampler object reused the captured loop
    assert torch.equal(torch.view_as_real(outs["graph"]), torch.view_as_real(outs["graph_again"]))
    assert rel_l2(outs["graph"].cpu(), outs["eager"].cpu()) <= 1e-6
    torch.cuda.manual_seed_all(78)
    other, _ = m.get_pc_sampler("reverse_diffusion", "ald", Y, N=2, corrector_steps=1, snr=0.5, graph=True)()
    assert rel_l2(other.cpu(), outs["graph"].cpu()) > 1e-3


def test_enhance_files_matches_per_file_enhance(v3, tmp_path):
    """wavio.enhance_files (the eval.py file loop: wav in -> batched sweep -> wav out + SI-SDR column) writes, for every
    file, the PCM16 rounding of what a per-file `enhance_batch` call returns on the same input."""
    from snr_aligned_diffse_b200 import wavio
    g = torch.Generator().manual_seed(5)
    files, waves = [], []
    for i, n in enumerate((6000, 9100, 6100)):
        w = (torch.randn(n, generator=g) * 0.05 + 0.1 * torch.sin(torch.arange(n) * 0.04)).clamp(-0.9, 0.9)
        f = str(tmp_path / "noisy" / f"u{i}.wav")
        wavio.write_wav(f, w)
        wavio.write_wav(str(tmp_path / "clean" / f"u{i}.wav"), w * 0.9)
        files.append(f)
        waves.append(wavio.read_wav(f)[0])

    def fn(y, n):
        return v3.enhance_batch(y, lengths=n, oracle=True, noise_over_clean=[0.3] * y.shape[0],
                                noise=torch.zeros(y.shape[0], 1, 256, (y.shape[1] + 1) // 128, dtype=torch.complex64))

    res = wavio.enhance_files(fn, files, str(tmp_path / "out"), clean_dir=str(tmp_path / "clean"), max_batch=2, device="cuda")
    assert sorted(res["files"]) == ["u0.wav", "u1.wav", "u2.wav"] and all(q == q for q in res["si_sdr"])
    for i, f in enumerate(files):
        L = waves[i].numel()
        tpad = 64 * (-(-(1 + L // 128) // 64))
        y = torch.zeros(1, 128 * tpad - 1)
        y[0, :L] = waves[i]
        alone = fn(y.cuda(), torch.tensor([L], dtype=torch.int32, device="cuda"))[0, :L].cpu()
        got, _ = wavio.read_wav(str(tmp_path / "out" / os.path.basename(f)))
        want = torch.from_numpy(np.clip(np.rint(alone.double().numpy() * 32767.0), -32768, 32767).astype(np.float32) / 32768.0)
        assert got.shape == want.shape and torch.equal(got, want)


def test_flat_weight_file_loads_into_a_fresh_engine(sd, tmp_path):
    """A file written by export_flat and uploaded with load_flat drives the network to the same bits as load_state_dict."""
    from snr_aligned_diffse_b200.engine import NCSNppEngine
    a = NCSNppEngine().load_state_dict(sd, "cuda")
    path = str(tmp_path / "w.snrse")
    a.export_flat(sd, path)
    b = NCSNppEngine().load_flat(path)
    g = torch.Generator().manual_seed(2)
    x = torch.view_as_complex(torch.randn(1, 2, 256, 64, 2, generator=g) * 0.3).cuda()
    t = torch.tensor([0.3], device="cuda")
    assert torch.equal(torch.view_as_real(a.forward(x[:, 0], x[:, 1], t, mode=1)),
                       torch.view_as_real(b.forward(x[:, 0], x[:, 1], t, mode=1)))


def test_log_transform_variant(sd):
    """transform_type='log' (data_module.py:249-251,262-264): stand-alone spec_fwd / spec_back and the fused STFT /
    iSTFT kernels against the oracle restatement; enhance_batch runs end to end with it."""
    from snr_aligned_diffse_b200 import ops
    from snr_aligned_diffse_b200.sgmse.data_module import SpecsDataModule
    dm = SpecsDataModule(transform_type="log", spec_factor=0.15)
    g = torch.Generator().manual_seed(8)
    w = torch.randn(2, 6000, generator=g) * 0.2
    ref = frontend.stft(w)
    fwd = dm.spec_fwd(ref)
    want = frontend.spec_fwd(ref, transform_type="log")
    assert (fwd - want).abs().max() <= 1e-6 * max(1.0, float(want.abs().max()))
    back = dm.spec_back(want)
    assert (back - ref).abs().max() <= 1e-4 * ref.abs().max()
    fused = ops.stft(w.cuda(), transform=2, beta=0.15, tpad=ref.shape[-1]).cpu()
    assert (fused - want).abs().max() <= 2e-5 * max(1.0, float(want.abs().max()))
    wave = ops.istft(want.cuda().contiguous(), 6000, transform=2, beta=0.15).cpu()
    assert (wave - frontend.istft(frontend.spec_back(want, transform_type="log"), 6000)).abs().max() <= 2e-5
    from snr_aligned_diffse_b200.sgmse.model import ScoreModel
    m = ScoreModel.from_state_dict(sd, backbone="ncsnpp", sde="ouve", model_type="sebridge_v3", snr_conditioned="true",
                                   fixed_snr=0.17783, theta=1.5, sigma_min=0.05, sigma_max=1.0, base_dir="",
                                   transform_type="log").eval(no_ema=True)
    out = m.enhance(w[:1], w[:1], oracle=True, clean_rms=1.0, noise_rms=0.3)
    assert out.shape == (6000,) and np.isfinite(out).all()
