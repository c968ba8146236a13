"""Keyed mode on the B200: the keyed noise of include/snrse_b200.h (`snrse_lincomb_keyed`), and every throughput path
enhancing each utterance as if alone, with the SNR estimator in the loop.

Bounds.  z_out against the float64 evaluation of the contract: logf and sincospif are within 1 ulp (CUDA math API),
sqrtf is correctly rounded, so with eps = 2^-24 the relative error of -logf(u1) is <= 2 eps, of r = sqrtf(.) <= 2 eps,
of cospi / sinpi <= 2 eps and the product adds eps: <= 5 eps per component, plus the float64 reference's own error
(cos(2 pi u2) with a rounded argument: <= r * 2 pi * 2^-53 absolute).  Statistics: 5 standard errors.  Against the
oracle: the existing end-to-end bounds (SI-SDR >= 30 dB, max-abs <= 4 % of peak, tests/test_gpu_api.py).
"""
import numpy as np
import pytest
import torch

from oracle import sampler as o_sampler, snrnet as o_snrnet
from oracle.topology import NCSNppConfig, param_specs, snrnet_param_specs
from snr_aligned_diffse_b200 import ops
from snr_aligned_diffse_b200.synth import synth_state_dict
from test_keyed_cpu import keyed_noise

pytestmark = pytest.mark.gpu

EPS = 2.0 ** -24
SEED = 0xFEDCBA9876543210
FIXED_SNR = 0.17783


@pytest.fixture(scope="module")
def sd():
    return synth_state_dict(param_specs(NCSNppConfig()), seed=0)


@pytest.fixture(scope="module")
def v3(sd):
    from snr_aligned_diffse_b200.sgmse.model import ScoreModel
    m = ScoreModel.from_state_dict(sd, backbone="ncsnpp", sde="ouve", model_type="sebridge_v3", snr_conditioned="true",
                                   fixed_snr=FIXED_SNR, theta=1.5, sigma_min=0.05, sigma_max=1.0, base_dir="")
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


def draw(keys, seed, tpad, lengths=None):
    B = len(keys)
    y = torch.zeros(B, 256, tpad, dtype=torch.complex64, device="cuda")
    one = torch.ones(B, dtype=torch.float32, device="cuda")
    _, _, z = ops.lincomb_keyed(y=y, b=one, d=one, keys=ops.key_tensor(keys).cuda(), seed=seed, lengths=lengths,
                                want_mean=False, want_x=False, want_z=True)
    return z


def test_keyed_stream_matches_the_contract():
    keys = [0, 0xFFFFFFFF00000001, 0xDEADBEEFCAFEF00D]
    z = draw(keys, SEED, 7552).cpu().numpy().reshape(3, -1)
    n = z.shape[1]
    for b, k in enumerate(keys):
        ref, r = keyed_noise(k, SEED, np.arange(n))
        for got, want in ((z[b].real, ref.real), (z[b].imag, ref.imag)):
            err = np.abs(got.astype(np.float64) - want)
            bound = 5 * EPS * np.abs(want) + r * 2 * np.pi * 2.0 ** -53
            assert (err <= bound).all(), (b, float((err / bound).max()), int(np.argmax(err / bound)))
    # the last pair of the Tpad 7552 item is part of the above; pin it explicitly too
    ref, _ = keyed_noise(keys[2], SEED, [n - 2, n - 1])
    assert np.allclose(z[2, -2:], ref, rtol=5 * EPS, atol=1e-14)


def test_keyed_draw_statistics():
    def corr(a, b):
        a, b = a - a.mean(), b - b.mean()
        return float((a * b).sum() / np.sqrt((a * a).sum() * (b * b).sum()))

    keys = [11, 12, 13, 14]
    z = draw(keys, 99, 2048).cpu().numpy().reshape(-1).astype(np.complex128)
    N = z.size
    assert N >= 2_000_000
    for part in (z.real, z.imag):
        assert abs(part.mean()) <= 5 * np.sqrt(0.5 / N)
        assert abs(part.var() - 0.5) <= 5 * np.sqrt(0.5 / N)        # Var(x^2) = 2 sigma^4 = 0.5
    p = np.abs(z) ** 2
    assert abs(p.mean() - 1) <= 5 / np.sqrt(N)                       # |z|^2 ~ Exp(1)
    from scipy import stats
    sub, cdf = z[::16], stats.norm(0.0, np.sqrt(0.5)).cdf
    assert stats.kstest(sub.real, cdf).pvalue > 1e-4
    assert stats.kstest(sub.imag, cdf).pvalue > 1e-4
    lim = 5 / np.sqrt(N)
    assert abs(corr(z.real, z.imag)) <= lim
    assert abs(corr(z.real[:-1], z.real[1:])) <= 5 / np.sqrt(N - 1)
    assert abs(corr(z.imag[:-1], z.imag[1:])) <= 5 / np.sqrt(N - 1)
    zk = draw([k + 1 for k in keys], 99, 2048).cpu().numpy().reshape(-1)      # keys k / k+1 (rows 0..2 overlap)
    zs = draw(keys, 100, 2048).cpu().numpy().reshape(-1)                      # seeds s / s+1
    m = N // 4
    for other in (zk, zs):
        assert abs(corr(z.real, other.real)) <= lim and abs(corr(z.imag, other.imag)) <= lim
    assert np.array_equal(zk[:3 * m], z[m:])                                   # key 12 is key 12 in any row


def test_keyed_kernel_equals_lincomb_on_its_draw_in_any_row():
    g = torch.Generator(device="cuda").manual_seed(5)
    B, tpad = 4, 128
    c = lambda: torch.randn(B, 1, 256, tpad, dtype=torch.complex64, device="cuda", generator=g)  # noqa: E731
    x, y, s = c(), c(), c()
    a, b, cc, d = (torch.rand(B, device="cuda", generator=g) for _ in range(4))
    keys = [3, 1 << 63, 77, (1 << 64) - 1]
    kt = ops.key_tensor(keys).cuda()
    m, xt, z = ops.lincomb_keyed(x, y, s, a, b, cc, d, keys=kt, seed=SEED, want_z=True)
    m2, xt2 = ops.lincomb(x, y, s, z, a, b, cc, d)
    assert torch.equal(m, m2) and torch.equal(xt, xt2) and torch.isfinite(xt).all()
    perm = [2, 0, 3, 1]
    _, xp, zp = ops.lincomb_keyed(x[perm], y[perm], s[perm], a[perm], b[perm], cc[perm], d[perm], keys=kt[perm],
                                  seed=SEED, want_mean=False, want_z=True)
    assert torch.equal(xp, xt[perm]) and torch.equal(zp, z[perm])
    for r in range(B):                                                        # batch of one
        _, x1, _ = ops.lincomb_keyed(x[r:r + 1], y[r:r + 1], s[r:r + 1], a[r:r + 1], b[r:r + 1], cc[r:r + 1],
                                     d[r:r + 1], keys=kt[r:r + 1], seed=SEED, want_mean=False)
        assert torch.equal(x1[0], xt[r])
    # lengths: 16255 pads to 128 frames, 16384 to 192 and 8191 to 64 -> items 1 and 2 are NaN, the rest unchanged
    lens = torch.tensor([16255, 16384, 8191, 12000], dtype=torch.int32, device="cuda")
    m3, x3, z3 = ops.lincomb_keyed(x, y, s, a, b, cc, d, keys=kt, seed=SEED, lengths=lens, want_z=True)
    for t_new, t_ref in ((m3, m), (x3, xt), (z3, z)):
        assert torch.equal(t_new[[0, 3]], t_ref[[0, 3]])
        assert torch.isnan(torch.view_as_real(t_new[[1, 2]])).all()
    with pytest.raises(ValueError):
        ops.lincomb_keyed(y=y[:, :, :128], b=b, d=d, keys=kt, seed=1)           # not [B, ..., 256, Tpad]
    with pytest.raises(ValueError):
        ops.lincomb_keyed(y=y, b=b, d=d, keys=kt.cpu(), seed=1)
    with pytest.raises(ValueError):
        ops.lincomb_keyed(y=y, b=b, d=d, keys=kt, seed=-1)


# one Tpad bucket (64 frames), 2..4 16-frame clusters each (one cluster would make the reference's estimate NaN)
LENS = [2200, 4500, 7000, 8191, 3000]
KEYS = [17, (1 << 64) - 9, 1 << 40, 5, 123456789]


def _mixtures(lens, seed=7):
    g = torch.Generator().manual_seed(seed)
    y = torch.zeros(len(lens), max(lens))
    for b, L in enumerate(lens):
        y[b, :L] = torch.randn(L, generator=g) * (0.02 + 0.08 * b) + 0.1 * torch.sin(torch.arange(L) * (0.03 + 0.01 * b))
    return y


def test_keyed_batch_equals_each_file_alone_with_the_estimator(v3, estimator, snr_sd, sd):
    y = _mixtures(LENS)
    lens = torch.tensor(LENS, dtype=torch.int32)
    out, aux = v3.enhance_batch(y, lengths=lens, keys=KEYS, seed=SEED, return_aux=True)
    out = out.cpu()
    assert torch.isfinite(out).all()
    for b, L in enumerate(LENS):
        alone = v3.enhance(None, y[b:b + 1, :L], key=KEYS[b], seed=SEED)
        assert np.array_equal(alone, out[b, :L].numpy()), b
        assert torch.count_nonzero(out[b, L:]) == 0
        ref_ratio = float(o_snrnet.estimate_noise_over_clean(snr_sd, y[b:b + 1, :L])[0, 0])
        idx, t, _ = o_sampler.v3_scalars(ref_ratio, FIXED_SNR, float(y[b, :L].abs().max()))
        assert int(aux["t_index"][b]) == idx and float(aux["t"][b]) == np.float32(t), b
    perm = [3, 0, 4, 2, 1]
    outp = v3.enhance_batch(y[perm], lengths=lens[perm], keys=[KEYS[p] for p in perm], seed=SEED).cpu()
    assert torch.equal(outp, out[perm])
    # device lengths, device keys: same bits
    outd = v3.enhance_batch(y.cuda(), lengths=lens.cuda(), keys=ops.key_tensor(KEYS).cuda(), seed=SEED).cpu()
    assert torch.equal(outd, out)
    # against the oracle on the file alone, fed the same Z
    for b in (0, 3):
        L = LENS[b]
        ref_ratio = float(o_snrnet.estimate_noise_over_clean(snr_sd, y[b:b + 1, :L])[0, 0])
        ref = o_sampler.enhance_v3(sd, y[b:b + 1, :L], aux["Z"][b:b + 1].cpu(), ref_ratio, FIXED_SNR,
                                   sigma_max=1.0)["x_hat"].double().numpy()
        got = out[b, :L].double().numpy()
        assert o_sampler.si_sdr(ref, got) >= 30.0
        assert np.abs(got - ref).max() <= 0.04 * np.abs(ref).max()


def test_keyed_enhance_batch_rejects_what_it_cannot_honour(v3, estimator):
    y = _mixtures([3000, 9000])
    with pytest.raises(ValueError):                                           # Tpad 64 vs the buffer's 128
        v3.enhance_batch(y, lengths=torch.tensor([3000, 9000]), keys=[1, 2], seed=1)
    with pytest.raises(ValueError):
        v3.enhance_batch(y, keys=[1, 2], seed=1, noise=torch.zeros(2, 1, 256, 128, dtype=torch.complex64))
    with pytest.raises(ValueError):
        v3.enhance_batch(y, keys=[1, 2], seed=1, generator=torch.Generator(device="cuda"))
    out = v3.enhance_batch(y.cuda(), lengths=torch.tensor([3000, 9000], device="cuda"), keys=[1, 2], seed=1)
    assert torch.isnan(out[0]).any() and torch.isfinite(out[1]).all()     # device lengths: the mismatched item is NaN


def test_keyed_sweep_and_graphs_return_each_file_alone(v3, estimator):
    from snr_aligned_diffse_b200.pipeline import GraphedEnhancer, GraphedEnhancerCache
    from snr_aligned_diffse_b200.sweep import enhance_sweep
    g = torch.Generator().manual_seed(11)
    lens = [5000, 9000, 8100, 16500, 8000, 5100, 23000]
    waves = [torch.randn(n, generator=g) * 0.05 + 0.1 * torch.sin(torch.arange(n) * 0.03) for n in lens]
    merged = {}
    for world, mb, tf in ((1, 3, None), (2, 3, None), (1, 1, 300), (2, 1, 160)):
        cache = GraphedEnhancerCache(v3, "cuda")
        for rank in range(world):
            r = enhance_sweep(cache, waves, rank=rank, world=world, max_batch=mb, target_frames=tf, device="cuda",
                              keep_audio=True, seed=SEED)
            for i, a in r["audio"].items():
                if i in merged:
                    assert torch.equal(merged[i], a), (world, mb, tf, i)
                merged[i] = a
    assert sorted(merged) == list(range(len(lens)))
    for i, w in enumerate(waves):
        alone = v3.enhance(None, w[None], key=i, seed=SEED)
        assert np.array_equal(alone, merged[i].numpy()), i

    y = _mixtures([8000, 6000, 7000])
    pipe = GraphedEnhancer(v3, 3, y.shape[1], "cuda", keyed=True, seed=SEED).capture()
    pipe.y_dev.copy_(y)
    torch.cuda.synchronize()
    for keys in ([4, 5, 6], [(1 << 64) - 1, 5, 9]):
        pipe.set_keys(keys)
        res = pipe.replay()
        pipe.stream.synchronize()
        got = res.clone()
        eager = v3.enhance_batch(y, keys=keys, seed=SEED)
        assert torch.equal(got, eager), keys
        if keys[0] == 4:
            first = got
    assert torch.equal(got[1], first[1]) and not torch.equal(got[0], first[0]) and not torch.equal(got[2], first[2])
