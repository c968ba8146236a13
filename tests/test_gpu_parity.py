"""GPU parity tests (run with -m gpu on a B200): every CUDA kernel, called through the C ABI, against
the CPU oracle / committed golden fixtures on the same seeded inputs.

Tolerances (stated per test):
  * integer / index results (frame counts, padded lengths, zero padding, t_30 index): bit-exact
  * fp32 kernels (STFT, iSTFT, SNRNet, FIR fp32, scalars): 1e-5-level relative to the signal peak
  * bf16-storage kernels: the bf16 rounding of the stored result (2^-8 relative) on top of an fp32 reference
    evaluated on the same bf16-rounded operands
  * whole network in bf16 vs the fp32 oracle: relative L2 <= 2e-2 on the network output (<= 2.5e-2 on every
    module's activation at the 256 x 64 fixture shape), SI-SDR of the enhanced waveform against the oracle waveform
    >= 30 dB in tests/test_gpu_api.py / test_gpu_configs.py (SURVEY 7: bf16 autocast of the reference
    itself sits at 1.5e-2 / 30.7 dB on these random weights)
"""
import math
import os

import numpy as np
import pytest
import torch

from oracle import frontend, ncsnpp as o_ncsnpp, sampler as o_sampler, snrnet as o_snrnet
from oracle.topology import NCSNppConfig, param_specs, snrnet_param_specs
from snr_aligned_diffse_b200.synth import synth_state_dict

pytestmark = pytest.mark.gpu

DEV = "cuda"


def _c(a):
    return torch.from_numpy(np.ascontiguousarray(a))


def rel_l2(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a - b).norm() / (b.norm() + 1e-30))


def si_sdr(ref, est):
    return o_sampler.si_sdr(ref.double().cpu().numpy(), est.double().cpu().numpy())


@pytest.fixture(scope="module")
def ops():
    from snr_aligned_diffse_b200 import ops
    return ops


@pytest.fixture(scope="module")
def sd():
    return synth_state_dict(param_specs(NCSNppConfig()), seed=0)


@pytest.fixture(scope="module")
def engine(sd):
    from snr_aligned_diffse_b200.engine import NCSNppEngine
    return NCSNppEngine().load_state_dict(sd, DEV)


# ----------------------------------------------------------------------------------------------- front end
def test_stft_matches_oracle_and_golden(ops, golden_dir):
    z = np.load(os.path.join(golden_dir, "frontend.npz"))
    wave = _c(z["wave"]).to(DEV)
    L = wave.shape[1]
    Y = ops.stft(wave)
    assert Y.shape == (2, 256, frontend.padded_frames(L))                      # bit-exact geometry
    nf = frontend.n_frames(L)
    assert torch.count_nonzero(torch.view_as_real(Y[..., nf:])) == 0           # pad_spec region is exactly zero
    ref = _c(z["spec"]).squeeze(1)
    peak = ref.abs().max()
    assert (Y.cpu() - ref).abs().max() <= 2e-5 * peak                           # fp32 shared-memory FFT vs torch.stft
    raw = ops.stft(wave, transform=False, tpad=nf)
    assert (raw.cpu() - _c(z["stft"])).abs().max() <= 2e-5 * _c(z["stft"]).abs().max()
    # SNR-branch features: y / max|y|, raw STFT, planar re/im, padded to a multiple of 16 (model.py:715-719)
    pk = ops.absmax(wave[:1])
    assert float(pk[0]) == float(wave[:1].abs().max())
    feat = ops.stft(wave[:1], scale=pk, scale_is_divisor=True, transform=False, planar=True, pad_multiple=16)
    g = _c(z["snr_feat"])
    assert feat.shape == g.shape
    assert (feat.cpu() - g).abs().max() <= 2e-5 * g.abs().max()


def test_absmax_is_exact_on_ragged_batches(ops):
    """max |y| per utterance (model.py:715,726): exact (a maximum has no rounding), also with ragged lengths, lengths that
    are not multiples of the 8192-sample block chunk, and values past len[b] that must be ignored."""
    g = torch.Generator().manual_seed(6)
    w = torch.randn(5, 70001, generator=g)
    lens = torch.tensor([70001, 1, 8192, 8193, 40000], dtype=torch.int32)
    w[1, 0] = -0.25
    w[2, 9000] = 99.0                                  # beyond len[2]: must not count
    got = ops.absmax(w.to(DEV), lens.to(DEV)).cpu()
    ref = torch.stack([w[b, :int(lens[b])].abs().max() for b in range(5)])
    assert torch.equal(got, ref)
    assert torch.equal(ops.absmax(w.to(DEV)).cpu(), w.abs().amax(dim=1))


def test_istft_matches_oracle_and_golden(ops, golden_dir):
    z = np.load(os.path.join(golden_dir, "frontend.npz"))
    spec = _c(z["spec"]).squeeze(1).to(DEV)
    L = z["wave"].shape[1]
    out = ops.istft(spec, L)
    ref = _c(z["istft"])
    assert out.shape == ref.shape
    assert (out.cpu() - ref).abs().max() <= 2e-5 * ref.abs().max()
    # padded frames participate (SURVEY 7 "padded-frame leak"): for a shorter requested length the frames
    # >= n_frames(Lq) act as padded frames; perturbing one must change exactly the tail from nf*128-255 on
    Lq = 7900
    nfq = frontend.n_frames(Lq)
    outq = ops.istft(spec, Lq)
    assert (outq.cpu() - frontend.istft(frontend.spec_back(spec.cpu()), Lq)).abs().max() <= 2e-5 * ref.abs().max()
    spec2 = spec.clone()
    spec2[:, :, nfq] += 0.05
    out2 = ops.istft(spec2, Lq)
    first = nfq * 128 - 255
    assert torch.equal(out2[:, :first], outq[:, :first]) and not torch.equal(out2[:, first:], outq[:, first:])


@pytest.mark.parametrize("L", [256, 383, 384, 8191, 8192, 8193, 64000])
def test_stft_istft_round_trip_and_ragged(ops, L):
    g = torch.Generator().manual_seed(L)
    w = (torch.randn(3, L, generator=g) * 0.1)
    lens = torch.tensor([L, max(256, L - 129), max(256, L // 2)], dtype=torch.int32)
    for b in range(3):
        w[b, lens[b]:] = 0
    Y = ops.stft(w.to(DEV), lengths=lens.to(DEV))
    for b in range(3):
        Lb = int(lens[b])
        ref = frontend.pad_spec(frontend.spec_fwd(frontend.stft(w[b:b + 1, :Lb])).unsqueeze(1)).squeeze(1)
        got = Y[b:b + 1, :, :ref.shape[-1]].cpu()
        assert (got - ref).abs().max() <= 3e-5 * ref.abs().max()
        assert torch.count_nonzero(torch.view_as_real(Y[b, :, frontend.n_frames(Lb):])) == 0
    back = ops.istft(Y, L, lengths=lens.to(DEV))
    for b in range(3):
        Lb = int(lens[b])
        # the reference inverts the PADDED spectrogram (all Tpad frames enter the window envelope), so the
        # last samples are attenuated exactly as torch.istft attenuates them; before that it is a round trip
        ref = frontend.istft(frontend.spec_back(Y[b:b + 1].cpu()), Lb)[0]
        assert (back[b, :Lb].cpu() - ref).abs().max() <= 1e-5
        exact = max(0, frontend.n_frames(Lb) * 128 - 255)
        assert (back[b, :exact].cpu() - w[b, :exact]).abs().max() <= 1e-4
        assert torch.count_nonzero(back[b, Lb:]) == 0


def test_v3_scalars_bit_exact(ops, golden_dir):
    z = np.load(os.path.join(golden_dir, "scalars.npz"))
    assert np.array_equal(z["t_30"], ops.T_30)
    rows = z["rows"]
    for fs in np.unique(rows[:, 0]):
        sel = rows[rows[:, 0] == fs]
        ratio = torch.tensor(sel[:, 1], dtype=torch.float32, device=DEV)
        peak = torch.ones_like(ratio)
        t, nf, idx = ops.v3_scalars(ratio, peak, float(fs))
        assert np.array_equal(idx.cpu().numpy(), sel[:, 2].astype(np.int32))          # snapped grid index: exact
        assert np.array_equal(t.cpu().numpy(), sel[:, 3].astype(np.float32))          # t: exact
        assert np.abs(nf.cpu().numpy() - sel[:, 4]).max() <= 2e-7                       # normfac: 1 ulp


@pytest.mark.filterwarnings("ignore:std")     # torch warns about the single-cluster case exercised on purpose
def test_snrnet_matches_golden(ops, golden_dir):
    z = np.load(os.path.join(golden_dir, "snrnet.npz"))
    net = ops.SNRNetEngine().load_state_dict(synth_state_dict(snrnet_param_specs(), seed=1), DEV)
    out = net.forward(_c(z["feat"]).to(DEV))
    assert np.abs(out.cpu().numpy() - z["out"][:, 0]).max() <= 2e-5
    # longer input / batch of 3: against the oracle
    feat = torch.randn(3, 2, 256, 96, generator=torch.Generator().manual_seed(3))
    ref = o_snrnet.snrnet_forward(synth_state_dict(snrnet_param_specs(), seed=1), feat)[:, 0]
    got = net.forward(feat.to(DEV)).cpu()
    assert (got - ref).abs().max() <= 2e-5
    # a single 16-frame cluster (utterances shorter than 16 frames): the unbiased std over one element is NaN in the
    # reference (torch.std, snrnet.py:84) and the NaN propagates to the estimate -- same here, for that sample only
    one = torch.randn(2, 2, 256, 16, generator=torch.Generator().manual_seed(4))
    ref1 = o_snrnet.snrnet_forward(synth_state_dict(snrnet_param_specs(), seed=1), one)[:, 0]
    got1 = net.forward(one.to(DEV)).cpu()
    assert torch.isnan(ref1).all() and torch.isnan(got1).all()


# ----------------------------------------------------------------------------------------------- operators
def _nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


def _pack_w3(w):  # [Cout,Cin,3,3] -> [Cout, 9*Cin] (tap-major, cin inner)
    return w.permute(0, 2, 3, 1).reshape(w.shape[0], -1).contiguous()


CONV_CASES = [
    # B, H, W, Cin, Cout, taps
    (2, 32, 64, 128, 128, 9),
    (1, 16, 24, 256, 256, 9),
    (2, 8, 8, 384, 128, 9),
    (1, 4, 3, 512, 256, 9),
    (1, 256, 64, 128, 128, 9),
    (2, 16, 16, 256, 768, 1),
    (3, 4, 1, 256, 256, 1),
    (16, 64, 64, 256, 256, 9),     # >= 148 super-tiles: two sub-tiles per weight tile, single TMEM buffer
    (4, 128, 112, 128, 128, 9),    # two sub-tiles, double-buffered TMEM, W not a multiple of 16... (112 = 7*16)
    (1, 24, 40, 128, 256, 9),      # ragged super-tiles (H % 16 != 0, W % 16 != 0)
    (2, 8, 16, 512, 256, 9),       # H = 8: one sub-tile
    (2, 40, 12, 128, 128, 9),      # W % 8 != 0, H % 16 != 0 (8-pixel-wide halo tiles of the 2-CTA kernel)
    (3, 72, 20, 128, 256, 9),      # odd number of super-tiles: the peer CTA of the last pair runs an all-padding tile
]


@pytest.mark.parametrize("impl", [0, 2, 1], ids=["tcgen05", "tcgen05gemm", "cudacore"])
@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_nhwc(ops, case, impl):
    B, H, W, Ci, Co, taps = case
    if impl == 1 and Co > 256:
        pytest.skip("cross-check kernel handles N <= 256")
    g = torch.Generator().manual_seed(hash(case) % 1000)
    x = torch.randn(B, Ci, H, W, generator=g).to(torch.bfloat16)
    k = 3 if taps == 9 else 1
    w = (torch.randn(Co, Ci, k, k, generator=g) / math.sqrt(Ci * taps)).to(torch.bfloat16)
    bias = torch.randn(Co, generator=g) * 0.1
    ref = torch.nn.functional.conv2d(x.float(), w.float(), bias, padding=k // 2)
    wt = _pack_w3(w) if taps == 9 else w.reshape(Co, Ci).contiguous()
    out = ops.conv_nhwc(_nhwc(x).to(DEV), wt.to(DEV), taps, bias=bias.to(DEV), impl=impl)
    got = out.float().cpu().permute(0, 3, 1, 2)
    err = (got - ref).abs()
    assert (err <= 2 ** -7 * ref.abs() + 2e-2 * ref.abs().mean()).all(), float(err.max())


@pytest.mark.parametrize("impl", [0, 2, 1], ids=["tcgen05", "tcgen05gemm", "cudacore"])
def test_conv_fused_shortcut_residual_tbias(ops, impl):
    # Conv_1 (3x3) + Conv_2 (1x1 shortcut) in one K loop, then * 1/sqrt(2)  (layerspp.py:268-276)
    g = torch.Generator().manual_seed(7)
    B, H, W, C1, C2, Co = 2, 16, 32, 128, 384, 128
    a = torch.randn(B, C1, H, W, generator=g).to(torch.bfloat16)
    x = torch.randn(B, C2, H, W, generator=g).to(torch.bfloat16)
    w1 = (torch.randn(Co, C1, 3, 3, generator=g) / math.sqrt(9 * C1)).to(torch.bfloat16)
    w2 = (torch.randn(Co, C2, 1, 1, generator=g) / math.sqrt(C2)).to(torch.bfloat16)
    b1, b2 = torch.randn(Co, generator=g) * 0.1, torch.randn(Co, generator=g) * 0.1
    s = 1 / math.sqrt(2)
    ref = (torch.nn.functional.conv2d(a.float(), w1.float(), b1, padding=1) +
           torch.nn.functional.conv2d(x.float(), w2.float(), b2)) * s
    wt = torch.cat([_pack_w3(w1), w2.reshape(Co, C2)], dim=1).contiguous()
    out = ops.conv_nhwc(_nhwc(a).to(DEV), wt.to(DEV), 9, x1=_nhwc(x).to(DEV), bias=(b1 + b2).to(DEV), scale=s, impl=impl)
    got = out.float().cpu().permute(0, 3, 1, 2)
    assert ((got - ref).abs() <= 2 ** -7 * ref.abs() + 2e-2 * ref.abs().mean()).all()
    # residual + per-sample time-embedding bias
    res = torch.randn(B, Co, H, W, generator=g).to(torch.bfloat16)
    tb = torch.randn(B, Co, generator=g) * 0.2
    ref2 = (torch.nn.functional.conv2d(a.float(), w1.float(), b1, padding=1) + tb[:, :, None, None] + res.float()) * s
    out2 = ops.conv_nhwc(_nhwc(a).to(DEV), _pack_w3(w1).to(DEV), 9, bias=b1.to(DEV), tbias=tb.to(DEV),
                         res=_nhwc(res).to(DEV), scale=s, impl=impl)
    got2 = out2.float().cpu().permute(0, 3, 1, 2)
    assert ((got2 - ref2).abs() <= 2 ** -7 * ref2.abs() + 2e-2 * ref2.abs().mean()).all()


@pytest.mark.parametrize("case", [(2, 32, 64, 128, 128, 0), (2, 40, 20, 256, 256, 0), (1, 16, 24, 384, 128, 384),
                                  (3, 72, 12, 128, 256, 0), (16, 64, 64, 256, 256, 0), (2, 8, 8, 512, 256, 512),
                                  # 128 output channels + shortcut: the shortcut operand's own ring, two sub-tiles, more
                                  # cluster tiles than clusters (persistent walk); ragged with an odd tile count
                                  (2, 160, 128, 128, 128, 256), (3, 72, 20, 128, 128, 128)])
def test_gn_silu_conv3x3_fused_equals_unfused(ops, case):
    """GroupNorm+SiLU applied inside the convolution (2-CTA kernel) == separate GroupNorm pass + convolution, bit for
    bit, and both match the fp32 PyTorch chain (layerspp.py:245-271)."""
    B, H, W, Ci, Co, Cs = case
    g = torch.Generator().manual_seed(sum(case))
    x = (torch.randn(B, Ci, H, W, generator=g) * 1.3 + 0.2).to(torch.bfloat16)
    xs = torch.randn(B, Cs, H, W, generator=g).to(torch.bfloat16) if Cs else None
    w = (torch.randn(Co, Ci, 3, 3, generator=g) / math.sqrt(9 * Ci)).to(torch.bfloat16)
    w2 = (torch.randn(Co, Cs, 1, 1, generator=g) / math.sqrt(Cs)).to(torch.bfloat16) if Cs else None
    gamma, beta = torch.rand(Ci, generator=g) + 0.5, torch.randn(Ci, generator=g) * 0.2
    bias, tb = torch.randn(Co, generator=g) * 0.1, torch.randn(B, Co, generator=g) * 0.2
    res = None if Cs else torch.randn(B, Co, H, W, generator=g).to(torch.bfloat16)
    wt = _pack_w3(w) if not Cs else torch.cat([_pack_w3(w), w2.reshape(Co, Cs)], dim=1).contiguous()
    dev = lambda t: None if t is None else t.to(DEV)
    kw = dict(x1=dev(None if xs is None else _nhwc(xs)), bias=dev(bias), tbias=dev(tb),
              res=dev(None if res is None else _nhwc(res)), scale=0.7)
    fused = ops.gn_silu_conv3x3_nhwc(dev(_nhwc(x)), dev(gamma), dev(beta), dev(wt), **kw)
    a = ops.groupnorm_nhwc(dev(_nhwc(x)), dev(gamma), dev(beta), silu=True)
    unfused = ops.conv_nhwc(a, dev(wt), 9, impl=0, **kw)
    assert torch.equal(fused, unfused)
    ref = torch.nn.functional.conv2d(torch.nn.functional.silu(torch.nn.functional.group_norm(x.float(), 32, gamma, beta, 1e-6)),
                                     w.float(), bias, padding=1) + tb[:, :, None, None]
    if Cs:
        ref = ref + torch.nn.functional.conv2d(xs.float(), w2.float())
    else:
        ref = ref + res.float()
    ref = ref * 0.7
    got = fused.float().cpu().permute(0, 3, 1, 2)
    err = (got - ref).abs()
    assert (err <= 2 ** -6 * ref.abs() + 3e-2 * ref.abs().mean()).all(), float(err.max())


def test_shortcut_ring_batch_invariance(ops):
    """The 128-channel fused-shortcut layers stream the 1x1 operand through its own ring with an interleaved K order
    (conv_halo2.cu).  The K order depends on the layer only: every sample of a batch equals the same sample run alone,
    bit for bit, although the batch of 6 walks two sub-tiles per weight tile and the single sample one; the result
    matches the fp32 convolution."""
    g = torch.Generator().manual_seed(5)
    B, H, W, C0, C1, Co = 6, 96, 64, 128, 256, 128
    a = torch.randn(B, C0, H, W, generator=g).to(torch.bfloat16)
    x = torch.randn(B, C1, H, W, generator=g).to(torch.bfloat16)
    w1 = (torch.randn(Co, C0, 3, 3, generator=g) / math.sqrt(9 * C0)).to(torch.bfloat16)
    w2 = (torch.randn(Co, C1, 1, 1, generator=g) / math.sqrt(C1)).to(torch.bfloat16)
    bias = torch.randn(Co, generator=g) * 0.1
    wt = torch.cat([_pack_w3(w1), w2.reshape(Co, C1)], dim=1).contiguous().to(DEV)
    an, xn = _nhwc(a).to(DEV), _nhwc(x).to(DEV)
    full = ops.conv_nhwc(an, wt, 9, x1=xn, bias=bias.to(DEV), impl=0)
    for b in (0, 5):
        alone = ops.conv_nhwc(an[b:b + 1].contiguous(), wt, 9, x1=xn[b:b + 1].contiguous(), bias=bias.to(DEV), impl=0)
        assert torch.equal(alone[0], full[b]), b
    ref = (torch.nn.functional.conv2d(a.float(), w1.float(), bias, padding=1) + torch.nn.functional.conv2d(x.float(), w2.float()))
    got = full.float().cpu().permute(0, 3, 1, 2)
    assert ((got - ref).abs() <= 2 ** -7 * ref.abs() + 2e-2 * ref.abs().mean()).all()


@pytest.mark.parametrize("case", [(2, 32, 64, 128, 128), (3, 40, 20, 128, 256), (16, 64, 64, 256, 256), (1, 24, 12, 256, 128),
                                  (5, 72, 20, 128, 128)])
def test_conv_epilogue_groupnorm_partials(ops, case):
    """The 2-CTA kernel's epilogue accumulates per-unit sums / sums of squares of its (pre-rounding fp32) result in
    64-bit fixed point; they must match the sums over the stored bf16 tensor up to the bf16 rounding of the elements,
    with ragged tiles, an odd tile count (all-padding peer tile) and several images per CTA."""
    B, H, W, Ci, Co = case
    g = torch.Generator().manual_seed(sum(case))
    x = torch.randn(B, Ci, H, W, generator=g).to(torch.bfloat16)
    w = (torch.randn(Co, Ci, 3, 3, generator=g) / math.sqrt(9 * Ci)).to(torch.bfloat16)
    bias = torch.randn(Co, generator=g) * 0.3
    res = torch.randn(B, Co, H, W, generator=g).to(torch.bfloat16)
    out, st, raw = ops.conv3x3_nhwc_stats(_nhwc(x).to(DEV), _pack_w3(w).to(DEV), bias=bias.to(DEV),
                                          res=_nhwc(res).to(DEV), scale=0.7)
    # integer accumulation: identical bits on a second run, and for a sample processed alone
    _, _, raw2 = ops.conv3x3_nhwc_stats(_nhwc(x).to(DEV), _pack_w3(w).to(DEV), bias=bias.to(DEV), res=_nhwc(res).to(DEV),
                                        scale=0.7)
    _, _, raw1 = ops.conv3x3_nhwc_stats(_nhwc(x[-1:]).to(DEV), _pack_w3(w).to(DEV), bias=bias.to(DEV),
                                        res=_nhwc(res[-1:]).to(DEV), scale=0.7)
    assert torch.equal(raw, raw2) and torch.equal(raw[-1:], raw1)
    plain = ops.conv_nhwc(_nhwc(x).to(DEV), _pack_w3(w).to(DEV), 9, bias=bias.to(DEV), res=_nhwc(res).to(DEV), scale=0.7)
    assert torch.equal(out, plain)
    o = out.double().cpu().reshape(B, H * W, Co // 4, 4)
    want_s, want_q = o.sum((1, 3)), (o * o).sum((1, 3))
    st = st.cpu()
    n = H * W * 4
    assert st.shape == (B, Co // 4, 2) and torch.isfinite(st).all()
    assert ((st[..., 0] - want_s).abs() <= 2 ** -8 * math.sqrt(n) * 2.0 + 2 ** -9 * want_s.abs()).all()
    assert ((st[..., 1] - want_q).abs() <= 2 ** -7 * want_q).all()


@pytest.mark.parametrize("C,H,W", [(128, 32, 64), (256, 16, 16), (384, 8, 12), (512, 4, 1), (128, 256, 64)])
@pytest.mark.parametrize("silu", [True, False])
def test_groupnorm(ops, C, H, W, silu):
    g = torch.Generator().manual_seed(C + H)
    x = (torch.randn(2, C, H, W, generator=g) * 1.7 + 0.4).to(torch.bfloat16)
    gamma, beta = 1 + 0.1 * torch.randn(C, generator=g), 0.1 * torch.randn(C, generator=g)
    ref = torch.nn.functional.group_norm(x.float(), 32, gamma, beta, eps=1e-6)
    if silu:
        ref = torch.nn.functional.silu(ref)
    out = ops.groupnorm_nhwc(_nhwc(x).to(DEV), gamma.to(DEV), beta.to(DEV), silu=silu)
    got = out.float().cpu().permute(0, 3, 1, 2)
    assert ((got - ref).abs() <= 2 ** -7 * ref.abs() + 2e-3).all()


@pytest.mark.parametrize("mag", [2e-3, 1.0, 400.0], ids=["tiny", "unit", "large"])
def test_groupnorm_statistics_hold_over_the_activation_range(ops, mag):
    """The 64-bit fixed-point GroupNorm sums (gn_fixed.cuh: 2^-30 / 2^-20) neither lose small activations to rounding
    nor wrap on large ones: rms 2e-3 (squares ~ eps) .. 400 on a 2 x 128 x 256 x 128 map, both the stand-alone statistics
    pass and the convolution epilogue's sums, against fp32 group_norm / exact fp64 sums of the stored tensor."""
    g = torch.Generator().manual_seed(3)
    C, H, W = 128, 128, 256
    x = (torch.randn(2, C, H, W, generator=g) * mag + 0.3 * mag).to(torch.bfloat16)
    gamma, beta = 1 + 0.1 * torch.randn(C, generator=g), 0.1 * torch.randn(C, generator=g)
    ref = torch.nn.functional.silu(torch.nn.functional.group_norm(x.float(), 32, gamma, beta, eps=1e-6))
    got = ops.groupnorm_nhwc(_nhwc(x).to(DEV), gamma.to(DEV), beta.to(DEV), silu=True).float().cpu().permute(0, 3, 1, 2)
    assert ((got - ref).abs() <= 2 ** -7 * ref.abs() + 4e-3).all()
    # epilogue sums of a convolution whose output has that magnitude (identity-like weights: centre tap only)
    wt = torch.zeros(C, 9 * C)
    wt[torch.arange(C), 4 * C + torch.arange(C)] = 1.0
    out, st, _ = ops.conv3x3_nhwc_stats(_nhwc(x).to(DEV), wt.to(torch.bfloat16).to(DEV))
    o = out.double().cpu()                                    # [B,H,W,C] as stored
    want_s = o.reshape(2, H * W, C // 4, 4).sum((1, 3))
    want_q = (o ** 2).reshape(2, H * W, C // 4, 4).sum((1, 3))
    st = st.cpu()
    assert ((st[..., 0] - want_s).abs() <= 1e-5 * want_s.abs() + 1e-3 * mag).all()
    # 1024 partials per unit, each rounded to 2^-20: ~1e-5 absolute on the unit total, i.e. 7e-11 on a per-element variance
    assert ((st[..., 1] - want_q).abs() <= 1e-5 * want_q + 4e-5).all()


def test_fir(ops, golden_dir):
    z = np.load(os.path.join(golden_dir, "fir.npz"))   # reference upfirdn2d_native outputs, fp32
    x = _c(z["x"])                                      # [2,3,6,10] -> use 4-channel fp32 path with a zero channel
    x4 = torch.cat([x, torch.zeros(2, 1, 6, 10)], dim=1)
    up = ops.fir_nhwc(_nhwc(x4).to(DEV), up=True).cpu().permute(0, 3, 1, 2)
    dn = ops.fir_nhwc(_nhwc(x4).to(DEV), up=False).cpu().permute(0, 3, 1, 2)
    assert (up[:, :3] - _c(z["up"])).abs().max() <= 1e-6 and (dn[:, :3] - _c(z["down"])).abs().max() <= 1e-6
    g = torch.Generator().manual_seed(5)
    xb = torch.randn(2, 128, 8, 12, generator=g).to(torch.bfloat16)
    for upf, fn in ((True, o_ncsnpp.fir_upsample_2d), (False, o_ncsnpp.fir_downsample_2d)):
        ref = fn(xb.float())
        got = ops.fir_nhwc(_nhwc(xb).to(DEV), up=upf).float().cpu().permute(0, 3, 1, 2)
        assert ((got - ref).abs() <= 2 ** -8 * ref.abs() + 1e-6).all()


def test_upfirdn2d_general_matches_reference_vectors(ops, golden_dir):
    """snrse_upfirdn2d (the reference's one native operator, general form) vs `upfirdn2d_native` outputs of the
    unmodified reference: output sizes exact, values within fp32 rounding (1e-6 of the peak)."""
    from snr_aligned_diffse_b200.sgmse.backbones.ncsnpp_utils import up_or_down_sampling as uds
    from snr_aligned_diffse_b200.sgmse.backbones.ncsnpp_utils.op.upfirdn2d import upfirdn2d, upfirdn2d_native
    z = np.load(os.path.join(golden_dir, "upfirdn2d.npz"))
    for i, c in enumerate(z["cases"]):
        c = [int(v) for v in c]
        x, k, ref = _c(z[f"x{i}"]), _c(z[f"k{i}"]), _c(z[f"y{i}"])
        got = upfirdn2d_native(x.to(DEV), k.to(DEV), *c[6:])
        assert got.is_cuda and tuple(got.shape) == tuple(ref.shape)
        assert (got.cpu() - ref).abs().max() <= 2e-6 * max(1.0, float(ref.abs().max()))
        oracle = o_ncsnpp.upfirdn2d_general(x, k, *c[6:])
        assert (got.cpu() - oracle).abs().max() <= 2e-6 * max(1.0, float(ref.abs().max()))
    # the reference's helpers on top of it, CPU tensor in -> CPU tensor out (the reference dispatches on device)
    fz = np.load(os.path.join(golden_dir, "fir.npz"))
    x = _c(fz["x"])
    up, dn = uds.upsample_2d(x, [1, 3, 3, 1], factor=2), uds.downsample_2d(x, [1, 3, 3, 1], factor=2)
    assert not up.is_cuda and (up - _c(fz["up"])).abs().max() <= 1e-6 and (dn - _c(fz["down"])).abs().max() <= 1e-6
    assert torch.equal(upfirdn2d(x, torch.ones(2, 2) / 4, down=2), uds.downsample_2d(x, factor=2))   # default k = box
    # a larger seeded case against the oracle, and half precision in -> half precision out
    g = torch.Generator().manual_seed(9)
    xb, kb = torch.randn(3, 5, 33, 47, generator=g), torch.randn(5, 7, generator=g)
    got = ops.upfirdn2d(xb.to(DEV), kb.to(DEV), (2, 3), (3, 2), (4, 1, 0, 6)).cpu()
    ref = o_ncsnpp.upfirdn2d_general(xb, kb, 2, 3, 3, 2, 4, 1, 0, 6)
    assert got.shape == ref.shape and (got - ref).abs().max() <= 1e-5
    assert ops.upfirdn2d(xb.half().to(DEV), kb.to(DEV), (1, 1), (1, 1), (3, 3, 2, 2)).dtype == torch.float16
    with pytest.raises(RuntimeError):
        ops.upfirdn2d(xb[:, :, :2, :2].to(DEV), kb.to(DEV))          # padded input smaller than the kernel
    with pytest.raises(RuntimeError):
        ops.upfirdn2d(xb[0].to(DEV), kb.to(DEV))                      # not [N, C, H, W]


@pytest.mark.parametrize("n", [4, 12, 64, 200, 128, 512, 1984])   # n % 64 == 0: tensor-core path
def test_attention(ops, n):
    g = torch.Generator().manual_seed(n)
    B, C = 2, 256
    q, k, v = (torch.randn(B, n, C, generator=g).to(torch.bfloat16) for _ in range(3))
    w = torch.softmax(torch.einsum("bic,bjc->bij", q.float(), k.float()) * C ** -0.5, dim=-1)
    ref = torch.einsum("bij,bjc->bic", w, v.float())
    got = ops.attention_nhwc(q.to(DEV), k.to(DEV), v.to(DEV)).float().cpu()
    # fp32 CUDA-core path: bf16 rounding of the output only; tensor-core path (n % 64 == 0): the softmax probabilities
    # are additionally rounded to bf16 before P V (absolute error <= 2^-9 * sum_j p_j |v_j|)
    atol = 1e-3 if n % 64 else 2 ** -9 * float(v.float().abs().max())
    assert ((got - ref).abs() <= 2 ** -7 * ref.abs() + atol).all()


def test_attention_query_blocks_bound_the_score_memory(ops):
    """n = 6016 tokens (between the 10 s and 60 s shapes): B*n*n*6 bytes exceeds the score budget, so the queries are
    walked in blocks (5568 + 448 rows) per utterance; every block is a full softmax over all keys -> same result as the
    single-pass formula, and the workspace stays below the budget + V^T instead of growing with n^2."""
    from snr_aligned_diffse_b200 import _lib
    n, C, B = 6016, 256, 2
    g = torch.Generator().manual_seed(n)
    q, k, v = (torch.randn(B, n, C, generator=g).to(torch.bfloat16) for _ in range(3))
    ws = int(_lib.load().snrse_attention_workspace_bytes(B, n, C))
    assert ws < (192 << 20) + B * C * n * 2 + 4096 < B * n * n * 6
    got = ops.attention_nhwc(q.to(DEV), k.to(DEV), v.to(DEV)).float().cpu()
    qd, kd, vd = q.to(DEV).float(), k.to(DEV).float(), v.to(DEV).float()      # fp32 torch reference, on the GPU for speed
    w = torch.softmax(torch.einsum("bic,bjc->bij", qd, kd) * C ** -0.5, dim=-1)
    ref = torch.einsum("bij,bjc->bic", w, vd).cpu()
    atol = 2 ** -9 * float(v.float().abs().max())
    assert ((got - ref).abs() <= 2 ** -7 * ref.abs() + atol).all()


# ----------------------------------------------------------------------------------------------- network
def _network_report(engine, sd, x, t, flags):
    """Run oracle + engine with activation taps; return (out_ref, out_gpu, per-module rel-L2 list)."""
    taps = {}
    with torch.no_grad():
        ref = o_ncsnpp.ncsnpp_forward(sd, x, t, taps=taps)
    B, _, F, T = x.shape
    out = engine.forward(x[:, 0].to(DEV), x[:, 1].to(DEV), t.to(DEV), mode=0, flags=flags | 1)
    torch.cuda.synchronize()
    rep = []
    for idx in sorted(taps):
        got = engine.read_tap(B, F, T, idx).cpu()
        rep.append((idx, rel_l2(got, taps[idx])))
    return ref[:, 0], out.cpu(), rep


# id -> (plan flags, check every module's output through the keep-all plan, PDL mask or None for the library default).
# Without taps the plan reuses activation buffers as the product does; PDL masks 0 (plain stream order) and 7 (every
# launch) are supported configurations (SNRSE_PDL) and must give the same bits as the default mask.
GOLDEN_RUNS = {
    "cuda-core-conv": (2, True, None), "tcgen05-conv": (0, True, None),
    "cuda-core-conv-reused-buffers": (2, False, None), "tcgen05-conv-reused-buffers": (0, False, None),
    "cuda-core-conv-pdl-off": (2, False, 0), "tcgen05-conv-pdl-off": (0, False, 0),
    "cuda-core-conv-pdl-all": (2, False, 7), "tcgen05-conv-pdl-all": (0, False, 7),
}


@pytest.mark.parametrize("run", list(GOLDEN_RUNS))
def test_ncsnpp_forward_vs_golden(engine, sd, golden_dir, run):
    from snr_aligned_diffse_b200 import _lib
    flags, taps, pdl = GOLDEN_RUNS[run]
    z = np.load(os.path.join(golden_dir, "ncsnpp_forward.npz"))
    x, t = _c(z["x"]), _c(z["t"])
    gold = _c(z["out"])[:, 0]
    if taps:
        ref, out, rep = _network_report(engine, sd, x, t, flags)
        assert (ref - gold).abs().max() <= 1e-4 * gold.abs().max()       # oracle == reference fixture
        worst = max(r for _, r in rep)
        msg = " ".join(f"{i}:{r:.1e}" for i, r in rep)
        assert worst <= 2.5e-2, msg                                      # every module output, bf16 vs fp32 oracle
    else:
        fwd = lambda: engine.forward(x[:, 0].to(DEV), x[:, 1].to(DEV), t.to(DEV), mode=0, flags=flags).cpu()  # noqa: E731
        out = fwd()
        msg = run
        if pdl is not None:
            lib = _lib.load()
            prev = lib.snrse_set_pdl(pdl)
            try:
                out_pdl = fwd()
            finally:
                lib.snrse_set_pdl(prev)
            assert torch.equal(torch.view_as_real(out_pdl), torch.view_as_real(out)), msg
    assert rel_l2(torch.view_as_real(out), torch.view_as_real(gold)) <= 2e-2, msg


def test_ncsnpp_batch_and_length_independence_tcgen05(engine, sd):
    # per-sample normalisation / attention: item b of a batch == the same item run alone; T=128 bucket
    g = torch.Generator().manual_seed(11)
    x = torch.view_as_complex(torch.randn(2, 2, 256, 128, 2, generator=g) * 0.3)
    t = torch.tensor([0.5, 0.05])
    both = engine.forward(x[:, 0].to(DEV), x[:, 1].to(DEV), t.to(DEV), mode=1)
    one = engine.forward(x[1:, 0].to(DEV), x[1:, 1].to(DEV), t[1:].to(DEV), mode=1)
    assert torch.equal(both[1:], one)                                 # deterministic kernels: bit-exact
    with torch.no_grad():
        ref = o_sampler.score_forward(sd, x[:, :1], t[:, None, None, None], x[:, 1:], "sebridge_v3")
    assert rel_l2(torch.view_as_real(both.cpu()), torch.view_as_real(ref[:, 0])) <= 2e-2
