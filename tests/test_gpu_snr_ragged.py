"""SNR estimation per utterance on ragged batches (`SNRModel.estimate_batch`, `snrse_snrnet_forward_varlen`).

`enhance` estimates one file at a time: its features are padded to its own multiple of 16 frames and SNRNet runs over
those clusters only (model.py:715-721).  In a padded batch every item shares one buffer of T16 frames; these tests check
that each item is still estimated over its own clusters: against the CPU oracle on the item alone, bit for bit against
the same item in other batches, with the frames and workspace rows past its clusters poisoned, through a CUDA graph, and
with out-of-range cluster counts inside guard bands.
"""
import numpy as np
import pytest
import torch

from oracle import snrnet as o_snrnet
from oracle.topology import snrnet_param_specs
from snr_aligned_diffse_b200.synth import synth_state_dict, synth_waves

pytestmark = pytest.mark.gpu

L = 24575                                          # 192 frames: T16 = 192, S = 12 clusters
LENS = [24447, 20480, 18000, 16500, 2047, 2048]    # 191, 161, 141, 129, 16, 17 frames
CLUSTERS = [12, 11, 9, 9, 1, 2]
ONE = LENS.index(2047)                             # one 16-frame cluster: NaN in the reference (unbiased std of one value)


def bits(t):
    return t.detach().float().contiguous().view(torch.int32).cpu()


def ragged(lens, length, seed):
    """Synthetic speech in the first lens[b] samples, loud noise after them (it must not reach any estimate)."""
    y = synth_waves(len(lens), length, seed=seed)
    g = torch.Generator().manual_seed(seed + 100)
    for b, n in enumerate(lens):
        y[b, n:] = 3.0 * torch.randn(length - n, generator=g)
    return y


@pytest.fixture(scope="module")
def snr_sd():
    return synth_state_dict(snrnet_param_specs(), seed=1)


@pytest.fixture(scope="module")
def est(snr_sd):
    from snr_aligned_diffse_b200.sgmse.snr_estimator import SNRModel
    m = SNRModel(base_dir="")
    m._error_loading_ema = True
    m.load_state_dict(snr_sd)
    return m.eval(no_ema=True)


@pytest.fixture(scope="module")
def y():
    return ragged(LENS, L, seed=5)


@pytest.fixture(scope="module")
def net(snr_sd):
    from snr_aligned_diffse_b200 import ops
    return ops.SNRNetEngine().load_state_dict(snr_sd, "cuda")


def forward_abi(net, feat, clusters, ws_fill=None):
    """One snrse_snrnet_forward(_varlen) call with a caller-owned workspace, optionally filled with a byte pattern."""
    from snr_aligned_diffse_b200 import _lib
    B, _, _, T16 = feat.shape
    ws = torch.empty(int(net.lib.snrse_snrnet_workspace_bytes(B, T16)), dtype=torch.uint8, device="cuda")
    if ws_fill is not None:
        ws.fill_(ws_fill)
    out = torch.empty(B, dtype=torch.float32, device="cuda")
    if clusters is None:
        rc = net.lib.snrse_snrnet_forward(_lib.ptr(net.blob), _lib.ptr(feat), _lib.ptr(out), B, T16, _lib.ptr(ws),
                                          _lib.stream_ptr())
    else:
        rc = net.lib.snrse_snrnet_forward_varlen(_lib.ptr(net.blob), _lib.ptr(feat), _lib.ptr(clusters), _lib.ptr(out),
                                                 B, T16, _lib.ptr(ws), _lib.stream_ptr())
    _lib.check(rc, "snrnet_forward")
    return out


@pytest.mark.filterwarnings("ignore:std")     # torch warns about the single-cluster item, exercised on purpose
def test_matches_oracle_per_utterance(est, snr_sd, y):
    ratio, aux = est.estimate_batch(y, torch.tensor(LENS, dtype=torch.int32), return_aux=True)
    assert ratio.is_cuda and ratio.dtype == torch.float32 and ratio.shape == (len(LENS),)
    assert aux["clusters"].tolist() == CLUSTERS
    assert aux["g"].shape == ratio.shape and aux["clusters"].dtype == torch.int32
    for b, n in enumerate(LENS):
        ref = float(o_snrnet.estimate_noise_over_clean(snr_sd, y[b:b + 1, :n])[0, 0])
        got = float(ratio[b])
        if b == ONE:
            assert np.isnan(ref) and np.isnan(got)
        else:
            assert abs(got / ref - 1) <= 1e-4, (n, got, ref)


def test_item_bits_do_not_depend_on_the_batch(est, y):
    lens = torch.tensor(LENS, dtype=torch.int32)
    in_batch = bits(est.estimate_batch(y, lens))
    # alone, at the utterance's own length (lengths=None)
    for b, n in enumerate(LENS):
        assert torch.equal(bits(est.estimate_batch(y[b:b + 1, :n]))[0], in_batch[b]), n
    # reversed, between other utterances, in a longer buffer (T16 = 320) with different samples past each length
    L2 = 40000
    others = ragged([39000, 5000, 30001], L2, seed=9)
    rows, lens2, where = [], [], {}
    for b in reversed(range(len(LENS))):
        row = 3.0 * torch.randn(L2, generator=torch.Generator().manual_seed(b))
        row[:LENS[b]] = y[b, :LENS[b]]
        where[b] = len(rows)
        rows.append(row)
        lens2.append(LENS[b])
        if b % 2 == 0:
            rows.append(others[b // 2])
            lens2.append([39000, 5000, 30001][b // 2])
    out2 = bits(est.estimate_batch(torch.stack(rows), torch.tensor(lens2, dtype=torch.int32, device="cuda")))
    for b in range(len(LENS)):
        assert torch.equal(out2[where[b]], in_batch[b]), LENS[b]


def test_frames_and_workspace_past_the_clusters_are_never_read(net, y):
    from snr_aligned_diffse_b200 import ops
    yd = y.cuda()
    ld = torch.tensor(LENS, dtype=torch.int32, device="cuda")
    feat = ops.stft(yd, ld, scale=ops.absmax(yd, ld), transform=False, planar=True, pad_multiple=16)
    cl = torch.tensor(CLUSTERS, dtype=torch.int32, device="cuda")
    ref = forward_abi(net, feat, cl, ws_fill=0)
    poisoned = feat.clone()
    for b, s in enumerate(CLUSTERS):
        poisoned[b, :, :, 16 * s:] = float("nan")
    got = forward_abi(net, poisoned, cl, ws_fill=0xFF)          # every workspace float starts as NaN
    assert torch.equal(bits(got), bits(ref))
    finite = torch.isfinite(got.cpu())
    assert finite.sum() == len(CLUSTERS) - 1 and not finite[ONE]


@pytest.mark.parametrize("B,T16", [(16, 512), (3, 96)])
def test_full_clusters_give_the_dense_bits(net, B, T16):
    feat = torch.randn(B, 2, 256, T16, generator=torch.Generator().manual_seed(T16)).cuda()
    dense = forward_abi(net, feat, None)
    full = torch.full((B,), T16 // 16, dtype=torch.int32, device="cuda")
    assert torch.isfinite(dense).all()
    assert torch.equal(bits(forward_abi(net, feat, full)), bits(dense))
    assert torch.equal(bits(net.forward(feat)), bits(dense))
    assert torch.equal(bits(net.forward(feat, full)), bits(dense))


def test_cuda_graph_replay_equals_eager(est, y):
    y_dev = y.cuda()
    len_dev = torch.tensor(LENS, dtype=torch.int32, device="cuda")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        est.estimate_batch(y_dev, len_dev)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = est.estimate_batch(y_dev, len_dev)
    lens2 = [20000, 24575, 3000, 2048, 17001, 9000]
    y2 = ragged(lens2, L, seed=11)
    y_dev.copy_(y2)
    len_dev.copy_(torch.tensor(lens2, dtype=torch.int32))
    graph.replay()
    torch.cuda.synchronize()
    eager = est.estimate_batch(y2, torch.tensor(lens2, dtype=torch.int32))
    assert torch.isfinite(eager).all()
    assert torch.equal(bits(out), bits(eager))


class GuardedAllocator:
    """torch.empty / empty_like on CUDA with 64 KB of 0xA5 on either side of every buffer."""
    PAD = 65536

    def __init__(self):
        self._empty, self._empty_like = torch.empty, torch.empty_like
        self.live = []

    def empty(self, *size, dtype=None, device=None, **kw):
        if len(size) == 1 and isinstance(size[0], (tuple, list, torch.Size)):
            size = tuple(size[0])
        dev = torch.device(device) if device is not None else None
        if dev is None or dev.type != "cuda" or kw.get("pin_memory"):
            return self._empty(*size, dtype=dtype, device=device, **kw)
        dtype = dtype or torch.get_default_dtype()
        n = int(np.prod(size)) * self._empty((), dtype=dtype).element_size()
        raw = self._empty(n + 2 * self.PAD, dtype=torch.uint8, device=dev)
        raw.fill_(0xA5)
        self.live.append((raw, n))
        return raw[self.PAD:self.PAD + n].view(dtype).view(*size)

    def empty_like(self, x, **kw):
        if not x.is_cuda:
            return self._empty_like(x, **kw)
        return self.empty(*x.shape, dtype=kw.get("dtype", x.dtype), device=x.device)

    def check(self):
        torch.cuda.synchronize()
        for raw, n in self.live:
            assert bool((raw[:self.PAD] == 0xA5).all()) and bool((raw[self.PAD + n:] == 0xA5).all()), \
                f"guard band of a {n}-byte buffer was overwritten"
        return len(self.live)


@pytest.fixture
def guard(monkeypatch):
    g = GuardedAllocator()
    monkeypatch.setattr(torch, "empty", g.empty)
    monkeypatch.setattr(torch, "empty_like", g.empty_like)
    return g


def test_out_of_range_clusters_are_clamped_inside_their_buffers(net, guard):
    B, T16 = 6, 96                                               # S = 6
    feat = guard.empty(B, 2, 256, T16, dtype=torch.float32, device="cuda")
    feat.copy_(torch.randn(B, 2, 256, T16, generator=torch.Generator().manual_seed(2)))
    bad = guard.empty(B, dtype=torch.int32, device="cuda")
    bad.copy_(torch.tensor([0, 11, 3, -7, 6, 1 << 30], dtype=torch.int32))   # 0, S+5, valid, negative, S, huge
    got = net.forward(feat, bad)
    assert guard.check() >= 4                                    # feat, clusters, workspace, out
    clamped = torch.tensor([1, 6, 3, 1, 6, 6], dtype=torch.int32, device="cuda")
    assert torch.equal(bits(got), bits(net.forward(feat, clamped)))
    assert torch.equal(bits(got)[[1, 4, 5]], bits(net.forward(feat))[[1, 4, 5]])
    assert guard.check() >= 8


def test_lengths_on_the_host_are_checked(est, y):
    for lens in ([0] + LENS[1:], LENS[:-1] + [L + 1], LENS[:-1]):
        with pytest.raises(ValueError):
            est.estimate_batch(y, torch.tensor(lens, dtype=torch.int32))
    with pytest.raises(ValueError):
        est.estimate_batch(y, torch.tensor(LENS, dtype=torch.float32))
