"""Keyed noise on the host: the Philox4x32-10 stream of include/snrse_b200.h in numpy (the reference the GPU test
compares the kernel with), and the key plumbing of the sweep and the file loop, which must hand every utterance its own
key whatever the batching or the rank count."""
import hashlib
import os

import numpy as np
import pytest
import torch

M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85


def philox4x32_10(c, k):
    """Philox4x32-10 on uint32 arrays: c [4, ...] counters, k [2, ...] keys (broadcast) -> [4, ...]."""
    c = [np.asarray(v, dtype=np.uint64) for v in c]
    k = [np.asarray(v, dtype=np.uint64) for v in k]
    mask = np.uint64(0xFFFFFFFF)
    for r in range(10):
        p0, p1 = np.uint64(M0) * c[0], np.uint64(M1) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k[0], p1 & mask, (p0 >> np.uint64(32)) ^ c[3] ^ k[1], p0 & mask]
        k = [(k[0] + np.uint64(W0)) & mask, (k[1] + np.uint64(W1)) & mask]
    return [v.astype(np.uint32) for v in c]


def keyed_noise(key, seed, idx):
    """Keyed draw z[i] (complex128, evaluated in float64) of the item with 64-bit `key` for element indices `idx`.
    Returns (z, r) with r = |z| in float64."""
    key, seed = int(key) % (1 << 64), int(seed) % (1 << 64)
    idx = np.asarray(idx, dtype=np.int64)
    lo, hi = lambda v: v & 0xFFFFFFFF, lambda v: v >> 32  # noqa: E731
    x = philox4x32_10([idx >> 1, np.zeros_like(idx), np.full_like(idx, lo(key)), np.full_like(idx, hi(key))],
                      [lo(seed), hi(seed)])
    odd = (idx & 1).astype(bool)
    xa, xb = np.where(odd, x[2], x[0]), np.where(odd, x[3], x[1])
    u1 = ((xa >> 8).astype(np.float64) + 1.0) * 2.0 ** -24
    u2 = (xb >> 8).astype(np.float64) * 2.0 ** -24
    r = np.sqrt(-np.log(u1))
    return r * np.cos(2 * np.pi * u2) + 1j * r * np.sin(2 * np.pi * u2), r


@pytest.mark.parametrize("counter,key,out", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(counter, key, out):
    assert tuple(int(v) for v in philox4x32_10(counter, key)) == out


def test_keyed_noise_reference_is_unit_complex_normal():
    z, _ = keyed_noise(12345, 7, np.arange(1 << 16))
    assert abs(np.mean(np.abs(z) ** 2) - 1) < 5 * 1 / np.sqrt(1 << 16)
    assert abs(np.mean(z.real)) < 5 * np.sqrt(0.5 / (1 << 16))


def test_key_tensor_wraps_unsigned_keys():
    from snr_aligned_diffse_b200.ops import key_tensor
    kt = key_tensor([0, 1, (1 << 64) - 1, 1 << 63, -5])
    assert kt.dtype == torch.int64 and kt.tolist() == [0, 1, -1, -(1 << 63), -5]
    with pytest.raises(ValueError):
        key_tensor([1 << 64])
    with pytest.raises(ValueError):
        key_tensor([1, 2], B=3)
    with pytest.raises(ValueError):
        key_tensor(torch.zeros(2))


def _waves(lens):
    # utterance i is the constant i + 1, so a fake enhance_fn can tell which utterance sits in each row
    return [torch.full((n,), float(i + 1)) for i, n in enumerate(lens)]


LENS = [5000, 9000, 8100, 16500, 8000, 5100, 23000, 300, 40000, 8191]


@pytest.mark.parametrize("world,max_batch,tf", [(1, 1, None), (1, 3, None), (2, 3, None), (1, 16, None), (2, 16, None),
                                                (1, 1, 300), (2, 1, 160)])
@pytest.mark.parametrize("keys", [None, [(1 << 64) - 1 - 3 * i for i in range(len(LENS))]])
def test_sweep_hands_every_utterance_its_key(world, max_batch, tf, keys):
    from snr_aligned_diffse_b200.sweep import enhance_sweep
    got, seeds = {}, set()

    def fn(y, n, k, s):
        assert k.dtype == torch.int64 and k.shape == (y.shape[0],)
        seeds.add(s)
        for r in range(y.shape[0]):
            got.setdefault(int(y[r, 0]) - 1, []).append(int(k[r]))
        return y

    waves = _waves(LENS)
    for rank in range(world):
        r = enhance_sweep(fn, waves, rank=rank, world=world, max_batch=max_batch, target_frames=tf, keep_audio=True,
                          seed=(1 << 64) - 2)
        for i, a in r["audio"].items():
            assert torch.equal(a, waves[i])
    want = list(range(len(LENS))) if keys is None else [k - (1 << 64) for k in keys]
    if keys is not None:      # the default keys again, by passing them explicitly
        got_default = dict(got)
        got.clear()
        for rank in range(world):
            enhance_sweep(fn, waves, rank=rank, world=world, max_batch=max_batch, target_frames=tf, seed=(1 << 64) - 2,
                          keys=keys)
        assert got_default == {i: [i] for i in range(len(LENS))}
    assert got == {i: [want[i]] for i in range(len(LENS))}
    assert seeds == {(1 << 64) - 2}


def test_sweep_without_seed_calls_two_argument_enhance_fn():
    from snr_aligned_diffse_b200.sweep import enhance_sweep
    r = enhance_sweep(lambda y, n: y, _waves(LENS[:3]), keep_audio=True)
    assert sorted(r["audio"]) == [0, 1, 2]
    with pytest.raises(ValueError):
        enhance_sweep(lambda y, n: y, _waves(LENS[:3]), keys=[1, 2, 3])


def test_file_keys_are_a_stable_hash_of_the_basename(tmp_path):
    from snr_aligned_diffse_b200 import wavio
    assert wavio.name_key("p232_001.wav") == int.from_bytes(
        hashlib.blake2b(b"p232_001.wav", digest_size=8).digest(), "little")
    assert wavio.name_key("p232_001.wav") == 0x912975D344AF26C6
    assert wavio.name_key("/some/dir/p232_001.wav") == wavio.name_key("p232_001.wav")
    assert wavio.name_key("ü.wav") == int.from_bytes(hashlib.blake2b("ü.wav".encode(), digest_size=8).digest(), "little")

    names = [f"f{i:02d}.wav" for i in range(7)]
    g = torch.Generator().manual_seed(3)
    paths = []
    for i, nm in enumerate(names):
        p = os.path.join(tmp_path, "in", nm)
        wavio.write_wav(p, torch.rand(1000 + 700 * i, generator=g) * 0.5)
        paths.append(p)

    def run(order, world):
        got = {}

        def fn(y, n, k, s):
            for r in range(y.shape[0]):
                got[int(n[r])] = (int(k[r]), s)
            return y
        for rank in range(world):
            wavio.enhance_files(fn, [paths[i] for i in order], os.path.join(tmp_path, "out"), rank=rank, world=world,
                                max_batch=2, seed=5)
        return got

    a = run(range(7), 1)
    b = run([6, 2, 4, 0, 1, 5, 3], 2)
    c = run([3, 5], 1)
    assert a == b and len(a) == 7
    want = {1000 + 700 * i: (wavio.name_key(nm) - (1 << 64) if wavio.name_key(nm) >= 1 << 63 else wavio.name_key(nm), 5)
            for i, nm in enumerate(names)}
    assert a == want and all(c[n] == a[n] for n in c)
