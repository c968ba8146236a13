"""Every convolution plan the NCSN++ executor can choose, enumerated on the host (no GPU).

snrse_ncsnpp_dbg_convs records the executor's plan for (B, F, T) without a device and reports every convolution it
records (operand views, operand combination, and the plan fields conv_halo2_make_plan / conv_gemm_make_plan_ex choose)
for a given SM count.  Over the product's range (B = 1..64 utterances per bucket, Tpad = 64..7552 frames) the rows fall
into a few hundred classes: configurations of the kernels that can run in production.  tests/test_gpu_conv_plans.py runs
the cheapest instance of every class against fp64; this module defines the classes and checks the dump against the
topology it comes from.
"""
import collections

import numpy as np
import pytest

F_BINS = 256
B_RANGE = range(1, 65)                 # shard.bucket_batches: up to 64 utterances per batch
T_RANGE = range(64, 7552 + 1, 64)      # Tpad: multiples of 64 up to 60 s
NUM_SMS_B200 = 148

PATH_NAMES = {(0, 0): "2-CTA", (0, 1): "2-CTA out4", (2, 0): "GEMM", (1, 1): "CUDA-core out4", (1, 0): "CUDA cores"}


def class_key(r):
    """The configuration a row runs: two rows with equal keys take the same code path through their kernel."""
    path, out4 = int(r["path"]), int(r["out4"])
    common = (
        path, out4,
        int(r["c0"]) // 64,            # operand channel chunks (K loop length, shortcut interleave pattern)
        int(r["c1"]) // 64,            # 1x1 shortcut chunks, 0: no shortcut
        int(r["taps"]),                # 3x3 or 1x1
        int(r["n"]),                   # output channels
        int(r["norm"]),                # GroupNorm + SiLU of the operand in flight
        int(r["res"]),                 # identity residual in the epilogue
        int(r["tbias"]),               # time-embedding bias (per image, row stride = the executor's row count)
        int(r["bias"]),                # bias
        int(r["stats"]),               # epilogue GroupNorm sums
        int(r["addend"]),              # out4: the up-sampled pyramid is added
    )
    if path == 0:
        n_ctiles = (int(r["n_tiles"]) + 1) // 2
        clusters = n_ctiles if int(r["nsplit"]) == 2 else int(r["grid"]) // 2
        return common + (
            int(r["sub"]),             # sub-tiles per super-tile (1 or 2)
            int(r["nsplit"]),          # N split over two clusters
            int(r["n_loc"]),           # output channels per cluster
            int(r["acc_bufs"]),        # TMEM accumulator sets
            int(r["na"]),              # halo ring depth
            int(r["nb"]),              # weight ring depth
            int(r["stg_bufs"]),        # epilogue staging tiles per warp
            int(r["nsc"]),             # separate shortcut ring slots, 0: shared ring
            int(n_ctiles > clusters),                          # persistent: a cluster walks several tiles
            int(n_ctiles % clusters != 0),                     # uneven walk: some clusters walk one tile fewer
            int(r["n_tiles"]) % 2,                             # odd tile count: the last peer CTA runs an all-padding tile
            int(int(r["H"]) % (16 * int(r["sub"])) != 0),      # ragged last tile row
            int(int(r["W"]) % 8 != 0),                         # ragged last tile column
            int(int(r["n_tiles"]) > 2 * clusters and int(r["B"]) > 1),   # a cluster's walk crosses images
        )
    if path == 2:
        return common + (
            int(r["th"]), int(r["tw"]),                        # pixel tile shape th x tw = 128
            int(r["n_tile"]),                                  # output channels per CTA
            int(r["small"]),                                   # small-map mode (64-column tiles, deep ring)
            int(r["stages"]),                                  # ring depth
            int(int(r["H"]) % int(r["th"]) != 0),              # ragged tile rows (clipped by the tensor map)
            int(int(r["W"]) % int(r["tw"]) != 0),              # ragged tile columns
        )
    return common


def macs(r):
    return int(r["B"]) * int(r["H"]) * int(r["W"]) * int(r["n"]) * (int(r["taps"]) * int(r["c0"]) + int(r["c1"]))


def enumerate_classes(eng, num_sms, b_range=B_RANGE, t_range=T_RANGE):
    """{class key: (MACs, B, T, row)} with the cheapest instance (fewest MACs) of every class over b_range x t_range."""
    best = {}
    for B in b_range:
        for T in t_range:
            for r in eng.conv_rows(B, F_BINS, T, 0, num_sms):
                if int(r["path"]) == 1:
                    continue           # CUDA-core fallbacks of the output head below the 2-CTA tiles: not a plan
                k = class_key(r)
                m = macs(r)
                if k not in best or m < best[k][0]:
                    best[k] = (m, B, T, r.copy())
    return best


def test_plan_entry_points_are_exported():
    """include/snrse_b200_plans.h: every declaration exported and in _lib.PLAN_PROTOTYPES, none in another header."""
    import os
    import re
    from snr_aligned_diffse_b200 import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def found(f):
        return set(re.findall(r"\b(snrse_[a-z0-9_]+)\s*\(", open(os.path.join(root, "include", f)).read()))

    plans = found("snrse_b200_plans.h")
    assert plans == {"snrse_ncsnpp_dbg_convs", "snrse_dbg_conv_plan"} == set(_lib.PLAN_PROTOTYPES)
    assert not plans & (found("snrse_b200.h") | found("snrse_b200_debug.h") | found("snrse_b200_layers.h"))
    assert not plans & (set(_lib.PROTOTYPES) | set(_lib.LAYER_PROTOTYPES))
    lib = _lib.load()
    for name in plans:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"


@pytest.fixture(scope="module")
def eng():
    from snr_aligned_diffse_b200.engine import NCSNppEngine
    return NCSNppEngine()


@pytest.fixture(scope="module")
def classes(eng):
    return enumerate_classes(eng, NUM_SMS_B200)


def test_every_plan_dimension_is_reached(classes):
    """Over B = 1..64 x T = 64..7552 on a 148-SM B200 every plan dimension takes every value its make_plan can give
    it; prints the class count per path and the cost of each class's cheapest instance."""
    per_path = collections.Counter(PATH_NAMES[k[0], k[1]] for k in classes)
    print("classes per path:", dict(per_path), "total", len(classes))
    for path in sorted(per_path):
        ks = sorted((v[0], v[1], v[2], k) for k, v in classes.items() if PATH_NAMES[k[0], k[1]] == path)
        total = sum(m for m, *_ in ks)
        print(f"{path}: {len(ks)} classes, cheapest instances {total:.3g} MAC in all "
              f"(min {ks[0][0]:.3g}, max {ks[-1][0]:.3g})")
        for m, B, T, k in ks:
            print(f"  B={B:2d} T={T:4d} {m:10.3g} MAC  {k}")
    assert all(m > 0 for m, *_ in classes.values())
    halo = [v[3] for k, v in classes.items() if k[0] == 0 and not k[1]]
    out4 = [v[3] for k, v in classes.items() if k[0] == 0 and k[1]]
    gemm = [v[3] for k, v in classes.items() if k[0] == 2]
    assert halo and out4 and gemm

    def values(rows, f):
        return {int(r[f]) for r in rows}

    assert values(halo, "sub") == {1, 2} and values(halo, "nsplit") == {1, 2} and values(halo, "acc_bufs") == {1, 2}
    assert values(halo, "n_loc") == {128, 256} and values(halo, "nsc") == {0, 2} and values(halo, "stg_bufs") == {1, 2}
    assert len(values(halo, "na")) >= 2 and len(values(halo, "nb")) >= 2
    assert values(out4, "sub") == {1, 2} and values(out4, "norm") == {1} and values(out4, "addend") == {1}
    hk = [k for k in classes if k[0] == 0]
    for i, what in ((-6, "persistent walk"), (-5, "uneven walk"), (-4, "odd tile count"), (-3, "ragged H"),
                    (-2, "ragged W"), (-1, "walk across images")):
        assert {k[i] for k in hk} == {0, 1}, what
    assert values(gemm, "small") == {0, 1} and values(gemm, "taps") == {1, 9} and len(values(gemm, "n_tile")) >= 2
    assert len({(int(r["th"]), int(r["tw"])) for r in gemm}) >= 3
    assert {(int(r["res"]), int(r["c1"]) > 0) for r in gemm} >= {(1, False), (0, True)}


def expected_convs(T, nf=128, ch_mult=(1, 1, 2, 2, 2, 2, 2), nrb=2, attn_res=16):
    """(level, taps, n_rows) of every convolution of the default NCSN++ (ncsnpp.py), from the network description."""
    L = len(ch_mult)
    convs = [(0, 9, nf)]                                   # conv_in
    attn = lambda lv: F_BINS >> lv == attn_res             # noqa: E731
    for lv in range(L):
        c = nf * ch_mult[lv]
        for _ in range(nrb):
            convs += [(lv, 9, c)] * 2
            if attn(lv):
                convs += [(lv, 1, 3 * c), (lv, 1, c)]
        if lv != L - 1:
            convs += [(lv + 1, 9, c)] * 2                  # down block: both convolutions on the halved map
    c = nf * ch_mult[-1]
    convs += [(L - 1, 9, c)] * 2 + [(L - 1, 1, 3 * c), (L - 1, 1, c)] + [(L - 1, 9, c)] * 2   # middle: res, attn, res
    for lv in reversed(range(L)):
        c = nf * ch_mult[lv]
        convs += [(lv, 9, c)] * (2 * (nrb + 1))
        if attn(lv):
            convs += [(lv, 1, 3 * c), (lv, 1, c)]
        convs += [(lv, 9, 4)]                              # output head
        if lv != 0:
            convs += [(lv - 1, 9, c)] * 2                  # up block
    return convs


@pytest.mark.parametrize("B,T", [(1, 64), (3, 192), (64, 7552), (17, 1216)])
def test_dump_matches_the_topology(eng, B, T):
    """The dump lists every convolution of the forward once, at the map size of its level, on the path the kernel
    choice gives it (2-CTA kernel: 3x3 with N in {128, 256} or the C -> 4 head on maps of at least 8 x 8; single-CTA
    GEMM: every other one; CUDA cores: the head below 8 x 8), with the operand combination the executor passes."""
    rows = eng.conv_rows(B, F_BINS, T)
    want = expected_convs(T)
    assert len(rows) == len(want) == 114
    counts = collections.Counter()
    for r, (lv, taps, n) in zip(rows, want):
        H, W = F_BINS >> lv, T >> lv
        assert (int(r["B"]), int(r["H"]), int(r["W"]), int(r["taps"]), int(r["n"])) == (B, H, W, taps, n)
        fits = H >= 8 and W >= 8
        path = (0 if fits else 1) if n == 4 else (0 if fits and taps == 9 else 2)
        assert (int(r["path"]), int(r["out4"])) == (path, int(n == 4))
        counts[PATH_NAMES[path, int(n == 4)]] += 1
        assert int(r["stats"]) == int(path == 0 and n != 4)
        assert int(r["off0"]) + int(r["c0"]) <= int(r["ld0"]) and int(r["off_out"]) + n <= int(r["ld_out"])
        if int(r["c1"]):
            assert int(r["off1"]) + int(r["c1"]) <= int(r["ld1"]) and not int(r["res"])
        if int(r["tbias"]):
            assert int(r["tb_stride"]) == 10880                # the rows of every block's Dense_0
        if path == 0:
            assert int(r["sub"]) in (1, 2) and int(r["grid"]) > 0 and int(r["smem_bytes"]) <= 227 * 1024
        elif path == 2:
            assert int(r["th"]) * int(r["tw"]) == 128 and int(r["grid"]) > 0
    levels_halo = sum(1 for lv in range(7) if (F_BINS >> lv) >= 8 and (T >> lv) >= 8)
    print(f"B={B} T={T}: {dict(counts)}; levels on the 2-CTA kernel: {levels_halo}")
    assert counts["2-CTA out4"] + counts["CUDA-core out4"] == 7 and counts["2-CTA out4"] == levels_halo
    # the first convolution is the input convolution on the 64-channel hi/lo operand, written as the skip half of the
    # last decoder concatenation (128 + 128 channels)
    r0 = rows[0]
    assert (int(r0["c0"]), int(r0["ld0"]), int(r0["off0"]), int(r0["ld_out"]), int(r0["off_out"])) == (64, 64, 0, 256, 128)
    assert not int(r0["norm"]) and int(r0["bias"]) and not int(r0["tbias"])


def test_dump_needs_no_device_and_caches_nothing(eng):
    """Dumping a plan records into a plan of its own: a later plan_bytes of the same (B,F,T) with other flags is
    unaffected, and the argument checks of snrse_ncsnpp_plan_bytes apply."""
    a = eng.conv_rows(2, F_BINS, 128, 0, 148)
    b = eng.conv_rows(2, F_BINS, 128, 0, 148)
    assert np.array_equal(a, b)
    c = eng.conv_rows(2, F_BINS, 128, 0, 16)                   # fewer SMs: bigger sub-tiles, no N split
    assert any(int(x["sub"]) != int(y["sub"]) or int(x["nsplit"]) != int(y["nsplit"]) for x, y in zip(a, c))
    with pytest.raises(RuntimeError, match="multiples"):
        eng.conv_rows(2, F_BINS, 96)
    with pytest.raises(RuntimeError, match="unknown flags"):
        eng.conv_rows(2, F_BINS, 128, 4)
