#!/usr/bin/env python
"""Keyed noise against generator noise, in one process.  python tools/keyed_bench.py

- kernel: X_T = Y + d*Z at 16 x 256 x 512 (the bench shape; 17 MB per operand, L2-resident) and 64 x 256 x 7552
  (64 x 60 s; 990 MB per operand, HBM): `lincomb_keyed` (reads Y, writes X_T: 16 B per element) against
  `randn_like` + `lincomb` (writes Z, reads Y and Z, writes X_T: 32 B per element).  Rates are algorithmic bytes over
  time, next to the rate of a device-to-device copy of the 64 x 256 x 7552 operand (same 16 B per element) measured in
  the same process.
- step: the graphed 16 x 4 s enhancement step (`GraphedEnhancer`, SNR estimator in the loop), keyed against a CUDA
  generator, the timing windows alternating.
- sweep: the 824-utterance sweep (`workloads.run_sweep824`'s utterances and batching, one graph per batch shape,
  captured in an untimed pass), keyed against the default, passes alternating.

Each kernel variant is timed from a captured graph of 10 calls; windows of REPLAYS replays alternate over ROUNDS
rounds (median, min, max).  The card's name and power limit are printed with the numbers."""
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import BATCH, SECONDS, SR, build_models, synth_waves  # noqa: E402
from snr_aligned_diffse_b200 import _lib, ops  # noqa: E402
from snr_aligned_diffse_b200.pipeline import GraphedEnhancer, GraphedEnhancerCache  # noqa: E402
from snr_aligned_diffse_b200.shard import batch_shards, synthetic_lengths  # noqa: E402
from snr_aligned_diffse_b200.sweep import enhance_sweep  # noqa: E402
from snr_aligned_diffse_b200.workloads import SWEEP_TARGET_FRAMES, synth_wave  # noqa: E402

ROUNDS, REPLAYS, SEED = 7, 10, 20261022


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        name, power = [s.strip() for s in q.strip().split(",")]
        return dict(gpu=name, power_limit=power)
    except (OSError, ValueError, subprocess.SubprocessError):
        return dict(gpu=torch.cuda.get_device_name(), power_limit="not read")


def capture(fn, calls=10):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(calls):
            fn()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    return g


def window_ms(g, per):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(REPLAYS):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (per * REPLAYS)


def alternate(graphs, per):
    times = {k: [] for k in graphs}
    names = list(graphs)
    for r in range(ROUNDS):
        for k in (names if r % 2 == 0 else names[::-1]):
            times[k].append(window_ms(graphs[k], per))
    return {k: dict(ms=round(statistics.median(t), 4), ms_min=round(min(t), 4), ms_max=round(max(t), 4))
            for k, t in times.items()}


def copy_rate_GBps():
    a = torch.randn(64, 256, 7552, dtype=torch.complex64, device="cuda")     # 990 MB
    b = torch.empty_like(a)
    g = capture(lambda: b.copy_(a), calls=5)
    ms = statistics.median(window_ms(g, 5) for _ in range(5))
    return 16 * a.numel() / (ms * 1e-3) / 1e9


def kernel_case(B, T, copy_GBps):
    gen = torch.Generator(device="cuda").manual_seed(1)
    Y = torch.randn(B, 256, T, dtype=torch.complex64, device="cuda", generator=gen)
    one = torch.ones(B, device="cuda")
    d = torch.rand(B, device="cuda", generator=gen)
    keys = torch.arange(B, dtype=torch.int64, device="cuda")
    graphs = {
        "keyed": capture(lambda: ops.lincomb_keyed(y=Y, b=one, d=d, keys=keys, seed=SEED, want_mean=False)),
        "randn_like+lincomb": capture(lambda: ops.lincomb(y=Y, z=torch.randn_like(Y), b=one, d=d,
                                                          want_mean=False)),
    }
    res = alternate(graphs, 10)
    n = Y.numel()
    for k, by in (("keyed", 16 * n), ("randn_like+lincomb", 32 * n)):
        res[k]["algorithmic_MB"] = round(by / 1e6, 1)
        res[k]["GBps"] = round(by / (res[k]["ms"] * 1e-3) / 1e9, 1)
        res[k]["frac_of_copy_rate"] = round(res[k]["GBps"] / copy_GBps, 3)
    res["keyed_over_baseline_time"] = round(res["keyed"]["ms"] / res["randn_like+lincomb"]["ms"], 3)
    del Y
    return dict(shape=[B, 256, T], **res)


def step_case(model, dev):
    L = int(SECONDS * SR)
    y = synth_waves(BATCH, L, seed=1000)
    pipes = {"keyed": GraphedEnhancer(model, BATCH, L, dev, oracle=False, keyed=True, seed=SEED),
             "generator": GraphedEnhancer(model, BATCH, L, dev, oracle=False,
                                          generator=torch.Generator(device=dev).manual_seed(100))}
    for p in pipes.values():
        p.y_dev.copy_(y)
        torch.cuda.synchronize()
        p.capture(warmup=1)
        p.stream.synchronize()
    graphs = {k: p.graph for k, p in pipes.items()}
    res = alternate(graphs, 1)
    out = pipes["keyed"].replay()
    torch.cuda.synchronize()
    eager = model.enhance_batch(y, oracle=False, keys=torch.arange(BATCH), seed=SEED)
    res["keyed_replay_equals_eager"] = bool(torch.equal(out, eager))
    res["keyed_over_generator_time"] = round(res["keyed"]["ms"] / res["generator"]["ms"], 4)
    return dict(shape=[BATCH, L], **res)


def sweep_case(model, dev, passes=3):
    lengths = synthetic_lengths(824, seed=0)
    waves = [synth_wave(int(n), seed=i) for i, n in enumerate(lengths)]
    mine = batch_shards([int(n) for n in lengths], 1, 16, target_frames=SWEEP_TARGET_FRAMES)[0]
    model.dnn.engine.reserve(max(model.dnn.engine.workspace_bytes(len(ix), 256, tp) for tp, ix in mine))
    fns = {"default": GraphedEnhancerCache(model, dev, min_uses=1, oracle=False),
           "keyed": GraphedEnhancerCache(model, dev, min_uses=1, oracle=False)}
    seeds = {"default": None, "keyed": SEED}
    run = lambda k: enhance_sweep(fns[k], waves, device=dev, max_batch=16, target_frames=SWEEP_TARGET_FRAMES,  # noqa: E731
                                  seed=seeds[k])
    for k in fns:
        run(k)                                   # captures every batch shape
    times = {k: [] for k in fns}
    names = list(fns)
    for r in range(passes):
        for k in (names if r % 2 == 0 else names[::-1]):
            times[k].append(run(k)["seconds"])
    audio = float(sum(int(n) for n in lengths)) / SR
    res = {k: dict(seconds=round(statistics.median(t), 4), seconds_min=round(min(t), 4), seconds_max=round(max(t), 4),
                   audio_s_per_s=round(audio / statistics.median(t), 1)) for k, t in times.items()}
    res["keyed_over_default_time"] = round(res["keyed"]["seconds"] / res["default"]["seconds"], 4)
    return dict(utterances=len(waves), batches=len(mine), audio_seconds=round(audio, 1), **res)


def main():
    _lib.load()
    _lib.require_device()
    dev = torch.device("cuda", 0)
    result = card()
    rate = copy_rate_GBps()
    result["copy_GBps"] = round(rate, 1)
    result["kernel"] = [kernel_case(16, 512, rate), kernel_case(64, 7552, rate)]
    torch.cuda.empty_cache()
    model, _ = build_models(dev)
    result["step"] = step_case(model, dev)
    result["sweep824"] = sweep_case(model, dev)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
