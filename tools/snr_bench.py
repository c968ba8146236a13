#!/usr/bin/env python
"""SNR estimator (SNRNet) forward timings.  python tools/snr_bench.py

- bench: the bench shape (16 x 4 s: 16 x 2 x 256 x 512 planar features) through `snrse_snrnet_forward` (dense) and
  through `snrse_snrnet_forward_varlen` with every item at its full 32 clusters (varlen_full).
- ragged: 16 utterances of the most populated Tpad bucket of the synthetic 824-utterance sweep
  (`shard.synthetic_lengths`), in the sweep's buffer (128 * Tpad - 1 samples), through the dense entry point (every item
  over all Tpad/16 clusters) and through the varlen one (each item over its own clusters).

Each variant is timed as ms per forward from a captured graph of 10 forwards; the variants of a case are captured once
and their timing windows alternate over ROUNDS rounds (median, min, max reported).  The inputs and workspaces (about
120 MB at the bench shape) are not flushed from L2 between forwards, as in the bench loop.  The card's name and power
limit are printed with the numbers; the per-kernel split of the bench shape comes from torch's profiler in a separate
pass."""
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from snr_aligned_diffse_b200 import ops, shard  # noqa: E402
from snr_aligned_diffse_b200.synth import synth_state_dict  # noqa: E402

ROUNDS, REPLAYS = 7, 20


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        name, power = [s.strip() for s in q.strip().split(",")]
        return dict(gpu=name, power_limit=power)
    except (OSError, ValueError, subprocess.SubprocessError):
        return dict(gpu=torch.cuda.get_device_name(), power_limit="not read")


def capture(fn):
    for _ in range(3):
        out = fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(10):
            out = fn()
    for _ in range(5):
        g.replay()
    return g, out


def window_ms(g):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(REPLAYS):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (10 * REPLAYS)


def compare(variants):
    """variants: name -> fn.  Returns name -> dict(ms median/min/max, finite), timing windows interleaved."""
    graphs = {k: capture(fn) for k, fn in variants.items()}
    times = {k: [] for k in variants}
    names = list(variants)
    for r in range(ROUNDS):
        for k in (names if r % 2 == 0 else names[::-1]):
            times[k].append(window_ms(graphs[k][0]))
    return {k: dict(ms_per_forward=round(statistics.median(t), 4), ms_min=round(min(t), 4), ms_max=round(max(t), 4),
                    finite=bool(torch.isfinite(graphs[k][1]).all())) for k, t in times.items()}


net = ops.SNRNetEngine()
net.load_state_dict(synth_state_dict(net.param_shapes(), seed=1), "cuda")
result = card()

feat = torch.randn(16, 2, 256, 512, generator=torch.Generator().manual_seed(0)).cuda()
full = torch.full((16,), 512 // 16, dtype=torch.int32, device="cuda")
bench = compare({"dense": lambda: net.forward(feat), "varlen_full": lambda: net.forward(feat, full)})
bench["bits_equal"] = bool(torch.equal(net.forward(feat), net.forward(feat, full)))
result["bench"] = dict(shape=[16, 2, 256, 512], **bench)

lengths = shard.synthetic_lengths()
buckets = {}
for n in lengths:
    buckets.setdefault(shard.tpad_of(n), []).append(int(n))
tpad = max(buckets, key=lambda t: len(buckets[t]))
lens = torch.tensor(buckets[tpad][:16], dtype=torch.int32, device="cuda")
T16 = ops.padded_frames(shard.HOP * tpad - 1, 16)
clusters = (lens // shard.HOP + 16) // 16
feat_r = torch.randn(len(lens), 2, 256, T16, generator=torch.Generator().manual_seed(1)).cuda()
ragged = compare({"dense": lambda: net.forward(feat_r), "varlen": lambda: net.forward(feat_r, clusters)})
result["ragged"] = dict(shape=list(feat_r.shape), tpad=tpad, lengths=lens.tolist(), clusters=clusters.tolist(),
                        valid_cluster_share=round(float(clusters.sum()) / (len(lens) * T16 // 16), 4), **ragged)

with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    for _ in range(5):
        net.forward(feat)
    torch.cuda.synchronize()
result["bench"]["kernels_us"] = {e.key.split("::")[-1][:28]: round(e.device_time_total / 5, 1)
                                 for e in prof.key_averages() if "snr_" in e.key}
print(json.dumps(result))
