#!/usr/bin/env python
"""A/B of programmatic-dependent-launch masks (snrse_set_pdl) on the REAL step: one captured CUDA graph of the full
16 x 4 s sebridge_v3 pass per variant (own model, own activation arena), replayed back to back; the variants are
interleaved round-robin so that thermal / power drift hits them equally.  Usage: python tools/step_ab.py [mask ...]
(default: 2 0, the library default against plain stream-ordered launches)"""
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from snr_aligned_diffse_b200.pipeline import GraphedEnhancer  # noqa: E402

from snr_aligned_diffse_b200 import _lib  # noqa: E402
# the mask is read when the graph is captured
variants = sys.argv[1:] or ["2", "0"]
dev = torch.device("cuda", 0)
torch.cuda.set_device(0)
L = int(bench.SECONDS * bench.SR)
y = bench.synth_waves(bench.BATCH, L, seed=1000).to(dev)
pipes = []
for i, v in enumerate(variants):
    _lib.load().snrse_set_pdl(int(v))
    model, _ = bench.build_models(dev, with_estimator=(i == 0))
    model.dnn._ensure_device_weights()
    p = GraphedEnhancer(model, bench.BATCH, L, dev, oracle=False)
    p.y_dev.copy_(y)
    p.capture(warmup=2)
    pipes.append(p)
torch.cuda.synchronize()
for p in pipes:
    for _ in range(10):
        p.replay()
torch.cuda.synchronize()
tot = {v: [] for v in variants}
for rnd in range(6):
    for v, p in zip(variants, pipes):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(p.stream):
            e0.record(p.stream)
            for _ in range(25):
                p.graph.replay()
            e1.record(p.stream)
        torch.cuda.synchronize()
        tot[v].append(e0.elapsed_time(e1) / 25)
print(json.dumps({v: dict(ms_per_step_rounds=[round(ms, 3) for ms in tot[v]], median=round(sorted(tot[v])[len(tot[v]) // 2], 3))
                  for v in variants}))
