#!/usr/bin/env python
"""Per-kind time of one NCSN++ forward for a (B, T) bucket, measured with CUDA events between launch groups
(snrse_ncsnpp_profile_forward).  Usage: python tools/profile_shape.py B T [flags]   (0 default, 2 CUDA-core cross-check)"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from snr_aligned_diffse_b200.engine import NCSNppEngine  # noqa: E402
from snr_aligned_diffse_b200.synth import synth_state_dict  # noqa: E402

B, T = int(sys.argv[1]), int(sys.argv[2])
flags = int(sys.argv[3]) if len(sys.argv) > 3 else 0
if flags not in (0, 1, 2):
    sys.exit("flags: 0 (default), 1 (keep every activation) or 2 (CUDA-core cross-check)")
eng = NCSNppEngine()
eng.load_state_dict(synth_state_dict(eng.param_shapes(), seed=0), "cuda")
g = torch.Generator().manual_seed(0)
x = torch.view_as_complex(torch.randn(B, 256, T, 2, generator=g)).cuda()
y = torch.view_as_complex(torch.randn(B, 256, T, 2, generator=g)).cuda()
t = torch.full((B,), 0.5, device="cuda")
names = {0: "other", 1: "conv_tcgen05", 2: "groupnorm", 3: "fir", 4: "attention", 5: "thin_conv", 6: "pack_temb_head"}
# STEADY=n: n untimed profiled passes first (~25 ms each), so the table below is the power-capped steady state
for _ in range(3 + int(os.environ.get("STEADY", "0"))):
    prof = eng.profile_forward(x, y, t, mode=1, flags=flags)
runs = [eng.profile_forward(x, y, t, mode=1, flags=flags) for _ in range(5)]
runs.sort(key=lambda pr: sum(q["ms"] for q in pr))
prof = runs[2]                      # median of five back-to-back passes
print(f"flags={flags}")
tot = sum(p["ms"] for p in prof)
by = {}
for p in prof:
    d = by.setdefault(names[p["kind"]], [0.0, 0, 0.0])
    d[0] += p["ms"]; d[1] += 1; d[2] += p["flops"]
print(f"B={B} T={T}: {tot:.3f} ms per forward, {B * T * 128 / 16000 / (tot * 1e-3):.0f} audio-s/s (network only)")
for k, (ms, n, fl) in by.items():
    extra = f"  {fl / (ms * 1e-3) / 1e12:.0f} TFLOP/s" if fl > 0 else ""
    print(f"  {k:16s} {ms:8.3f} ms {n:4d} groups {100 * ms / tot:5.1f} %{extra}")
slow = sorted(prof, key=lambda p: -p["ms"])[:8]
print("  slowest groups:", [(names[p["kind"]], round(p["ms"], 3)) for p in slow])
# implicit-GEMM convolution launches grouped by (flops, bytes) signature: where the time above the tensor roofline sits
sig = {}
for p in prof:
    if p["kind"] == 1:
        d = sig.setdefault((p["flops"], p["bytes"]), [0, 0.0])
        d[0] += 1; d[1] += p["ms"]
PEAK = 1414.8e12
rows = sorted(sig.items(), key=lambda kv: -(kv[1][1] - kv[0][0] * kv[1][0] / PEAK * 1e3))
print("  conv signatures (GFLOP, MB, launches, ms total, TFLOP/s, ms above the sustained-peak time):")
for (fl, by), (n, ms) in rows:
    print(f"    {fl / 1e9:9.1f} GF {by / 1e6:8.1f} MB x{n:3d} {ms:7.3f} ms {fl * n / (ms * 1e-3) / 1e12:7.0f} TF/s "
          f"{ms - fl * n / PEAK * 1e3:+7.3f} ms")
# time by launch size class (latency-bound small maps vs throughput-bound large maps)
cls = {}
for (fl, by), (n, ms) in sig.items():
    key = "<3 GF" if fl < 3e9 else "<30 GF" if fl < 30e9 else "<100 GF" if fl < 100e9 else ">=100 GF"
    d = cls.setdefault(key, [0, 0.0, 0.0])
    d[0] += n; d[1] += ms; d[2] += fl * n
print("  conv launches by size class (launches, ms, ms at sustained peak, TFLOP/s):")
for key in ("<3 GF", "<30 GF", "<100 GF", ">=100 GF"):
    if key in cls:
        n, ms, fl = cls[key]
        print(f"    {key:9s} x{n:3d} {ms:7.3f} ms  ideal {fl / PEAK * 1e3:6.3f} ms  {fl / (ms * 1e-3) / 1e12:6.0f} TF/s")
