#!/usr/bin/env python
"""Micro-benchmark of the implicit-GEMM convolution kernels on the shapes of the 16 x 4 s workload.
Usage: python tools/conv_bench.py [--impl 0,2] [--iters 20] [--only IDX]"""
import argparse
import json
import math
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from snr_aligned_diffse_b200 import ops  # noqa: E402

SHAPES = [  # B, H, W, Cin, Cout, Cshortcut
    (16, 256, 512, 128, 128, 0),
    (16, 256, 512, 128, 128, 256),
    (16, 128, 256, 128, 128, 0),
    (16, 64, 128, 256, 256, 0),
    (16, 64, 128, 256, 256, 512),
    (16, 32, 64, 256, 256, 0),
    (16, 16, 32, 256, 256, 0),
    (16, 8, 16, 256, 256, 0),
    (16, 4, 8, 256, 256, 0),
]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--impl", default="0,2")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--only", type=int, default=-1)
    ap.add_argument("--debug", action="store_true")
    args = ap.parse_args()
    impls = [int(i) for i in args.impl.split(",")]
    g = torch.Generator().manual_seed(0)
    for idx, (B, H, W, Ci, Co, Cs) in enumerate(SHAPES):
        if args.only >= 0 and idx != args.only:
            continue
        x = (torch.randn(B, H, W, Ci, generator=g) * 0.5).to(torch.bfloat16).cuda()
        x1 = (torch.randn(B, H, W, Cs, generator=g) * 0.5).to(torch.bfloat16).cuda() if Cs else None
        wt = (torch.randn(Co, 9 * Ci + Cs, generator=g) / math.sqrt(9 * Ci + Cs)).to(torch.bfloat16).cuda()
        bias = torch.randn(Co, generator=g).cuda()
        flops = 2.0 * B * H * W * Co * (9 * Ci + Cs)
        row = dict(shape=(B, H, W, Ci, Co, Cs), gflop=flops / 1e9)
        outs = {}
        gamma = (torch.rand(Ci, generator=g) + 0.5).cuda()
        beta = (torch.randn(Ci, generator=g) * 0.2).cuda()

        def run(impl):
            if impl == 5:   # GroupNorm statistics + convolution normalising its operand in flight (timed together)
                return ops.gn_silu_conv3x3_nhwc(x, gamma, beta, wt, x1=x1, bias=bias)
            if impl == 6:   # 2-CTA kernel with GroupNorm partial sums in the epilogue (includes the host-side reduction)
                return ops.conv3x3_nhwc_stats(x, wt, x1=x1, bias=bias)[0]
            return ops.conv_nhwc(x, wt, 9, x1=x1, bias=bias, impl=impl)

        for impl in impls:
            for _ in range(3):
                out = run(impl)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.iters):
                out = run(impl)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / args.iters
            if impl in (0, 2, 3, 5, 6) and args.debug:
                from snr_aligned_diffse_b200 import _lib
                dbg = torch.zeros(148 * 8, dtype=torch.int64, device="cuda")
                _lib.load().snrse_conv_halo_set_debug(_lib.ptr(dbg))
                run(impl)
                torch.cuda.synchronize()
                _lib.load().snrse_conv_halo_set_debug(None)
                d = dbg.view(148, 8).double()
                d = d[d[:, 3] > 0]
                names = ["mma_wait_a", "mma_wait_b", "mma_wait_acc", "mma_total", "epi_wait_full", "epi_body", "prodA_wait", "prodB_wait"]
                if impl == 2:
                    names = ["prod_wait_empty", "prod_total", "mma_wait_full", "mma_total", "mma_first_wait", "-", "-", "-"]
                row[f"dbg{impl}_kcycles"] = {n: round(float(d[:, i].mean()) / 1e3, 1) for i, n in enumerate(names)}
            row[f"impl{impl}_ms"] = round(ms, 4)
            row[f"impl{impl}_tflops"] = round(flops / ms / 1e9, 1)
            outs[impl] = out
        if len(outs) == 2:
            a, b = (outs[i].float() for i in impls)
            row["max_diff"] = float((a - b).abs().max())
        print(json.dumps(row), flush=True)


if __name__ == "__main__":
    main()
