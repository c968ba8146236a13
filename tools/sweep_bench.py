#!/usr/bin/env python
"""Stand-alone CLI over snr_aligned_diffse_b200/workloads.py (BASELINE.json configs 3-5 and the 60-NFE PC loop) on
1..8 GPUs: one process per GPU under torchrun, or a single process.  bench.py prints the same records as sub-records of
its line; this tool exists for ad-hoc runs with other sizes.

    python tools/sweep_bench.py --workload vbd [--fixed-snr 0.31623] [--count 824] [--graphs 0]
    python tools/sweep_bench.py --workload long --count 2
    python tools/sweep_bench.py --workload pc [--graphs 0|1]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tools/sweep_bench.py --workload vbd
"""
import argparse
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from snr_aligned_diffse_b200 import workloads as wl  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="vbd", choices=["vbd", "long", "pc"])
    ap.add_argument("--count", type=int, default=0, help="utterances (vbd: total, default 824; long: per rank, default 2)")
    ap.add_argument("--fixed-snr", type=float, default=bench.FIXED_SNR)
    ap.add_argument("--max-batch", type=int, default=16)
    ap.add_argument("--target-frames", type=int, default=wl.SWEEP_TARGET_FRAMES,
                    help="vbd: padded frames per batch (0: at most --max-batch utterances per batch)")
    ap.add_argument("--repeat", type=int, default=2, help="passes over the list; the last one is timed")
    ap.add_argument("--enhancers", type=int, default=2, help="pc workload: independent batches in flight per GPU (graph mode)")
    ap.add_argument("--graphs", default="1", choices=["0", "1"], help="1: CUDA graphs (default), 0: eager launches")
    args = ap.parse_args()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    graphs = args.graphs == "1"
    if args.workload == "pc":
        out = wl.run_pc60(dev, rank, world, batch=bench.BATCH, seconds=bench.SECONDS, enhancers=args.enhancers,
                          reps=max(1, args.repeat - 1), graph=graphs)
    else:
        model, _ = bench.build_models(dev, fixed_snr=args.fixed_snr)
        if args.workload == "vbd":
            out = wl.run_sweep824(model, dev, rank, world, count=args.count or 824, max_batch=args.max_batch,
                                  graphs=graphs, repeat=args.repeat, target_frames=args.target_frames)
        else:
            out = wl.run_longform60(model, dev, rank, world, count=args.count or 2, graphs=graphs, repeat=args.repeat)
    if rank == 0:
        print(json.dumps(dict(workload=args.workload, unit=bench.UNIT, n_gpus=world, **out)), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
