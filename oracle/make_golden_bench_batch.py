#!/usr/bin/env python
"""Golden vectors of the reference path on the benchmark's batches, for tests/test_gpu_reference.py.

    python oracle/make_golden_bench_batch.py     # writes tests/golden/bench_batch.npz

Inputs are the benchmark's: `synth_waves(B, L, seed=1000)`, the explicit noise draw `synth_noise(B, Tpad, seed=1001)`,
the seeded synthetic score-model (seed 0) and SNR-estimator (seed 1) weights.  Every utterance goes through the CPU
oracle in fp32: SNR estimator -> t snap / norm factor -> sebridge_v3 pass (oracle.snrnet, oracle.sampler).  The oracle
restates the reference and reproduces its stored outputs bit for bit (tests/golden/oracle_vs_reference.json,
tests/test_oracle_golden.py), so these vectors stand for the unmodified reference run on the same inputs.  Where a
copy of the reference is installed (baseline/_ref), `baseline/ref_runner.py --task parity` computes the same
quantities with the reference's own code.

Per case (`16x4s`: 16 x 4 s, the batch bench.py times; `2x10s`: 2 x 10 s) the file holds every utterance's
noise/clean ratio, snapped t_30 index and t, norm factor and the peak of its enhanced waveform, and the enhanced
waveforms at a fixed, seeded set of N_POS sample positions (the whole waveforms would not fit a small file).
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import sampler as o_sampler, snrnet as o_snrnet  # noqa: E402
from oracle.topology import NCSNppConfig, param_specs, snrnet_param_specs  # noqa: E402
from snr_aligned_diffse_b200.synth import synth_noise, synth_state_dict, synth_waves  # noqa: E402

FIXED_SNR, SR, N_POS = 0.17783, 16000, 2048
CASES = {"16x4s": (16, 4.0), "2x10s": (2, 10.0)}


def main():
    torch.set_num_threads(os.cpu_count() or 1)
    sd = synth_state_dict(param_specs(NCSNppConfig()), seed=0)
    snr_sd = synth_state_dict(snrnet_param_specs(), seed=1)
    out = {}
    for tag, (batch, seconds) in CASES.items():
        L = int(seconds * SR)
        tpad = 64 * ((1 + L // 128 + 63) // 64)
        y = synth_waves(batch, L, seed=1000)
        Z = synth_noise(batch, tpad, seed=1001)
        pos = np.sort(np.random.default_rng(2024).choice(L, N_POS, replace=False)).astype(np.int32)
        rows = {k: [] for k in ("ratio", "t_index", "t", "norm_factor", "peak", "x_hat")}
        for b in range(batch):
            with torch.no_grad():
                ratio = float(o_snrnet.estimate_noise_over_clean(snr_sd, y[b:b + 1])[0, 0])
                o = o_sampler.enhance_v3(sd, y[b:b + 1], Z[b:b + 1], ratio, FIXED_SNR, sigma_max=1.0)
            x_hat = o["x_hat"].numpy()
            for k, v in (("ratio", ratio), ("t_index", o["t_index"]), ("t", o["t"]), ("norm_factor", o["norm_factor"]),
                         ("peak", float(np.abs(x_hat).max())), ("x_hat", x_hat[pos])):
                rows[k].append(v)
            print(f"{tag} item {b}: t_index {o['t_index']}, ratio {ratio:.6g}", flush=True)
        out[tag + "_pos"] = pos
        for k, v in rows.items():
            out[f"{tag}_{k}"] = np.asarray(v, dtype={"t_index": np.int64, "x_hat": np.float32}.get(k, np.float64))
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", "bench_batch.npz"), **out)


if __name__ == "__main__":
    main()
