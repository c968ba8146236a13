#!/usr/bin/env python
"""Parity numbers of the CUDA path against the committed reference fixtures (tests/golden, generated from the
unmodified reference by oracle/make_golden.py): prints a small markdown table.  Run on the GPU box."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import sampler as o_sampler  # noqa: E402  (checker only)
from oracle.topology import NCSNppConfig, param_specs  # noqa: E402
from snr_aligned_diffse_b200.sgmse.model import ScoreModel  # noqa: E402
from snr_aligned_diffse_b200.synth import synth_state_dict  # noqa: E402

G = os.path.join(ROOT, "tests", "golden")
c = lambda a: torch.from_numpy(np.ascontiguousarray(a))  # noqa: E731


def rel_l2(a, b):
    a, b = torch.view_as_real(a).double().flatten(), torch.view_as_real(b).double().flatten()
    return float((a - b).norm() / b.norm())


sd = synth_state_dict(param_specs(NCSNppConfig()), seed=0)
m = ScoreModel.from_state_dict(sd, backbone="ncsnpp", sde="ouve", model_type="sebridge_v3", snr_conditioned="true",
                               fixed_snr=0.17783, theta=1.5, sigma_min=0.05, sigma_max=1.0, base_dir="").eval(no_ema=True)
z = np.load(os.path.join(G, "enhance_v3.npz"))
y, Z = c(z["y"]), c(z["Z"])
x_hat = m.enhance(y, y, oracle=True, clean_rms=1.0, noise_rms=float(z["ratio"]), noise=Z)
ref = z["x_hat"]
out, aux = m.enhance_batch(y, oracle=True, noise_over_clean=[float(z["ratio"])], noise=Z, return_aux=True)
print("| quantity (fixture enhance_v3.npz: reference ScoreModel.enhance path on seeded weights / input / noise) | value | test bound |")
print("|---|---:|---:|")
print(f"| snapped timestep t == reference | {float(aux['t'][0]) == np.float32(z['t'])} | exact |")
print(f"| norm factor relative error | {abs(float(aux['norm_factor'][0]) / float(z['norm_factor']) - 1):.2e} | 1e-6 |")
print(f"| network output (spectrogram) rel-L2 vs reference fp32 | {rel_l2(aux['sample'].cpu(), c(z['sample'])[:, 0]):.3e} | 3e-2 |")
print(f"| enhanced waveform SI-SDR vs reference waveform | {o_sampler.si_sdr(ref.astype(np.float64), x_hat.astype(np.float64)):.1f} dB | >= 28 dB |")
print(f"| enhanced waveform max-abs error / peak | {np.abs(x_hat - ref).max() / np.abs(ref).max():.3e} | 8e-2 |")
zn = np.load(os.path.join(G, "ncsnpp_forward.npz"))
x, t = c(zn["x"]), c(zn["t"])
eng = m.dnn.engine
for flags, name in ((0, "default (2-CTA tcgen05, GroupNorm in flight)"), (2, "fp32 CUDA-core convolutions")):
    o = eng.forward(x[:, 0].cuda(), x[:, 1].cuda(), t.cuda(), mode=0, flags=flags).cpu()
    print(f"| NCSN++ forward rel-L2 vs reference, {name} | {rel_l2(o, c(zn['out'])[:, 0]):.3e} | 3e-2 |")
