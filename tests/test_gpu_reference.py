"""The CUDA path against the reference path on the benchmark's batch, every utterance.

tests/golden/bench_batch.npz (written by oracle/make_golden_bench_batch.py) holds what the fp32 reference path computes
for the bench batch (16 x 4 s, `synth_waves(16, 64000, seed=1000)`, estimator in the loop, explicit noise draw
`synth_noise(16, 512, seed=1001)`) and for a 2 x 10 s batch drawn the same way: every utterance's noise/clean ratio,
snapped timestep, norm factor, the peak of its enhanced waveform and the enhanced waveform at 2048 fixed, seeded sample
positions.  The vectors come from the CPU oracle, which reproduces the unmodified reference's stored outputs bit for
bit (tests/test_oracle_golden.py).  ALL utterances are then compared with `ScoreModel.enhance_batch` of this package:
snapped timestep exact, noise/clean ratio 1e-4, norm factor 1e-6, waveform SI-SDR >= 30 dB and max-abs error <= 5 % of
the peak at the stored positions -- bf16 activations vs the fp32 reference.
"""
import json
import os

import numpy as np
import pytest

from oracle import sampler as o_sampler
from oracle.topology import NCSNppConfig, param_specs, snrnet_param_specs
from snr_aligned_diffse_b200.synth import synth_noise, synth_state_dict, synth_waves

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("batch,seconds", [(16, 4.0), (2, 10.0)], ids=["config2_16x4s", "2x10s"])
def test_bench_batch_matches_reference_run_on_this_gpu(golden_dir, batch, seconds):
    z = np.load(os.path.join(golden_dir, "bench_batch.npz"))
    ref = {k: z[f"{batch}x{seconds:g}s_{k}"] for k in ("pos", "ratio", "t_index", "t", "norm_factor", "peak", "x_hat")}

    from snr_aligned_diffse_b200.sgmse import model as sg_model
    from snr_aligned_diffse_b200.sgmse.model import ScoreModel
    from snr_aligned_diffse_b200.sgmse.snr_estimator import SNRModel
    est = SNRModel(base_dir="")
    est._error_loading_ema = True
    est.load_state_dict(synth_state_dict(snrnet_param_specs(), seed=1))
    est.eval(no_ema=True)
    sg_model.set_snr_model(est)
    m = ScoreModel.from_state_dict(synth_state_dict(param_specs(NCSNppConfig()), seed=0), backbone="ncsnpp", sde="ouve",
                                   model_type="sebridge_v3", snr_conditioned="true", fixed_snr=0.17783, theta=1.5,
                                   sigma_min=0.05, sigma_max=1.0, base_dir="").eval(no_ema=True)
    L = int(seconds * 16000)
    tpad = 64 * ((1 + L // 128 + 63) // 64)
    y = synth_waves(batch, L, seed=1000)
    Z = synth_noise(batch, tpad, seed=1001)
    out, aux = m.enhance_batch(y, oracle=False, noise=Z, return_aux=True)
    got = out.cpu().numpy().astype(np.float64)
    assert got.shape == (batch, L) and ref["x_hat"].shape == (batch, len(ref["pos"]))
    rows = []
    for b in range(batch):
        assert float(aux["t"][b]) == np.float32(ref["t"][b]) and int(aux["t_index"][b]) == int(ref["t_index"][b])
        assert abs(float(aux["ratio"][b]) / float(ref["ratio"][b]) - 1) <= 1e-4
        assert abs(float(aux["norm_factor"][b]) / float(ref["norm_factor"][b]) - 1) <= 1e-6
        assert np.isfinite(got[b]).all()
        want = ref["x_hat"][b].astype(np.float64)
        g = got[b, ref["pos"]]
        sdr = o_sampler.si_sdr(want, g)
        mx = float(np.abs(g - want).max() / ref["peak"][b])
        rows.append((sdr, mx))
    d = os.path.join(ROOT, "gpurun_out")
    os.makedirs(d, exist_ok=True)
    with open(os.path.join(d, "parity_rows.jsonl"), "a") as f:
        f.write(json.dumps(dict(case=f"reference_{batch}x{seconds:g}s (all items, stored vectors)", si_sdr_db_min=min(r_[0] for r_ in rows),
                                si_sdr_db_mean=float(np.mean([r_[0] for r_ in rows])),
                                maxabs_of_peak_max=max(r_[1] for r_ in rows))) + "\n")
    # SI-SDR >= 30 dB for EVERY item.  The max-abs figure here is the worst single sample of the whole batch (16 x 2048 or
    # 2 x 2048 stored samples): an extreme-value statistic of the bf16 rounding noise whose realisation changes whenever the
    # arithmetic changes anywhere (3.2 % / 4.3 % for two accumulation orders of the same 16 x 4 s batch), hence 5 % for
    # the batch maximum; the single-utterance cases of test_gpu_configs.py keep 4 % for utterances up to 4 s.
    assert min(r_[0] for r_ in rows) >= 30.0 and max(r_[1] for r_ in rows) <= 5e-2, rows
