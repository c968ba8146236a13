"""CPU-only tests of the host side: the C ABI loads and exports every symbol the header declares, the
native parameter table matches the reference inventory, the `sgmse` mirror keeps the reference's
names / errors, checkpoints (Lightning layout + EMA) load without a GPU, utterance sharding."""
import ctypes
import json
import os
import re
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_abi_exports_every_declared_symbol():
    from snr_aligned_diffse_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "snrse_b200.h")).read()
    dbg = open(os.path.join(ROOT, "include", "snrse_b200_debug.h")).read()
    product = set(re.findall(r"\b(snrse_[a-z0-9_]+)\s*\(", hdr))
    debug = set(re.findall(r"\b(snrse_[a-z0-9_]+)\s*\(", dbg))
    # measurement / debug entry points live in their own header, not in the product ABI
    assert debug == {"snrse_ncsnpp_num_launch_groups", "snrse_ncsnpp_profile_forward", "snrse_ncsnpp_read_tap",
                     "snrse_conv_halo_set_debug"} and not (debug & product)
    declared = product | debug
    lib = _lib.load()
    assert declared, "no declarations found"
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert declared == set(_lib.PROTOTYPES), declared ^ set(_lib.PROTOTYPES)
    assert lib.snrse_version() == 100


def test_abi_exports_every_layer_entry_point():
    """The executor's launchers as entry points (include/snrse_b200_layers.h): all exported, all in
    _lib.LAYER_PROTOTYPES, none in the product ABI or the measurement header."""
    from snr_aligned_diffse_b200 import _lib
    found = lambda f: set(re.findall(r"\b(snrse_[a-z0-9_]+)\s*\(", open(os.path.join(ROOT, "include", f)).read()))  # noqa: E731
    layers = found("snrse_b200_layers.h")
    assert layers == {"snrse_dbg_conv", "snrse_dbg_gn_stats", "snrse_dbg_gn_finalize", "snrse_dbg_gn_apply",
                      "snrse_dbg_fir", "snrse_dbg_fir_dual", "snrse_dbg_conv_out4", "snrse_dbg_pack_input",
                      "snrse_dbg_conv_in4", "snrse_dbg_combine4", "snrse_dbg_temb", "snrse_dbg_final",
                      "snrse_dbg_attention"}
    assert not layers & (found("snrse_b200.h") | found("snrse_b200_debug.h"))
    assert layers == set(_lib.LAYER_PROTOTYPES), layers ^ set(_lib.LAYER_PROTOTYPES)
    lib = _lib.load()
    for name in layers:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"


def test_pdl_mask_round_trip():
    """snrse_set_pdl is host-only state: returns the previous mask, keeps three bits, a negative argument only queries."""
    from snr_aligned_diffse_b200 import _lib
    lib = _lib.load()
    prev = lib.snrse_set_pdl(-1)
    try:
        assert 0 <= prev <= 7
        assert lib.snrse_set_pdl(5) == prev and lib.snrse_set_pdl(-1) == 5
        assert lib.snrse_set_pdl(0xFF) == 5 and lib.snrse_set_pdl(-1) == 7
        assert lib.snrse_set_pdl(0) == 7 and lib.snrse_set_pdl(-1) == 0
    finally:
        lib.snrse_set_pdl(prev)


def test_product_has_no_oracle_or_fallback_imports():
    pkg = os.path.join(ROOT, "snr_aligned_diffse_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith(".py"):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, re.M), f"{f} imports the oracle"
                assert "/root/reference" not in src


def test_native_param_table_matches_reference_inventory(golden_dir):
    from snr_aligned_diffse_b200.engine import NCSNppEngine
    ref = json.load(open(os.path.join(golden_dir, "ncsnpp_param_specs.json")))
    eng = NCSNppEngine()
    shapes = eng.param_shapes()
    assert set(shapes) == set(ref)
    assert all(tuple(shapes[k]) == tuple(ref[k]) for k in ref)
    assert eng.lib.snrse_ncsnpp_num_modules(eng.h) == 77
    # plan sizes are computable without a GPU and grow with the bucket
    a, b = eng.workspace_bytes(1, 256, 64), eng.workspace_bytes(2, 256, 128)
    assert 0 < a < b
    with pytest.raises(RuntimeError):
        eng.workspace_bytes(1, 256, 96)      # T must be a multiple of 64 (6 halvings, util/other.py:83-90)
    with pytest.raises(RuntimeError):
        eng.workspace_bytes(1, 128, 64)      # attention placement was built for F = image_size
    assert all(eng.workspace_bytes(1, 256, 64, flags=f) > 0 for f in (1, 2, 3))
    for f in (4, 128, -1):                   # only bit0 (keep every activation) and bit1 (cross-check) are defined
        with pytest.raises(RuntimeError, match="unknown flags"):
            eng.workspace_bytes(1, 256, 64, flags=f)


def test_weight_packing_layouts():
    from snr_aligned_diffse_b200.engine import NCSNppEngine
    from snr_aligned_diffse_b200.synth import synth_state_dict
    eng = NCSNppEngine()
    sd = synth_state_dict(eng.param_shapes(), seed=3)
    blob = eng.pack_state_dict(sd)
    tab = {p["name"]: p for p in eng.param_table()}
    b16, f32 = blob.view(torch.bfloat16), blob.view(torch.float32)
    # 3x3 conv: K-major rows [cout][(r*3+s)*Cin + cin]
    p = tab["dnn.all_modules.4.Conv_0.weight"]
    w = sd[p["name"]]
    rows = b16[p["offset"] // 2: p["offset"] // 2 + 128 * p["row_stride"]].view(128, p["row_stride"])
    assert rows[5, (1 * 3 + 2) * 128 + 7] == w[5, 7, 1, 2].to(torch.bfloat16)
    # fused Conv_1 | Conv_2 rows and summed bias (layerspp.py:268-272)
    p1, p2 = tab["dnn.all_modules.12.Conv_1.weight"], tab["dnn.all_modules.12.Conv_2.weight"]
    assert p1["offset"] == p2["offset"] and p1["row_stride"] == 9 * 256 + 128 and p2["k_offset"] == 9 * 256
    rows = b16[p1["offset"] // 2: p1["offset"] // 2 + 256 * p1["row_stride"]].view(256, p1["row_stride"])
    assert rows[9, 9 * 256 + 100] == sd[p2["name"]][9, 100, 0, 0].to(torch.bfloat16)
    pb = tab["dnn.all_modules.12.Conv_1.bias"]
    got = f32[pb["offset"] // 4: pb["offset"] // 4 + 256]
    assert torch.equal(got, sd["dnn.all_modules.12.Conv_1.bias"] + sd["dnn.all_modules.12.Conv_2.bias"])
    # NIN W[in,out] -> rows [out][in]
    pn = tab["dnn.all_modules.21.NIN_1.W"]
    rows = b16[pn["offset"] // 2: pn["offset"] // 2 + 256 * 256].view(256, 256)
    assert rows[3, 200] == sd[pn["name"]][200, 3].to(torch.bfloat16)


def test_registries_and_constructor_errors():
    from snr_aligned_diffse_b200.sgmse import sampling
    from snr_aligned_diffse_b200.sgmse.backbones import BackboneRegistry
    from snr_aligned_diffse_b200.sgmse.model import ScoreModel, t_30
    from snr_aligned_diffse_b200.sgmse.sdes import SDERegistry
    assert set(SDERegistry.get_all_names()) >= {"ouve", "bbed"}
    assert set(BackboneRegistry.get_all_names()) >= {"ncsnpp", "snrnet"}
    assert sampling.PredictorRegistry.get_all_names() == ['euler_maruyama', 'reverse_diffusion', 'none']
    assert sampling.CorrectorRegistry.get_all_names() == ['langevin', 'ald', 'none']
    with pytest.raises(ValueError):
        SDERegistry.get_by_name("nope")
    with pytest.raises(ValueError):
        ScoreModel(backbone="nope", sde="ouve", theta=1.5, sigma_min=0.05, sigma_max=0.5)
    with pytest.raises(NotImplementedError):
        ScoreModel(backbone="ncsnpp", sde="ouve", theta=1.5, sigma_min=0.05, sigma_max=0.5, resblock_type="ddpm")
    assert t_30.dtype == np.float64 and t_30[0] == pytest.approx(0.001) and t_30[-1] == 1.0
    m = ScoreModel(backbone="ncsnpp", sde="ouve", model_type="sebridge_v3", snr_conditioned="fixed", theta=1.5,
                   sigma_min=0.05, sigma_max=1.0)
    with pytest.raises(NotImplementedError):
        m.enhance(torch.zeros(1, 4000), torch.zeros(1, 4000))      # model.py:792-793
    # eval.py pokes these attributes (eval.py:105-108)
    assert m.sde.__class__.__name__ == "OUVESDE"
    m.sde._T = 0.5
    assert m.sde.T == 0.5
    b = SDERegistry.get_by_name("bbed")(T_sampling=0.999, k=2.6, theta=0.52, N=30)
    b.T = 0.5
    assert b.copy().T == 0.5


def test_lightning_checkpoint_with_ema_loads_on_cpu(tmp_path):
    from snr_aligned_diffse_b200.sgmse.data_module import SpecsDataModule
    from snr_aligned_diffse_b200.sgmse.model import ScoreModel
    from snr_aligned_diffse_b200.synth import synth_state_dict
    hp = dict(backbone="ncsnpp", sde="ouve", model_type="sebridge_v3", snr_conditioned="true", fixed_snr=0.31623,
              theta=1.5, sigma_min=0.05, sigma_max=1.0, data_module_cls=SpecsDataModule, base_dir="/data")
    probe = ScoreModel(**hp)
    names = list(probe.dnn.param_shapes())
    sd = synth_state_dict({"dnn." + k: v for k, v in probe.dnn.param_shapes().items()}, seed=5)
    shadow = [sd["dnn." + n] * 0.5 for n in names if n != "all_modules.0.W"]
    path = str(tmp_path / "m.ckpt")
    torch.save({"state_dict": sd, "hyper_parameters": hp,
                "ema": {"decay": 0.999, "num_updates": 7, "shadow_params": shadow, "collected_params": None}}, path)
    m = ScoreModel.load_from_checkpoint(path, base_dir="", batch_size=16, num_workers=0, kwargs=dict(gpu=False))
    assert m.fixed_snr == 0.31623 and m.data_module.base_dir == ""
    key = "all_modules.4.Conv_0.weight"
    assert torch.equal(m.dnn.state_dict()[key], sd["dnn." + key])
    m.eval(no_ema=False)                                            # EMA weights become live (model.py:120-126)
    assert torch.equal(m.dnn.state_dict()[key], sd["dnn." + key] * 0.5)
    assert torch.equal(m.dnn.state_dict()["all_modules.0.W"], sd["dnn.all_modules.0.W"])   # frozen: not in EMA
    m.train(True)
    assert torch.equal(m.dnn.state_dict()[key], sd["dnn." + key])
    m.eval(no_ema=True)
    assert torch.equal(m.dnn.state_dict()[key], sd["dnn." + key])
    with pytest.warns(UserWarning, match="no CPU path"):
        assert m.cpu() is m                                         # accepted, a stated no-op (eval.py:101 call site)
    assert m.to("cuda") is m and m.to("cpu") is m


def test_param_table_order_equals_reference_ema_order():
    """torch-ema's shadow_params follow the reference's `parameters()` order (requires_grad only).  `_ema_state_dict`
    zips them with the native table order, so that order -- not just the set of names -- must equal the list
    oracle/make_golden.py took from the live reference object (tests/golden/ncsnpp_ema_order.json)."""
    import json
    from snr_aligned_diffse_b200.engine import NCSNppEngine
    ref_order = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "ncsnpp_ema_order.json")))
    mine = [n for n in NCSNppEngine().param_shapes() if n != "dnn.all_modules.0.W"]
    assert mine == ref_order


def test_checkpoint_load_does_not_clobber_a_foreign_sgmse_package(tmp_path):
    import sys
    import types
    from snr_aligned_diffse_b200.sgmse._checkpoint import load_checkpoint_file
    path = str(tmp_path / "x.ckpt")
    torch.save({"state_dict": {}, "hyper_parameters": {}}, path)
    fake = types.ModuleType("sgmse")
    fake_dm = types.ModuleType("sgmse.data_module")
    saved = {k: v for k, v in sys.modules.items() if k == "sgmse" or k.startswith("sgmse.")}
    for k in saved:
        del sys.modules[k]
    sys.modules["sgmse"], sys.modules["sgmse.data_module"] = fake, fake_dm
    try:
        load_checkpoint_file(path)
        assert sys.modules["sgmse"] is fake and sys.modules["sgmse.data_module"] is fake_dm
        assert "sgmse.model" not in sys.modules
    finally:
        for k in [k for k in sys.modules if k == "sgmse" or k.startswith("sgmse.")]:
            del sys.modules[k]
        sys.modules.update(saved)


def test_missing_library_or_gpu_fails_loudly():
    from snr_aligned_diffse_b200 import _lib, ops
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError):
        _lib.require_device()
    with pytest.raises((RuntimeError, AssertionError)):
        ops.stft(torch.zeros(1, 4000))


def test_sharding_lpt():
    from snr_aligned_diffse_b200.shard import bucket_batches, lpt_shards, synthetic_lengths
    L = synthetic_lengths(824, seed=0)
    assert len(L) == 824 and L.min() >= 24000 and L.max() <= 160000
    for g in (1, 2, 4, 8):
        shards = lpt_shards(L, g)
        flat = sorted(i for s in shards for i in s)
        assert flat == list(range(824))                              # a partition: nothing lost, nothing doubled
        loads = [sum(64 * (-(-(1 + L[i] // 128) // 64)) for i in s) for s in shards]
        assert max(loads) - min(loads) <= 1280                       # within one longest utterance
    batches = bucket_batches(L, list(range(824)), max_batch=16)
    assert sorted(i for _, idx in batches for i in idx) == list(range(824))
    for tpad, idx in batches:
        assert len(idx) <= 16 and all(64 * (-(-(1 + L[i] // 128) // 64)) == tpad for i in idx)
    # frame-budget batching: still a partition into equal-Tpad batches, short utterances in larger batches (<= 64),
    # long ones never below max_batch, fewer batches overall
    big = bucket_batches(L, list(range(824)), max_batch=16, target_frames=16384)
    assert sorted(i for _, idx in big for i in idx) == list(range(824)) and len(big) < len(batches)
    for tpad, idx in big:
        assert len(idx) <= max(16, min(64, 16384 // tpad)) and all(64 * (-(-(1 + L[i] // 128) // 64)) == tpad for i in idx)
    # batch-level sharding (what the sweep uses): a partition into the SAME global batches, full batches stay full,
    # and the modelled job time (slowest rank) beats utterance-level sharding + per-rank batching
    from snr_aligned_diffse_b200.shard import batch_cost, batch_shards
    for g in (1, 2, 4, 8):
        per_rank = batch_shards(L, g, max_batch=16)
        got = sorted((tpad, tuple(idx)) for r in per_rank for tpad, idx in r)
        assert got == sorted((tpad, tuple(idx)) for tpad, idx in batches)
        new = max(sum(batch_cost(t, len(i)) for t, i in r) for r in per_rank)
        old = max(sum(batch_cost(t, len(i)) for t, i in bucket_batches(L, s, 16)) for s in lpt_shards(L, g))
        assert new <= old
        if g == 8:
            assert new <= 0.85 * old and max(len(r) for r in per_rank) <= 8


def test_wav_io_round_trip_and_file_loop(tmp_path):
    """wavio: PCM16 read (x / 32768, torchaudio's normalisation) and write; the eval.py-style file loop with a fake
    enhancer (halves the signal) writes one wav per input and reports SI-SDR-less metrics in id order."""
    import numpy as np
    from snr_aligned_diffse_b200 import wavio
    g = torch.Generator().manual_seed(0)
    noisy_dir, out_dir = tmp_path / "noisy", tmp_path / "out"
    files = []
    for i, n in enumerate((3000, 5200, 4100)):
        w = (torch.randn(n, generator=g) * 0.1).clamp(-0.99, 0.99)
        f = str(noisy_dir / f"p{i:03d}.wav")
        wavio.write_wav(f, w)
        back, sr = wavio.read_wav(f)
        assert sr == 16000 and back.shape == w.shape and (back - w).abs().max() <= 1.0 / 32767 + 1e-7
        files.append(f)
    res = wavio.enhance_files(lambda y, n: 0.5 * y, files, str(out_dir), max_batch=2)
    assert sorted(res["files"]) == ["p000.wav", "p001.wav", "p002.wav"] and len(res["ids"]) == 3
    for f in files:
        a, _ = wavio.read_wav(f)
        b, _ = wavio.read_wav(str(out_dir / os.path.basename(f)))
        assert b.shape == a.shape and (b - 0.5 * a).abs().max() <= 1.5 / 32767
    with pytest.raises(ValueError):
        import wave
        with wave.open(str(tmp_path / "stereo.wav"), "wb") as w:
            w.setnchannels(2); w.setsampwidth(2); w.setframerate(16000); w.writeframes(b"\x00" * 8)
        wavio.read_wav(str(tmp_path / "stereo.wav"))


def test_rk45_step_controller_equals_scipy_on_cpu():
    """The host-side step controller of the on-device ODE sampler (sgmse/sampling/ode.py) restates scipy's RK45
    (`select_initial_step`, `rk_step`, `_step_impl`).  With the two CUDA operators replaced by float64 torch stand-ins
    (same formulas as csrc/sampler.cu) it must take exactly scipy's steps: equal nfev and the same end state."""
    import math
    from scipy import integrate
    from snr_aligned_diffse_b200.sgmse.sampling.ode import rk45_integrate

    class CpuKernels:                      # what rk_combine_kernel / rk_scaled_sqnorm_kernel compute, in complex128
        @staticmethod
        def rk_combine(y, K, coef, h):
            acc = sum(float(c) * K[j] for j, c in enumerate(coef))
            return (y if y is not None else 0) + h * acc

        @staticmethod
        def rk_scaled_norm(K, coef, h, y, y2, atol, rtol):
            num = h * sum(float(c) * K[j] for j, c in enumerate(coef))
            mag = y.abs() if y2 is None else torch.maximum(y.abs(), y2.abs())
            return math.sqrt(float(((num.abs() / (atol + rtol * mag)) ** 2).mean()))

    g = torch.Generator().manual_seed(12)
    y0 = torch.view_as_complex(torch.randn(3, 40, 2, generator=g, dtype=torch.float64))
    lam = torch.view_as_complex(torch.stack([torch.rand(3, 40, generator=g, dtype=torch.float64) * 3 + 0.5,
                                             torch.randn(3, 40, generator=g, dtype=torch.float64) * 4], -1))
    lam_n = lam.numpy().reshape(-1)
    for (t0, t1), rtol, atol in (((1.0, 0.03), 1e-5, 1e-5), ((1.0, 0.03), 1e-3, 1e-6), ((0.0, 0.7), 1e-6, 1e-8)):
        res = rk45_integrate(lambda t, y: lam * y * (0.5 + t) + (1.0 - t), t0, y0, t1, rtol=rtol, atol=atol,
                             _kernels=CpuKernels)
        sol = integrate.solve_ivp(lambda t, y: lam_n * y * (0.5 + t) + (1.0 - t), (t0, t1), y0.numpy().reshape(-1),
                                  rtol=rtol, atol=atol, method="RK45")
        assert res.status == 0 and res.t == t1 and res.nfev == sol.nfev
        ref = torch.from_numpy(sol.y[:, -1]).reshape(y0.shape)
        assert (res.y - ref).abs().max() <= 1e-12 * float(ref.abs().max())
    # a CPU state without stand-in kernels is refused: there is no CPU implementation behind the sampler
    with pytest.raises(ValueError):
        rk45_integrate(lambda t, y: y, 1.0, y0.to(torch.complex64), 0.5)


def test_flat_weight_file_round_trip(tmp_path):
    """export_flat / read_flat (SURVEY 8f-2): header describes the packed layout, the blob is byte-identical to
    pack_state_dict, corruption and foreign files are rejected."""
    from snr_aligned_diffse_b200.engine import NCSNppEngine
    from snr_aligned_diffse_b200.synth import synth_state_dict
    eng = NCSNppEngine()
    sd = synth_state_dict(eng.param_shapes(), seed=3)
    path = str(tmp_path / "w.snrse")
    header = eng.export_flat(sd, path)
    assert header["weight_bytes"] == eng.weight_bytes and len(header["params"]) == len(eng.param_table())
    h2, blob = NCSNppEngine.read_flat(path)
    assert h2 == header and torch.equal(blob, eng.pack_state_dict(sd))
    raw = bytearray(open(path, "rb").read())
    raw[-5] ^= 0xFF
    open(path, "wb").write(bytes(raw))
    with pytest.raises(ValueError, match="corrupt"):
        NCSNppEngine.read_flat(path)
    open(path, "wb").write(b"not a weight file")
    with pytest.raises(ValueError, match="not a snrse_b200"):
        NCSNppEngine.read_flat(path)
