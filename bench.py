#!/usr/bin/env python
"""Benchmark of the SNR-aligned diffusion enhancement hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): sebridge_v3 NCSN++ (65.6 M parameters, seeded synthetic
"de-degenerated" weights), a batch of 16 synthetic 4 s / 16 kHz utterances per GPU, the full
reference-exact sebridge_v3 pass per step: max|y| -> SNR estimator -> t snap / norm factor -> STFT +
exponent transform -> X_T = Y + sigma t Z -> preconditioned NCSN++ (1 NFE) -> inverse transform + iSTFT,
captured in one CUDA graph.  Metric: enhanced audio-seconds per wall-second (inverse RTF), whole job.

  value    : inputs resident in HBM, CUDA-graph replay, CUDA-event timed, max over ranks (two independent enhancers
             whose steps alternate on two streams; `latency` holds the strictly back-to-back single-enhancer step).
  e2e      : the public API call with HOST buffers: pinned-host -> device copy of the waveforms and device ->
             pinned-host copy of the enhanced waveforms inside the timed region, every step.
  roofline : the implicit-GEMM convolution kernels (tensor bound): algorithmic FLOPs of all their launches in one step /
             their summed duration, CUDA events on the launch stream, measured in STEADY STATE (>= 2 s of back-to-back
             steps immediately before and between the profiled passes) against the sustained measured bf16 peak; the
             same measurement from an idle start against the burst peak is reported beside it.
  parity   : utterance 0 of the timed batch against the CPU oracle (outside the timed region): finite, SI-SDR >= 30 dB.
  gpu_eager_baseline : the UNMODIFIED reference (baseline/_ref) run in torch eager mode on the same GPU, same inputs
             (cuDNN / cuBLAS / cuFFT kernel set): the bar on the same box.  N = 1 only.
  cpu_baseline / --impl reference : the reference's own `ScoreModel.enhance` driven as eval.py does (NCSN++ on the host
             CPU, all host threads), on a bounded sample; the oracle port (oracle/) only if baseline/_ref is absent.
  sweep824 / longform60 / pc60 : BASELINE configs 3-5 and the 60-NFE PC loop at this N (snr_aligned_diffse_b200/workloads.py).
Multi-GPU (torchrun, one rank per GPU): utterances are independent, every rank processes its own batch of
16 (weak scaling), no data-path collective; NCCL only for the barrier and the max-over-ranks timing.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BATCH, SECONDS, SR = 16, 4.0, 16000
FIXED_SNR = 0.17783
METRIC = "enhanced audio-sec/sec (inverse RTF), sebridge_v3 1 NFE"
UNIT = "audio_s/s"
# the workload both arms (--impl b200 / --impl reference) are measured on; `config` is identical in both lines
WORKLOAD = ("sebridge_v3 NCSN++ 65.6M (synthetic de-degenerated weights), 16 x 4 s @ 16 kHz per GPU (Tpad=512), 1 NFE, "
            "SNR estimator in the loop")
REF_RUNNER = os.path.join(ROOT, "baseline", "ref_runner.py")


def synth_waves(batch, length, seed):
    from snr_aligned_diffse_b200.synth import synth_waves as sw
    return sw(batch, length, seed, SR)


def config_dict(world):
    return dict(workload=WORKLOAD, global_batch=world * BATCH, seconds_per_utterance=SECONDS, nfe=1,
                parallelism=f"dp{world} (utterance-sharded, no collective)",
                l2="per-step working set 5.4 GB >> 126 MB L2, no flush needed")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.path = tempfile.mktemp(suffix=".csv")
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(index)], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[])
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                s_, m_, p_ = float(f[1]), float(f[2]), float(f[3])
            except ValueError:
                continue
            if p_ < 350.0:          # idle sample (between regions): not "under load"
                continue
            sm.append(s_); mx.append(m_); pw.append(p_)
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if sm:
            sm.sort()
            out = dict(sm_mhz=sm[len(sm) // 2], sm_min_mhz=sm[0], sm_max_mhz=max(mx), power_w_max=max(pw),
                       reasons=sorted(reasons), samples=len(sm))
        try:
            os.remove(self.path)
        except OSError:
            pass
        return out


def _cpu_model():
    try:
        for l in open("/proc/cpuinfo"):
            if l.startswith("model name"):
                return l.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def _run_ref_runner(argv, timeout):
    """baseline/ref_runner.py in its own process (the reference's `sgmse` package must not share a process with the
    mirror).  Returns the parsed JSON line or dict(unavailable=...)."""
    if not os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "sgmse-bbed")):
        return dict(unavailable="baseline/_ref absent (created by __graft_entry__.build() where /root/reference exists)")
    try:
        r = subprocess.run([sys.executable, REF_RUNNER] + argv, capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    except subprocess.TimeoutExpired:
        return dict(unavailable=f"reference runner exceeded {timeout} s")
    for line in reversed(r.stdout.splitlines()):
        if line.startswith("{"):
            return json.loads(line)
    return dict(unavailable=("reference runner failed: " + (r.stderr.strip().splitlines() or ["no output"])[-1])[:300])


# ----------------------------------------------------------------------------------------------- reference arm
def cpu_port_step(sd, snr_sd, wave, Z):
    """One utterance through the CPU oracle port of ScoreModel.enhance (fallback when baseline/_ref is absent)."""
    import torch
    from oracle import sampler as o_sampler, snrnet as o_snrnet
    with torch.no_grad():
        ratio = float(o_snrnet.estimate_noise_over_clean(snr_sd, wave)[0, 0])
        return o_sampler.enhance_v3(sd, wave, Z, ratio, FIXED_SNR, sigma_max=1.0)["x_hat"]


def reference_cpu(steps, warmup, utts_per_step):
    """The reference's CPU path on a bounded sample of the 16 x 4 s workload: `utts_per_step` utterances of the batch
    per step (rotating through the 16), each through the unmodified `ScoreModel.enhance` as eval.py:94-132 drives it.
    -> (audio_s_per_s, seconds_total, cores, kind, sample description)."""
    r = _run_ref_runner(["--task", "enhance_cpu", "--batch", str(BATCH), "--seconds", str(SECONDS), "--seed", "1000",
                         "--steps", str(steps), "--warmup", str(warmup), "--utts-per-step", str(utts_per_step)], 1500)
    if "unavailable" not in r:
        sample = (f"{utts_per_step} of the 16 utterances (4 s each) per step, rotating through the batch, {steps} timed "
                  f"steps after {warmup} warm-up; unmodified reference ScoreModel.enhance as eval.py drives it "
                  "(model.cpu(): NCSN++ on the host, SNR estimator + front-end STFT where the reference puts them), fp32")
        return r["audio_s_per_s"], r["seconds_total"], r["cores"], "reference", sample, r.get("cpu_model", _cpu_model())
    # fallback: oracle port (baseline/_ref missing, or no CUDA device for the reference's hard-coded .cuda() calls)
    import torch
    from oracle.topology import NCSNppConfig, param_specs, snrnet_param_specs
    from snr_aligned_diffse_b200.synth import synth_noise, synth_state_dict
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = synth_state_dict(param_specs(NCSNppConfig()), seed=0)
    snr_sd = synth_state_dict(snrnet_param_specs(), seed=1)
    L = int(SECONDS * SR)
    waves = synth_waves(BATCH, L, seed=1000)
    Z = synth_noise(1, 512, seed=1)

    def step(i):
        for u in range(utts_per_step):
            b = (i * utts_per_step + u) % BATCH
            cpu_port_step(sd, snr_sd, waves[b:b + 1], Z)
    for i in range(warmup):
        step(i)
    t0 = time.perf_counter()
    for i in range(steps):
        step(warmup + i)
    dt = time.perf_counter() - t0
    sample = (f"{utts_per_step} of the 16 utterances per step, {steps} timed steps; CPU port of the reference path (oracle/) "
              f"because the reference itself was unavailable: {r['unavailable']}")
    return steps * utts_per_step * SECONDS / dt, dt, cores, "port", sample, _cpu_model()


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    total = args.steps + args.warmup
    # ~1.4 s per 4 s utterance on 16 cores: keep the whole run near two to three minutes
    upt = max(1, min(BATCH, int(150.0 / (1.4 * max(1, total)))))
    value, dt, cores, kind, sample, cpu = reference_cpu(args.steps, args.warmup, upt)
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=1e3 * dt / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="f32", data="synthetic", impl="reference", config=config_dict(args.gpus),
                implementation="unmodified reference, NCSN++ on the host CPU (fp32, all host threads)" if kind == "reference"
                else "CPU port of the reference path (oracle/)",
                ms_per_step_note=f"one step here = the bounded sample ({upt} of the 16 utterances); a full 16-utterance step "
                                 f"takes {BATCH / upt:g}x as long",
                cpu_model=cpu, cpu_baseline=dict(value=value, unit=UNIT, cores=cores, kind=kind, sample=sample),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------- B200 arm
def build_models(device, with_estimator=True, fixed_snr=None):
    """Score model + SNR estimator with seeded synthetic weights, packed on `device`.  with_estimator=False: another
    score model that shares the process-wide estimator already installed (sgmse.model.set_snr_model)."""
    from snr_aligned_diffse_b200.sgmse import model as sg_model
    from snr_aligned_diffse_b200.sgmse.model import ScoreModel
    from snr_aligned_diffse_b200.sgmse.snr_estimator import SNRModel
    from snr_aligned_diffse_b200.synth import synth_state_dict
    model = ScoreModel(backbone="ncsnpp", sde="ouve", model_type="sebridge_v3", snr_conditioned="true",
                       fixed_snr=FIXED_SNR if fixed_snr is None else fixed_snr, theta=1.5, sigma_min=0.05, sigma_max=1.0,
                       base_dir="")
    model._error_loading_ema = True
    model.load_state_dict(synth_state_dict({"dnn." + k: v for k, v in model.dnn.param_shapes().items()}, seed=0))
    model.eval(no_ema=True)
    if not with_estimator:
        return model, sg_model.get_snr_model()
    est = SNRModel(base_dir="")
    est._error_loading_ema = True
    est.load_state_dict(synth_state_dict(est.dnn.engine.param_shapes(), seed=1))
    est.eval(no_ema=True)
    sg_model.set_snr_model(est)
    return model, est


def profile_roofline(model, pipe, y_dev, peaks):
    """Tensor-bound roofline of the implicit-GEMM convolution launches, CUDA events between launch groups on the launch
    stream.  Steady state: >= 2 s of back-to-back graph replays, then five profiled passes with 10 replays between them
    (the board settles on its power-capped clock); idle start: the same pass after 1 s of idle (boost clocks)."""
    import torch
    aux = model.enhance_batch(y_dev, oracle=False, return_aux=True)[1]
    eng = model.dnn.engine
    X, Y, t = aux["X_T"], aux["Y"], aux["t"]
    eng.profile_forward(X, Y, t, mode=1)                                     # warm (plans, attributes)
    torch.cuda.synchronize()

    def summarise(prof):
        gemm = [p for p in prof if p["kind"] == 1]
        return dict(g_ms=sum(p["ms"] for p in gemm), g_fl=sum(p["flops"] for p in gemm), n=len(gemm),
                    tot_ms=sum(p["ms"] for p in prof), prof=prof)

    t0 = time.perf_counter()
    while time.perf_counter() - t0 < 2.0:
        for _ in range(10):
            pipe.replay()
        torch.cuda.synchronize()
    passes = []
    for _ in range(5):
        for _ in range(10):
            pipe.replay()
        passes.append(summarise(eng.profile_forward(X, Y, t, mode=1)))
    passes.sort(key=lambda q: q["g_ms"])
    steady = passes[len(passes) // 2]
    time.sleep(1.0)
    burst = summarise(eng.profile_forward(X, Y, t, mode=1))

    sustained = float(peaks.get("bf16_tflops_sustained", 1400.0))
    burst_peak = float(peaks.get("bf16_tflops", 1650.0))
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    src = "MEASURED_PEAKS.json" if peaks else "fallback (B200_PROFILING.md)"
    achieved = steady["g_fl"] / (steady["g_ms"] * 1e-3) / 1e12
    achieved_b = burst["g_fl"] / (burst["g_ms"] * 1e-3) / 1e12
    names = {0: "other", 1: "conv_gemm_tcgen05", 2: "groupnorm_silu", 3: "fir", 4: "attention", 5: "thin_conv",
             6: "pack_temb_head"}
    by_kind = {}
    for p in steady["prof"]:
        d = by_kind.setdefault(names[p["kind"]], dict(ms=0.0, launches=0, bytes=0.0))
        d["ms"] += p["ms"]; d["launches"] += 1; d["bytes"] += p["bytes"]
    for d in by_kind.values():
        d["ms"] = round(d["ms"], 4)
        d["share"] = round(d["ms"] / steady["tot_ms"], 4)
        by = d.pop("bytes")
        d["algo_GBps"] = round(by / (d["ms"] * 1e-3) / 1e9, 1) if d["ms"] > 0 else None
        d["frac_of_hbm"] = round(d["algo_GBps"] / hbm, 3) if d["algo_GBps"] else None
    traffic, traffic_note = None, None
    try:   # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture (profiles/)
        cap = json.load(open(os.path.join(ROOT, "profiles", "r02_conv_halo2_ncu.json")))
        c = cap["gn_silu_in_flight"]
        traffic = int(c["dram_bytes_read"] + c["dram_bytes_write"])
        traffic_note = (f"bytes per launch of {cap['shape']}; algorithmic bytes of that launch "
                        f"{cap['algorithmic_bytes']}; tensor pipe active {c['tensor_subpipe_hmma_cycles_active_pct']} %")
    except Exception:
        pass
    return dict(bound="tensor", kernel="conv_halo2_kernel (3x3, W>=8) + conv_gemm_kernel (1x1 / NIN / 4x8 maps)",
                achieved=round(achieved, 2), peak=sustained, unit="TFLOP/s", frac=round(achieved / sustained, 4),
                state="steady (>= 2 s of back-to-back steps before and between the profiled passes; median of 5)",
                peak_source=f"{src} bf16_tflops_sustained (cuBLAS bf16 back to back for 4 s)",
                idle_start=dict(achieved=round(achieved_b, 2), peak=burst_peak, frac=round(achieved_b / burst_peak, 4),
                                peak_source=f"{src} bf16_tflops (burst, best of 10)",
                                frac_of_sustained=round(achieved_b / sustained, 4)),
                traffic=traffic, traffic_note=traffic_note, launches_per_step=steady["n"],
                avg_launch_ms=round(steady["g_ms"] / max(1, steady["n"]), 4),
                algorithmic_tflop_per_step=round(steady["g_fl"] / 1e12, 3),
                flop_note="input conv booked at its algorithmic K = 9 x 4 (runs on a zero-padded 64-channel hi/lo tile)",
                kernel_share_of_network=round(steady["g_ms"] / steady["tot_ms"], 4), hbm_peak_GBps=hbm,
                network_ms_profiled=round(steady["tot_ms"], 3), by_kind=by_kind)


def parity_check(model, y_dev, host_in, out_dev):
    """Utterance 0 of the timed batch against the CPU oracle, outside the timed region: the graph's output must be finite
    everywhere, and a pass with an explicit noise draw must match the oracle's waveform (SI-SDR >= 30 dB)."""
    import numpy as np
    import torch
    from oracle import sampler as o_sampler, snrnet as o_snrnet
    from oracle.topology import NCSNppConfig, param_specs, snrnet_param_specs
    from snr_aligned_diffse_b200.synth import synth_noise, synth_state_dict
    finite = bool(torch.isfinite(out_dev).all().item())
    Z = synth_noise(BATCH, 512, seed=77)
    out, aux = model.enhance_batch(y_dev, oracle=False, noise=Z, return_aux=True)
    torch.set_num_threads(os.cpu_count() or 1)
    sd = synth_state_dict(param_specs(NCSNppConfig()), seed=0)
    snr_sd = synth_state_dict(snrnet_param_specs(), seed=1)
    with torch.no_grad():
        ratio = float(o_snrnet.estimate_noise_over_clean(snr_sd, host_in[:1])[0, 0])
        o = o_sampler.enhance_v3(sd, host_in[:1], Z[:1], ratio, FIXED_SNR, sigma_max=1.0)
    ref = o["x_hat"].numpy().astype(np.float64)
    got = out[0].cpu().numpy().astype(np.float64)
    sdr = o_sampler.si_sdr(ref, got)
    mx = float(np.abs(got - ref).max() / np.abs(ref).max())
    ok = finite and bool(np.isfinite(got).all()) and sdr >= 30.0 and int(aux["t_index"][0]) == o["t_index"]
    return dict(ok=ok, finite=finite, si_sdr_db_vs_oracle=round(sdr, 2), maxabs_of_peak=round(mx, 4),
                t_index_equal=int(aux["t_index"][0]) == o["t_index"], bound="SI-SDR >= 30 dB, finite, same t_30 index",
                checked="utterance 0 of the timed batch, explicit noise draw, CPU oracle (outside the timed region)")


def run_b200(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from snr_aligned_diffse_b200 import _lib
    lib = _lib.load()
    _lib.require_device()          # no CUDA extension / no B200 -> fail loudly, there is no fallback
    model, est = build_models(dev)

    L = int(SECONDS * SR)
    host_in = synth_waves(BATCH, L, seed=1000 + rank).pin_memory()
    host_out = torch.empty(BATCH, L, dtype=torch.float32).pin_memory()
    y_dev = host_in.to(dev)
    stream = torch.cuda.Stream(device=dev)

    from snr_aligned_diffse_b200.pipeline import GraphedEnhancer

    def noise_generator(k):
        # a seeded generator per enhancer: the enhancers' replays overlap, and graphs that share torch's default generator
        # would read each other's noise offsets (pipeline.GraphedEnhancer)
        return torch.Generator(device=dev).manual_seed(100 * rank + k)

    pipe = GraphedEnhancer(model, BATCH, L, dev, oracle=False, stream=stream, generator=noise_generator(0))
    pipe.y_dev.copy_(y_dev)
    y_dev = pipe.y_dev
    # --streams 2: a second, independent enhancer (own network workspace, own streams); consecutive steps alternate
    # between the two so that the small kernels of one batch (grids below 148 CTAs on the 32x64 and smaller maps, the
    # front end, the SNR estimator, the iSTFT) overlap the other batch's work.  Every step is still one full pass over
    # one batch of 16 utterances.
    pipes = [pipe]
    for k in range(1, args.streams):
        model2, _ = build_models(dev, with_estimator=False)   # the estimator (weights, read-only) is shared
        pipe2 = GraphedEnhancer(model2, BATCH, L, dev, oracle=False, generator=noise_generator(k))
        pipe2.y_dev.copy_(y_dev)
        with torch.cuda.stream(pipe2.stream):
            pipe2._step()
            pipe2.capture(warmup=1)
            pipe2.stream.synchronize()
        pipes.append(pipe2)

    with torch.cuda.stream(stream):
        pipe._step()                           # first eager pass: packs weights, builds the plan
        stream.synchronize()
        n0 = lib.snrse_launch_count()
        pipe.capture(warmup=1)
        launches_per_step = int(lib.snrse_launch_count() - n0) // 2     # one eager warm-up + the captured pass
        W = max(args.warmup, 3)
        for _ in range(W):
            for p in pipes:
                p.replay()
        torch.cuda.synchronize()

        def barrier():
            stream.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        def timed(body, flush=False):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for p in pipes[1:]:
                p.stream.wait_event(e0)                    # the other enhancer's stream starts inside the timed region
            for i in range(args.steps):
                body(i)
            if flush:
                for p in pipes:
                    p.flush()                              # the last read-backs are inside the timed region
            for p in pipes[1:]:
                stream.wait_stream(p.stream)               # ... and ends inside it
            e1.record(stream)
            barrier()
            ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            return float(ms.item())

        clocks = ClockSampler(local) if rank == 0 else None
        # the three timed regions run back to back (no idle gaps between them): W warm-up steps above, then K steps each
        ms_dev = timed(lambda i: pipes[i % len(pipes)].replay())
        # the enhanced batch of the last timed step; later regions overwrite the enhancers' output buffers
        last_out = pipes[(args.steps - 1) % len(pipes)].out_dev.clone() if args.dump_outputs else None
        ms_single = timed(lambda i: pipes[0].replay()) if len(pipes) > 1 else ms_dev

        host_outs = [host_out] + [torch.empty_like(host_out).pin_memory() for _ in pipes[1:]]

        def e2e_body(i=0):
            # the package's host-buffer API: pinned host -> device copy of this step's inputs, graph replay, device ->
            # pinned host copy of this step's result; copies run on a second stream and overlap the neighbouring steps
            k = i % len(pipes)
            pipes[k].enhance_host(host_in, host_outs[k])

        for i in range(4):
            e2e_body(i)
        for p in pipes:
            p.flush()
        ms_e2e = timed(e2e_body, flush=True)
        e2e_finite = bool(torch.isfinite(host_outs[0]).all().item())

        # ---- sustained figure: the same alternating replay for >= 2 s (every rank, so the clocks line sees load)
        barrier()
        nv, j0 = None, None
        if rank == 0:                      # board energy over the sustained region (NVML total-energy counter, mJ)
            try:
                import pynvml
                pynvml.nvmlInit()
                nv = pynvml.nvmlDeviceGetHandleByIndex(torch.cuda._get_nvml_device_index(local) if hasattr(torch.cuda, "_get_nvml_device_index") else local)
                j0, tj0 = pynvml.nvmlDeviceGetTotalEnergyConsumption(nv), time.perf_counter()
            except Exception:
                nv = None
        n_sus, e0, e1 = 0, torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for p in pipes[1:]:
            p.stream.wait_event(e0)
        n_target = max(args.steps, int(2200.0 / max(1e-3, ms_dev / args.steps)))
        for i in range(n_target):
            pipes[i % len(pipes)].replay()
            n_sus += 1
        for p in pipes[1:]:
            stream.wait_stream(p.stream)
        e1.record(stream)
        barrier()
        energy = None
        if nv is not None:
            try:
                joule = (pynvml.nvmlDeviceGetTotalEnergyConsumption(nv) - j0) * 1e-3
                energy = dict(J_per_step=round(joule / n_sus, 3), avg_watts=round(joule / (time.perf_counter() - tj0), 1),
                              steps=n_sus, source="NVML total-energy counter over the sustained region, rank 0's GPU",
                              note="the sustained region sits at the board's power cap (clocks.reasons: sw_power_cap): time per "
                                   "step ~ Joules per step / cap.  tools/energy_bench.py (profiles/r02_energy.md): cuBLAS bf16 "
                                   "8192^3 under the same cap 0.70 pJ/FLOP at 1386 TFLOP/s, idle board 258 W")
            except Exception:
                energy = None
        ms_sus = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms_sus, op=dist.ReduceOp.MAX)
        ms_sus = float(ms_sus.item())
        clk = clocks.stop() if clocks else None

        # ---- the r01 measurement for comparison: the same K alternating steps started from an idle GPU (boost clocks for
        # the first ~0.1 s before the power cap bites).  NOT the headline: `value` above is the steady state.
        time.sleep(1.0)
        saved_steps = args.steps
        args.steps = min(args.steps, 10)
        ms_idle = timed(lambda i: pipes[i % len(pipes)].replay())
        idle_steps = args.steps
        args.steps = saved_steps

        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        roof = profile_roofline(model, pipe, y_dev, peaks) if rank == 0 else None
        if energy and roof:
            energy["pJ_per_algorithmic_FLOP"] = round(energy["J_per_step"] / roof["algorithmic_tflop_per_step"], 4)
        parity = None
        if rank == 0:
            pipe.replay()
            stream.synchronize()
            parity = parity_check(model, y_dev, host_in, pipe.out_dev)
            parity["e2e_output_finite"] = e2e_finite

    audio_s = world * BATCH * SECONDS * args.steps
    value = audio_s / (ms_dev * 1e-3)
    e2e_value = audio_s / (ms_e2e * 1e-3)

    # ---- BASELINE configs 3-5 + the 60-NFE PC loop at this N (all ranks take part)
    extras = {}
    if not args.no_extras:
        del pipes, pipe
        torch.cuda.empty_cache()
        from snr_aligned_diffse_b200 import workloads as wl
        torch.cuda.set_stream(torch.cuda.default_stream(dev))
        try:
            sweeps = {}
            for fs in (0.17783, 0.31623, 0.56234):
                model.fixed_snr = fs
                r = wl.run_sweep824(model, dev, rank, world, repeat=3)
                sweeps[str(fs)] = dict(value=round(r["value"], 1), job_seconds=round(r["job_seconds"], 4), finite=r["finite"],
                                       batches_rank0=r["batches_rank0"])
            model.fixed_snr = FIXED_SNR
            extras["sweep824"] = dict(metric="enhanced audio-sec/sec, 824 VoiceBank-DEMAND-shaped utterances (1.5-10 s), "
                                             "SNR estimator in the loop", unit=UNIT, scaling="strong", n_gpus=world,
                                      utterances=r["utterances"], audio_seconds=round(r["audio_seconds"], 1),
                                      value=sweeps["0.17783"]["value"], by_fixed_snr=sweeps, mode=r["mode"],
                                      sharding="equal-Tpad batches of <= 16 assigned to ranks by LPT on a fitted per-batch cost")
            r = wl.run_longform60(model, dev, rank, world, count=2, repeat=3)
            extras["longform60"] = dict(metric="enhanced audio-sec/sec, 60 s utterances (Tpad 7552), batch 1", unit=UNIT,
                                        scaling="weak", n_gpus=world, utterances=r["utterances"], value=round(r["value"], 1),
                                        ms_per_utterance=round(1e3 * r["job_seconds"] / 2, 2), finite=r["finite"])
            model.dnn.engine._ws.clear()
            model.dnn.engine.__dict__.pop("_arena", None)
            torch.cuda.empty_cache()
            r = wl.run_pc60(dev, rank, world, batch=BATCH, seconds=SECONDS, enhancers=2, reps=1)
            extras["pc60"] = dict(metric="enhanced audio-sec/sec, PC sampler 60 NFE (N=30, reverse diffusion + ALD), 16 x 4 s per GPU",
                                  unit=UNIT, n_gpus=world, **{k: (round(v, 1) if k == "value" else v) for k, v in r.items()})
        except Exception as ex:                       # an extra must never take the headline down with it
            extras["error"] = f"{type(ex).__name__}: {str(ex)[:300]}"

    if args.dump_outputs:
        # inputs, weights and noise draws (seeded per enhancer) are identical from run to run for the same arguments
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, f"enhanced_rank{rank}.npy"), last_out.cpu().numpy())

    if rank == 0:
        cpu, eager = None, None
        if world == 1 and not args.no_cpu_baseline:
            v, dt, cores, kind, sample, cpum = reference_cpu(steps=4, warmup=1, utts_per_step=2)
            cpu = dict(value=v, unit=UNIT, cores=cores, kind=kind, cpu_model=cpum, sample=sample)
        if world == 1 and not args.no_eager_baseline:
            torch.cuda.empty_cache()
            r = _run_ref_runner(["--task", "eager_gpu", "--batch", str(BATCH), "--seconds", str(SECONDS), "--seed", "1000",
                                 "--precision", "fp32,tf32,fp16,bf16", "--reps", "5"], 900)
            if "unavailable" in r:
                eager = r
            else:
                eager = dict(what="UNMODIFIED reference (baseline/_ref) in torch eager mode on this GPU, same 16 x 4 s inputs, "
                                  "its own stft / SNRNet / ScoreModel.forward / to_audio composed for a batch (model.py:713-830)",
                             torch=r["torch"], cudnn=r["cudnn"], unit=UNIT, modes=r["results"],
                             mode_notes=dict(fp32="torch defaults: cuDNN convolutions may use TF32, matmuls fp32",
                                             tf32="additionally torch.backends.cuda.matmul.allow_tf32",
                                             fp16="torch.autocast(float16) around ScoreModel.forward",
                                             bf16="torch.autocast(bfloat16) around ScoreModel.forward; the unmodified reference "
                                                  "cannot run it (upfirdn2d CUDA op and view_as_complex reject bf16), so two "
                                                  "upcast wrappers in baseline/ref_runner.py are active (reference files untouched)"))
                best = max((m.get("audio_s_per_s", 0.0) for m in r["results"].values()), default=0.0)
                eager["best_value"] = best
                eager["speedup_e2e_over_best_eager"] = round(e2e_value / best, 2) if best else None
        line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=W,
                    ms_per_step=ms_dev / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="bf16",
                    data="synthetic", config=config_dict(world),
                    implementation=dict(graph="one CUDA graph per step", enhancers_per_gpu=args.streams,
                                        accumulate="fp32", storage="bf16 activations",
                                        note="value / e2e: K steps alternate over two independent enhancers on two streams; "
                                             "latency: the same K steps strictly back to back through one enhancer"),
                    e2e=dict(value=e2e_value, unit=UNIT, ms_per_step=ms_e2e / args.steps,
                             h2d_bytes_per_step=int(host_in.numel() * 4), d2h_bytes_per_step=int(host_out.numel() * 4)),
                    latency=dict(ms_per_step_single_enhancer=ms_single / args.steps,
                                 value_single_enhancer=audio_s / (ms_single * 1e-3), unit=UNIT,
                                 note="per-step latency of the full pass (NCSN++ forward is ~97 % of it), one enhancer, "
                                      "steps back to back"),
                    sustained=dict(steps=n_sus, seconds=round(ms_sus * 1e-3, 3), ms_per_step=ms_sus / n_sus,
                                   value=world * BATCH * SECONDS * n_sus / (ms_sus * 1e-3), unit=UNIT,
                                   note="same alternating replay kept up for >= 2 s (power-capped steady state)"),
                    idle_start=dict(steps=idle_steps, ms_per_step=ms_idle / idle_steps,
                                    value=world * BATCH * SECONDS * idle_steps / (ms_idle * 1e-3), unit=UNIT,
                                    note="same alternating replay after 1 s of idle (boost clocks until the power cap bites): "
                                         "how r01 measured its 17.6 ms; for comparison only"),
                    gpu_launches=launches_per_step * args.steps, launches_per_step=launches_per_step,
                    clocks=clk, energy=energy, roofline=roof, parity=parity, cpu_baseline=cpu, gpu_eager_baseline=eager, impl="b200",
                    **extras)
        print(json.dumps(line), flush=True)
        if parity is not None and not parity["ok"]:
            print("bench.py: PARITY CHECK FAILED: " + json.dumps(parity), file=sys.stderr, flush=True)
            sys.exit(3)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the sweep824 / longform60 / pc60 sub-records")
    ap.add_argument("--streams", type=int, default=2, choices=[1, 2, 3, 4],
                    help="independent enhancers per GPU whose steps alternate (2: small kernels of one batch overlap the other batch)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the enhanced waveforms [16, 64000] of the last timed step as DIR/enhanced_rank<R>.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
