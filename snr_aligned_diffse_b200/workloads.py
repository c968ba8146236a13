"""BASELINE.json configs 3-5 and the 60-NFE predictor-corrector loop as functions over an existing process group
(bench.py prints them as sub-records of its JSON line at every N; tools/sweep_bench.py is the stand-alone CLI).

  sweep824   824 synthetic VoiceBank-DEMAND-test-shaped utterances (1.5-10 s, SURVEY 8d config 3), equal-Tpad batches
             of <= 16 assigned to the ranks by LPT (`shard.batch_shards`), SNR estimator in the loop; config 4 = the
             same at fixed_snr 0.17783 / 0.31623 / 0.56234.  STRONG scaling: the list is fixed, ranks share it.
  longform60 60 s utterances (config 5), `count` per rank, batch 1.  Weak scaling.
  pc60       OUVE score model on the same NCSN++, eval.py PC defaults (N=30, reverse diffusion + 1 annealed-Langevin
             step = 60 network evaluations) on 16 x 4 s per rank, the whole loop replayed from one CUDA graph.  Weak.

All timings are device timings (CUDA events on the launching stream, synchronised on both sides), max over ranks.
No data-path collective anywhere: torch.distributed only carries the barrier, the max-over-ranks and the metric gather.
"""
import torch

from .shard import batch_shards, synthetic_lengths
from .sweep import enhance_sweep, gather_metrics
from .synth import synth_waves

SR = 16000
SWEEP_TARGET_FRAMES = 16384     # padded frames per batch of the 824-utterance sweep (two bench-shape batches' worth)


def synth_wave(length, seed):
    """One synthetic utterance of `length` samples (pitch, envelope and noise level vary with the seed)."""
    g = torch.Generator().manual_seed(seed)
    t = torch.arange(length) / SR
    f0 = 100.0 + (seed % 37) * 5.0
    speech = sum(torch.sin(2 * torch.pi * f0 * (k + 1) * t + k) / (k + 1) for k in range(5))
    env = 0.5 + 0.5 * torch.sin(2 * torch.pi * (1.5 + 0.01 * (seed % 50)) * t)
    return (0.1 * speech * env + (0.01 + 0.0005 * (seed % 40)) * torch.randn(length, generator=g)).float()


def _dist():
    import torch.distributed as dist
    return dist if dist.is_available() and dist.is_initialized() else None


def _barrier(dev):
    torch.cuda.synchronize(dev)
    d = _dist()
    if d is not None:
        d.barrier()
    torch.cuda.synchronize(dev)


def _max_over_ranks(ms, dev):
    v = torch.tensor([ms], dtype=torch.float64, device=dev)
    d = _dist()
    if d is not None:
        d.all_reduce(v, op=d.ReduceOp.MAX)
    return float(v.item())


def run_utterance_sweep(model, waves, dev, rank, world, max_batch=16, graphs=True, repeat=2, target_frames=None):
    """Enhance the list `waves` (sharded over the ranks) `repeat` times; the LAST pass is timed.  Pass 1 builds the
    plans and, with graphs=True, captures one CUDA graph per batch shape (all Tpad buckets are therefore captured before
    the clock of the timed pass starts).  Returns dict(job_seconds, audio_seconds, utterances, batches_rank0, finite)."""
    from .pipeline import GraphedEnhancerCache
    lengths = [int(w.numel()) for w in waves]
    mine = batch_shards(lengths, world, max_batch, target_frames=target_frames)[rank]
    model.dnn._ensure_device_weights()
    if mine:
        need = max(model.dnn.engine.workspace_bytes(len(idx), 256, tpad) for tpad, idx in mine)
        model.dnn.engine.reserve(need)            # one activation arena for all buckets: the largest (batch, Tpad)
    fn = GraphedEnhancerCache(model, dev, min_uses=1, oracle=False) if graphs else (
        lambda y, lens: model.enhance_batch(y, lengths=lens, oracle=False))
    res = None
    for _ in range(max(1, repeat)):
        _barrier(dev)
        res = enhance_sweep(fn, waves, rank=rank, world=world, max_batch=max_batch, device=dev, target_frames=target_frames)
    allm = gather_metrics(res, world)
    audio_s = sum(allm["samples"]) / SR
    return dict(job_seconds=allm["job_seconds"], audio_seconds=audio_s, utterances=len(allm["ids"]),
                batches_rank0=res["batches"], finite=all(c == c for c in allm["checksum"]),
                value=audio_s / allm["job_seconds"])


def run_sweep824(model, dev, rank, world, count=824, max_batch=16, graphs=True, repeat=2, target_frames=SWEEP_TARGET_FRAMES):
    lengths = synthetic_lengths(count, seed=0)
    waves = [synth_wave(int(l), seed=i) for i, l in enumerate(lengths)]
    out = run_utterance_sweep(model, waves, dev, rank, world, max_batch, graphs, repeat, target_frames or None)
    out.update(scaling="strong", fixed_snr=float(model.fixed_snr), max_batch=max_batch, target_frames=target_frames,
               mode=("one CUDA graph per batch shape, all captured in the untimed first pass" if graphs
                     else "eager launches"))
    return out


def run_longform60(model, dev, rank, world, count=2, graphs=True, repeat=2):
    waves = [synth_wave(60 * SR, seed=i) for i in range(count * world)]
    out = run_utterance_sweep(model, waves, dev, rank, world, 1, graphs, repeat)
    out.update(scaling="weak", seconds_per_utterance=60.0, per_rank=count, tpad=7552)
    return out


def run_pc60(dev, rank, world, batch=16, seconds=4.0, enhancers=2, reps=1, N=30, graph=True):
    """60-NFE predictor-corrector loop (bbed-style score head on the OUVE SDE) on `batch` x `seconds` per rank;
    `enhancers` independent batches in flight per GPU (own executor + arena), each loop one CUDA graph."""
    from . import ops
    from .sgmse.model import ScoreModel
    from .synth import synth_state_dict
    n_enh = max(1, enhancers) if graph else 1
    L = int(seconds * SR)
    peaks, samplers = [], []
    keep = []
    for e in range(n_enh):
        model = ScoreModel(backbone="ncsnpp", sde="ouve", model_type="bbed", snr_conditioned="false", theta=1.5,
                           sigma_min=0.05, sigma_max=0.5, N=N, base_dir="")
        model._error_loading_ema = True
        model.load_state_dict(synth_state_dict({"dnn." + k: v for k, v in model.dnn.param_shapes().items()}, seed=0))
        model.eval(no_ema=True)
        y = synth_waves(batch, L, seed=2000 + rank + 100 * e).to(dev)
        peak = ops.absmax(y)
        Y = ops.stft(y, scale=peak, scale_is_divisor=True)[:, None]
        sampler = model.get_pc_sampler("reverse_diffusion", "ald", Y, N=N, corrector_steps=1, snr=0.5, graph=bool(graph))
        sampler()                                       # warm-up: plans, weights, graph capture
        keep.append((model, Y))
        peaks.append(peak)
        samplers.append(sampler)
    _barrier(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    main_s = torch.cuda.current_stream(dev)
    side = [torch.cuda.Stream(device=dev) for _ in samplers]   # one caller stream per enhancer
    e0.record(main_s)
    for st in side:
        st.wait_stream(main_s)
    nfe = 0
    for _ in range(max(1, reps)):
        x_hats = []
        for sm, st, pk in zip(samplers, side, peaks):   # graph mode: each call only enqueues; the loops run concurrently
            with torch.cuda.stream(st):
                o, nfe = sm()
                x_hats.append(ops.istft(o[:, 0].contiguous(), L, scale=pk))
    for st in side:
        main_s.wait_stream(st)
    e1.record(main_s)
    _barrier(dev)
    sec = _max_over_ranks(e0.elapsed_time(e1), dev) * 1e-3 / (max(1, reps) * n_enh)
    finite = all(bool(torch.isfinite(x).all()) for x in x_hats)
    del keep
    return dict(value=world * batch * seconds / sec, nfe=int(nfe), ms_per_batch=round(sec * 1e3, 2),
                ms_per_nfe=round(sec * 1e3 / max(1, nfe), 3), batch=batch, seconds_per_utterance=seconds,
                enhancers_per_gpu=n_enh, finite=finite, scaling="weak",
                mode=(f"whole {N}-step loop (corrector + predictor per step) replayed from ONE CUDA graph, {n_enh} "
                      "independent batches in flight per GPU") if graph else "host loop, eager launches")
