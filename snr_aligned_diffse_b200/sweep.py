"""Multi-utterance / multi-GPU enhancement driver (SURVEY 8e, 8f-1; BASELINE configs 3-5).

The reference enhances one utterance per `ScoreModel.enhance` call (B/eval.py:119-132).  Utterances are
independent (per-utterance normalisation, per-sample GroupNorm / attention), so a list is
  1. grouped into equal-Tpad batches (`shard.bucket_batches`),
  2. the batches partitioned over the ranks by LPT on a per-batch cost (`shard.batch_shards`),
  3. enhanced batch by batch with `ScoreModel.enhance_batch` (ragged lengths inside a batch),
with NO collective on the data path.  Only the per-utterance metrics (id, samples, checksum, SI-SDR) and the
rank timings are gathered at the end (`torch.distributed`: NCCL on GPUs, gloo in the CPU tests).
"""
import time

import torch

from .shard import HOP, batch_shards


def pack_batch(waves, idx, tpad, pin=False):
    """Zero-padded batch [len(idx), 128*tpad - 1] + int32 lengths for utterances `idx` of one Tpad bucket.
    The buffer length is the longest waveform with `tpad` padded frames (1 + L//128 <= tpad), so it depends on the
    bucket only and every batch of a bucket has the same shape."""
    lbuf = HOP * tpad - 1
    # pinned staging (torch's caching host allocator recycles the blocks): the host -> device copy of this batch is then
    # truly asynchronous and overlaps the previous batch's kernels
    y = torch.zeros(len(idx), lbuf, dtype=torch.float32, pin_memory=pin)
    lens = torch.empty(len(idx), dtype=torch.int32, pin_memory=pin)
    for r, i in enumerate(idx):
        w = waves[i].reshape(-1)
        y[r, :w.numel()] = w
        lens[r] = w.numel()
    return y, lens


def enhance_sweep(enhance_fn, waves, rank=0, world=1, max_batch=16, device=None, keep_audio=False, references=None,
                  on_audio=None, target_frames=None, keys=None, seed=None):
    """Enhance the utterances `waves` (list of 1-D float tensors) this rank owns.

    enhance_fn(y [B, L] , lengths [B] int32) -> enhanced [B, L] (e.g. `lambda y, n: model.enhance_batch(y, lengths=n)`).
    references: optional list of clean waveforms (same lengths): adds the per-utterance SI-SDR in dB, computed on the
    device (`ops.si_sdr`; the reference computes it on host numpy arrays per file, B/eval.py:140-144).
    target_frames: batches of about that many padded frames instead of at most `max_batch` utterances (`shard.bucket_batches`).
    on_audio(i, waveform): optional sink called with every enhanced utterance (host tensor) right after its batch, while
    the following batches are still being enqueued (used by `wavio.enhance_files` to write wavs off the critical path).
    seed: keyed noise.  enhance_fn is then called as enhance_fn(y, lengths, keys [B] int64, seed), e.g.
    `lambda y, n, k, s: model.enhance_batch(y, lengths=n, keys=k, seed=s)` or a `pipeline.GraphedEnhancerCache`, with
    keys[i] (default: i, the utterance's index in `waves`; 64-bit ints) for utterance i, so that every utterance's
    result depends on its samples, its key and the seed only -- not on the batching, the rank count or its neighbours.
    Returns dict(ids, samples, checksum, si_sdr, seconds, batches, audio) for this rank's shard."""
    lengths = [int(w.numel()) for w in waves]
    if seed is not None:
        from .ops import key_tensor
        all_keys = key_tensor(range(len(waves)) if keys is None else keys, len(waves))
    elif keys is not None:
        raise ValueError("enhance_sweep: keys need a seed")
    batches = batch_shards(lengths, world, max_batch, target_frames=target_frames)[rank]
    ids, samples, checks, sdrs, audio = [], [], [], [], {}
    on_gpu = device is not None and torch.device(device).type == "cuda"
    if on_gpu:       # device timing of the whole shard (host packing gaps included), on the stream the work is launched on
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(torch.cuda.current_stream(device))
    t0 = time.perf_counter()
    # host packing runs a few batches ahead of the launches on two worker threads (the copies release the GIL), so the
    # GPU never waits for the host to zero-pad the next batch; intra-op threading is switched off meanwhile (a 16-thread
    # OpenMP pool spinning between 100 us copies slowed the packing 4x on a box whose cores were shared by two ranks)
    import collections
    import concurrent.futures
    prev_threads = torch.get_num_threads()
    torch.set_num_threads(1)
    pool = concurrent.futures.ThreadPoolExecutor(max_workers=2)
    ahead, nxt = collections.deque(), 0
    depth = 6

    def refill():
        nonlocal nxt
        while nxt < len(batches) and len(ahead) < depth:
            tp, ix = batches[nxt]
            ahead.append(pool.submit(pack_batch, waves, ix, tp, on_gpu))
            nxt += 1
    try:
        refill()
        for tpad, idx in batches:
            y, lens = ahead.popleft().result()
            refill()
            if device is not None:
                y, lens = y.to(device, non_blocking=True), lens.to(device, non_blocking=True)
            if seed is None:
                out = enhance_fn(y, lens)
            else:
                kt = all_keys[list(idx)]
                out = enhance_fn(y, lens, kt if device is None else kt.to(device, non_blocking=True), seed)
            pos = torch.arange(out.shape[1], device=out.device)[None, :]
            valid = pos < lens.to(out.device)[:, None].to(pos.dtype)
            cs = (out.double() * valid).sum(1)            # per-utterance checksum over the valid samples only
            for r, i in enumerate(idx):
                ids.append(i)
                samples.append(lengths[i])
            checks.append(cs)
            if references is not None:
                from . import ops
                x, _ = pack_batch(references, idx, tpad)
                sdrs.append(ops.si_sdr(x.to(out.device, non_blocking=True), out, lens.to(out.device)))
            if keep_audio or on_audio is not None:
                host = out.detach().to("cpu", non_blocking=False)     # one copy per batch
                for r, i in enumerate(idx):
                    a = host[r, :lengths[i]].clone()
                    if keep_audio:
                        audio[i] = a
                    if on_audio is not None:
                        on_audio(i, a)
    finally:
        pool.shutdown(wait=True)
        torch.set_num_threads(prev_threads)
    if on_gpu:
        ev1.record(torch.cuda.current_stream(device))
        torch.cuda.synchronize(device)
    wall = time.perf_counter() - t0
    seconds = ev0.elapsed_time(ev1) * 1e-3 if on_gpu else wall
    checksum = torch.cat(checks).cpu().tolist() if checks else []
    si_sdr = torch.cat(sdrs).cpu().tolist() if sdrs else [float("nan")] * len(ids)
    return dict(ids=ids, samples=samples, checksum=checksum, si_sdr=si_sdr, seconds=seconds, wall_seconds=wall,
                batches=len(batches), audio=audio)


def gather_metrics(local, world=1):
    """All ranks' (id, samples, checksum) rows sorted by id + the slowest rank's wall time (the job time).
    The only communication of the sweep (a few KB)."""
    sdr = local.get("si_sdr") or [float("nan")] * len(local["ids"])
    rows = torch.tensor([[float(i), float(n), float(c), float(q)]
                         for i, n, c, q in zip(local["ids"], local["samples"], local["checksum"], sdr)],
                        dtype=torch.float64).reshape(-1, 4)
    sec = torch.tensor([local["seconds"]], dtype=torch.float64)
    if world > 1:
        import torch.distributed as dist
        dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
        n = torch.tensor([rows.shape[0]], dtype=torch.int64, device=dev)
        counts = [torch.zeros_like(n) for _ in range(world)]
        dist.all_gather(counts, n)
        cap = int(max(int(c.item()) for c in counts))
        pad = torch.zeros(cap, 4, dtype=torch.float64, device=dev)
        pad[:rows.shape[0]] = rows.to(dev)
        parts = [torch.zeros_like(pad) for _ in range(world)]
        dist.all_gather(parts, pad)
        rows = torch.cat([p[:int(c.item())].cpu() for p, c in zip(parts, counts)])
        sec = sec.to(dev)
        dist.all_reduce(sec, op=dist.ReduceOp.MAX)
        sec = sec.cpu()
    order = torch.argsort(rows[:, 0])
    rows = rows[order]
    return dict(ids=rows[:, 0].long().tolist(), samples=rows[:, 1].long().tolist(), checksum=rows[:, 2].tolist(),
                si_sdr=rows[:, 3].tolist(), job_seconds=float(sec.item()))
