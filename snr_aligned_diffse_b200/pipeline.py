"""Graph-captured, copy-overlapped batch enhancement (SURVEY 8f-1: batched, sync-free `enhance`).

`ScoreModel.enhance` (sgmse/model.py) moves one utterance to the GPU, enhances it and copies it back, one call at
a time.  For fixed-shape batches `GraphedEnhancer` captures the whole sebridge_v3 pass (peak -> SNR estimate -> t / norm
factor -> STFT + transform -> X_T -> NCSN++ -> inverse transform + iSTFT) in one CUDA graph and runs the host <-> device
copies of consecutive batches on a second stream, so that the copy of batch i+1 and the read-back of batch i-1 overlap
the computation of batch i:

    compute stream : [y_dev <- y_stage] [graph replay] [out_stage <- out_dev]          per batch
    upload stream  : [y_stage <- pinned host input]
    read-back stream :                                        [pinned host output <- out_stage]

No host synchronisation inside `enhance_host`; `flush()` joins the two streams.

With keyed=True the noise is the keyed draw of `ScoreModel.enhance_batch(..., keys=, seed=)`: the per-row keys live in
a device buffer read by the captured graph, so new keys (`set_keys`) take effect at the next replay without a re-capture,
and every row's result is that utterance enhanced alone.
"""
import torch

from . import ops


class GraphedEnhancer:
    def __init__(self, model, batch, length, device, oracle=False, noise_over_clean=None, noise=None, stream=None,
                 ragged=False, generator=None, keyed=False, seed=0):
        self.model, self.batch, self.length, self.device = model, batch, length, torch.device(device)
        # generator: CUDA torch.Generator for this enhancer's noise draws.  Every graph that draws from torch's default
        # generator reads its seed / offset from one shared device slot, which each replay rewrites, so enhancers whose
        # replays overlap on different streams need a generator each for reproducible draws.
        self.generator = generator
        self.stream = stream or torch.cuda.Stream(device=self.device)
        # separate streams for the two copy directions: on one in-order stream the upload of batch i+1 would queue
        # behind the read-back of batch i, i.e. behind the end of batch i's computation
        self.copy_stream = torch.cuda.Stream(device=self.device)      # host -> device
        self.copy_stream_out = torch.cuda.Stream(device=self.device)  # device -> host
        self.y_dev = torch.zeros(batch, length, dtype=torch.float32, device=self.device)
        self.y_stage = torch.zeros_like(self.y_dev)
        self.out_stage = torch.zeros_like(self.y_dev)
        if noise_over_clean is not None:   # device-resident before capture (no host copy inside the graph)
            noise_over_clean = torch.as_tensor(noise_over_clean, dtype=torch.float32).reshape(-1).to(self.device)
        self._kw = dict(oracle=oracle, noise_over_clean=noise_over_clean, noise=noise,   # noise: fixed draw (tests)
                        generator=generator)
        # ragged: per-utterance valid lengths live in a device buffer read by the captured graph
        self.len_dev = torch.full((batch,), length, dtype=torch.int32, device=self.device) if ragged else None
        # keyed: per-row noise keys (int64, read as uint64) in a device buffer read by the captured graph; rows start
        # with distinct keys (their index) until `set_keys`
        self.key_dev = torch.arange(batch, dtype=torch.int64, device=self.device) if keyed else None
        if keyed:
            self._kw["seed"] = seed
        self.graph = None
        self.out_dev = None
        self._h2d_done = torch.cuda.Event()
        self._y_consumed = torch.cuda.Event()
        self._out_ready = torch.cuda.Event()
        self._d2h_done = torch.cuda.Event()
        self._first = True

    def _step(self):
        return self.model.enhance_batch(self.y_dev, lengths=self.len_dev, keys=self.key_dev, **self._kw)

    def set_keys(self, keys):
        """Write the per-row noise keys (`ops.key_tensor` forms) used by the following replays (keyed=True only).
        Ordered on this enhancer's stream, so a replay already enqueued keeps the keys it was launched with."""
        if self.key_dev is None:
            raise ValueError("set_keys: this enhancer was built without keyed=True")
        kt = ops.key_tensor(keys, self.batch)
        with torch.cuda.stream(self.stream):
            self.key_dev.copy_(kt, non_blocking=kt.is_cuda)

    def capture(self, warmup=2):
        """Eager warm-up (packs weights, builds the plan, sets function attributes), then graph capture."""
        with torch.cuda.stream(self.stream):
            for _ in range(warmup):
                self.out_dev = self._step()
            self.stream.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            if self.generator is not None:
                self.graph.register_generator_state(self.generator)
            with torch.cuda.graph(self.graph, stream=self.stream):
                self.out_dev = self._step()
        return self

    def replay(self):
        """One pass over the batch resident in `y_dev` on this enhancer's stream; result in `out_dev` (device)."""
        with torch.cuda.stream(self.stream):
            self.graph.replay()
        return self.out_dev

    def enhance_host(self, host_in, host_out, keys=None):
        """Enqueue one batch: pinned `host_in` [B, L] -> enhanced pinned `host_out` [B, L].  Returns immediately;
        `host_out` is valid after `flush()` (or once the next call's read-back has been ordered behind it).
        keys: optional per-row noise keys for this batch (keyed=True)."""
        cs, co, ms = self.copy_stream, self.copy_stream_out, self.stream
        if keys is not None:
            self.set_keys(keys)
        if not self._first:
            cs.wait_event(self._y_consumed)            # the previous batch has left the staging buffer
        with torch.cuda.stream(cs):
            self.y_stage.copy_(host_in, non_blocking=True)
            self._h2d_done.record(cs)
        with torch.cuda.stream(ms):
            ms.wait_event(self._h2d_done)
            self.y_dev.copy_(self.y_stage, non_blocking=True)
            self._y_consumed.record(ms)
            self.graph.replay()
            if not self._first:
                ms.wait_event(self._d2h_done)          # the previous result has left the output staging buffer
            self.out_stage.copy_(self.out_dev, non_blocking=True)
            self._out_ready.record(ms)
        with torch.cuda.stream(co):
            co.wait_event(self._out_ready)
            host_out.copy_(self.out_stage, non_blocking=True)
            self._d2h_done.record(co)
        self._first = False

    def flush(self):
        """Order the compute stream behind every outstanding copy (call before timing / reading host buffers)."""
        self.stream.wait_stream(self.copy_stream)
        self.stream.wait_stream(self.copy_stream_out)


class GraphedEnhancerCache:
    """enhance_fn(y [B, L], lengths [B], keys=None, seed=None) for `sweep.enhance_sweep`: one captured graph per batch
    shape (the equal-Tpad buckets of a sweep repeat the same few shapes) and, with keys, per seed; eager `enhance_batch`
    for those seen fewer than `min_uses` times.  keys (int64 [B]) with seed select the keyed noise, the keys being
    written into the graph's key buffer at every call.  The returned tensor is the graph's output buffer: valid until
    the next call with the same shape."""

    def __init__(self, model, device, min_uses=2, **kw):
        self.model, self.device, self.min_uses, self.kw = model, torch.device(device), min_uses, kw
        self.pipes, self.uses = {}, {}
        self.cap_stream = torch.cuda.Stream(device=self.device)   # graphs cannot be captured on the default stream

    def __call__(self, y, lengths, keys=None, seed=None):
        keyed = keys is not None
        if keyed and seed is None:
            raise ValueError("GraphedEnhancerCache: keys need a seed")
        key = (tuple(y.shape), seed if keyed else None)
        self.uses[key] = self.uses.get(key, 0) + 1
        kw = dict(self.kw, keys=keys, seed=seed) if keyed else self.kw
        if key not in self.pipes:
            if self.uses[key] < self.min_uses:
                return self.model.enhance_batch(y, lengths=lengths, **kw)
            pipe = GraphedEnhancer(self.model, key[0][0], key[0][1], self.device, ragged=True, stream=self.cap_stream,
                                   keyed=keyed, seed=seed if keyed else 0, **self.kw)
            pipe.y_dev.copy_(y)
            pipe.len_dev.copy_(lengths)
            if keyed:
                pipe.key_dev.copy_(keys)
            torch.cuda.current_stream(self.device).synchronize()
            self.pipes[key] = pipe.capture(warmup=1)
            self.cap_stream.synchronize()
        pipe = self.pipes[key]
        pipe.y_dev.copy_(y, non_blocking=True)
        pipe.len_dev.copy_(lengths, non_blocking=True)
        if keyed:
            pipe.key_dev.copy_(keys, non_blocking=True)
        pipe.graph.replay()
        return pipe.out_dev
