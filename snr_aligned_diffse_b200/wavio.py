"""16 kHz PCM wav files in and out, off the critical path.

The reference's evaluation loop (sgmse-bbed/eval.py:117-140) does, per file and serially on the host:
`torchaudio.load(noisy)` / `load(clean)` -> `model.enhance` -> `soundfile.write(target, x_hat, 16000)` -> metrics.
Here the file loop is `enhance_files`: a reader thread pool decodes every file up front (PCM16 -> float32 / 32768, the
same normalisation torchaudio applies), the utterances go through `sweep.enhance_sweep` (LPT shards, equal-Tpad
batches, SI-SDR on the device when clean files are given), and a writer pool encodes the enhanced waveforms
(float -> PCM16, what soundfile writes for .wav by default) while later batches are still on the GPU.
Only the Python standard library's `wave` module is used for the container format.
"""
import hashlib
import os
import wave
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import torch


def read_wav(path):
    """-> (float32 tensor [L] in [-1, 1), sample rate).  Mono PCM16 (VoiceBank-DEMAND's format); other layouts raise."""
    with wave.open(path, "rb") as w:
        if w.getnchannels() != 1 or w.getsampwidth() != 2 or w.getcomptype() != "NONE":
            raise ValueError(f"{path}: expected mono 16-bit PCM, got {w.getnchannels()} ch x {8 * w.getsampwidth()} bit")
        sr, raw = w.getframerate(), w.readframes(w.getnframes())
    pcm = np.frombuffer(raw, dtype="<i2")
    return torch.from_numpy(pcm.astype(np.float32) / 32768.0), sr


def write_wav(path, samples, sr=16000):
    """float waveform -> mono PCM16 wav (rounded, clipped to the int16 range)."""
    x = samples.detach().cpu().numpy() if torch.is_tensor(samples) else np.asarray(samples)
    pcm = np.clip(np.rint(x.astype(np.float64).reshape(-1) * 32767.0), -32768, 32767).astype("<i2")
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with wave.open(path, "wb") as w:
        w.setnchannels(1)
        w.setsampwidth(2)
        w.setframerate(int(sr))
        w.writeframes(pcm.tobytes())


def name_key(name):
    """64-bit noise key of a file: blake2b-64 of its basename's UTF-8 bytes, as an unsigned int (stable across runs and
    machines, unlike Python's salted `hash`)."""
    return int.from_bytes(hashlib.blake2b(os.path.basename(name).encode("utf-8"), digest_size=8).digest(), "little")


def enhance_files(enhance_fn, noisy_files, target_dir, clean_dir=None, rank=0, world=1, max_batch=16, device=None,
                  io_threads=8, sr=16000, seed=None):
    """The eval.py file loop over `noisy_files` (this rank's shard of it): returns the `enhance_sweep` metrics dict with
    `files` (basename per id) added; enhanced wavs are written to `target_dir/<basename>`.

    enhance_fn(y [B, L], lengths [B]) -> enhanced [B, L]   (e.g. `lambda y, n: model.enhance_batch(y, lengths=n)`).
    seed: keyed noise (see `sweep.enhance_sweep`; enhance_fn then also takes keys and seed), each file keyed by
    `name_key(basename)`, so a file's output does not depend on which other files are in the list."""
    from .sweep import enhance_sweep
    names = [os.path.basename(f) for f in noisy_files]
    with ThreadPoolExecutor(max_workers=io_threads) as pool:
        noisy = list(pool.map(read_wav, noisy_files))
        clean = list(pool.map(read_wav, [os.path.join(clean_dir, n) for n in names])) if clean_dir else None
    for f, (_, r) in zip(noisy_files, noisy):
        if r != sr:
            raise ValueError(f"{f}: sample rate {r}, expected {sr}")
    waves = [w for w, _ in noisy]
    refs = None
    if clean is not None:
        refs = [c[:w.numel()] if c.numel() >= w.numel() else torch.nn.functional.pad(c, (0, w.numel() - c.numel()))
                for (c, _), w in zip(clean, waves)]
    writers = ThreadPoolExecutor(max_workers=io_threads)
    pending = []

    def sink(i, audio):            # called by the sweep as soon as a batch's audio is on the host
        pending.append(writers.submit(write_wav, os.path.join(target_dir, names[i]), audio, sr))

    res = enhance_sweep(enhance_fn, waves, rank=rank, world=world, max_batch=max_batch, device=device, references=refs,
                        on_audio=sink, keys=None if seed is None else [name_key(n) for n in names], seed=seed)
    for p in pending:
        p.result()
    writers.shutdown()
    res["files"] = [names[i] for i in res["ids"]]
    return res
