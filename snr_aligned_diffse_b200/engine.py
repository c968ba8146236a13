"""Host-side owner of the native NCSN++ executor: weight packing, workspace, plans, CUDA graphs.

The network itself (topology, kernels, buffer plan) lives in `csrc/engine.cu`; this module only
moves a reference-format `state_dict` into the packed device blob the executor describes and
hands torch-owned device memory to it.
"""
import ctypes
from ctypes import byref, c_int, c_int64, c_void_p, create_string_buffer

import torch

from . import _lib

PK_RAW_F32, PK_CONV3_K_BF16, PK_CONV1_K_BF16, PK_NIN_K_BF16, PK_CONV3_TAP_F32, PK_CONV3_K_BF16_HILO64 = range(6)

DEFAULT_CONFIG = dict(nf=128, ch_mult=(1, 1, 2, 2, 2, 2, 2), num_res_blocks=2, attn_resolutions=(16,), image_size=256)

FLAG_KEEP_ALL = 1     # keep every activation (debug taps)
FLAG_SIMT_CONV = 2    # CUDA-core cross-check convolutions instead of tcgen05

MODE_RAW, MODE_SEBRIDGE, MODE_NEG = 0, 1, 2

# snrse_conv_plan / snrse_conv_row of include/snrse_b200_plans.h, field for field
CONV_PLAN_FIELDS = ("sub", "nsplit", "n_loc", "acc_bufs", "na", "nb", "stg_bufs", "nsc", "th", "tw", "n_tile", "small",
                    "stages", "tiles_h", "tiles_w", "n_tiles", "grid", "smem_bytes")
CONV_ROW_FIELDS = ("path", "out4", "B", "H", "W", "c0", "ld0", "off0", "c1", "ld1", "off1", "res", "ld_res", "off_res",
                   "ld_out", "off_out", "taps", "n", "norm", "bias", "tbias", "tb_stride", "stats", "addend", "scale") \
    + CONV_PLAN_FIELDS


class NCSNppEngine:
    """One packed copy of the weights on one GPU + per-(B,F,T) launch plans."""

    def __init__(self, nf=128, ch_mult=(1, 1, 2, 2, 2, 2, 2), num_res_blocks=2, attn_resolutions=(16,),
                 image_size=256, **unused):
        self.lib = _lib.load()
        self.cfg = dict(nf=nf, ch_mult=tuple(ch_mult), num_res_blocks=num_res_blocks,
                        attn_resolutions=tuple(attn_resolutions), image_size=image_size)
        cm = (c_int * len(ch_mult))(*ch_mult)
        ar = (c_int * max(1, len(attn_resolutions)))(*attn_resolutions)
        h = c_void_p()
        _lib.check(self.lib.snrse_ncsnpp_create(byref(h), nf, cm, len(ch_mult), num_res_blocks, ar,
                                                len(attn_resolutions), image_size), "ncsnpp_create")
        self.h = h
        self.blob = None
        self.device = None
        self._ws = {}       # (B,F,T) -> (workspace tensor, flags)
        self.weights_generation = 0    # bumped by every load_state_dict: tag for caches of captured CUDA graphs

    def __del__(self):
        try:
            if getattr(self, "h", None):
                self.lib.snrse_ncsnpp_destroy(self.h)
                self.h = None
        except Exception:
            pass

    # ------------------------------------------------------------------ weights
    def param_table(self):
        n = self.lib.snrse_ncsnpp_num_params(self.h)
        out = []
        name = create_string_buffer(256)
        kind, acc = c_int(), c_int()
        off, rs, ko = c_int64(), c_int64(), c_int64()
        for i in range(n):
            _lib.check(self.lib.snrse_ncsnpp_param_info(self.h, i, name, 256, byref(kind), byref(off), byref(rs),
                                                        byref(ko), byref(acc)), "param_info")
            out.append(dict(name=name.value.decode(), kind=kind.value, offset=off.value, row_stride=rs.value,
                            k_offset=ko.value, accumulate=acc.value))
        return out

    def param_shapes(self):
        """name -> shape of the reference state-dict tensor each table entry expects (table order)."""
        out = {}
        dims, nd = (c_int64 * 4)(), c_int()
        for i, p in enumerate(self.param_table()):
            _lib.check(self.lib.snrse_ncsnpp_param_shape(self.h, i, dims, byref(nd)), "param_shape")
            out[p["name"]] = tuple(int(dims[j]) for j in range(nd.value))
        return out

    @property
    def weight_bytes(self):
        return int(self.lib.snrse_ncsnpp_weight_bytes(self.h))

    def pack_state_dict(self, sd):
        """Reference state dict (fp32, any device) -> packed host blob (uint8 tensor)."""
        blob = torch.zeros(self.weight_bytes, dtype=torch.uint8)
        f32 = blob.view(torch.float32)
        b16 = blob.view(torch.bfloat16)
        for p in self.param_table():
            if p["name"] not in sd:
                raise KeyError(f"state dict lacks {p['name']}")
            w = sd[p["name"]].detach().to("cpu", torch.float32)
            k, off = p["kind"], p["offset"]
            if k == PK_RAW_F32:
                flat = w.reshape(-1)
                dst = f32[off // 4: off // 4 + flat.numel()]
                if p["accumulate"]:
                    dst += flat
                else:
                    dst.copy_(flat)
                continue
            if k == PK_CONV3_TAP_F32:
                flat = w.permute(0, 2, 3, 1).reshape(-1)
                f32[off // 4: off // 4 + flat.numel()].copy_(flat)
                continue
            if k == PK_CONV3_K_BF16_HILO64:
                # input convolution on the 64-channel hi/lo operand (pack_input64): [cout][tap*64 + c], the Cin
                # weights repeated for the hi (c < Cin) and lo (Cin <= c < 2 Cin) halves, zero above
                co, ci = w.shape[0], w.shape[1]
                rows = torch.zeros(co, 9, 64)
                taps = w.permute(0, 2, 3, 1).reshape(co, 9, ci)
                rows[:, :, :ci] = taps
                rows[:, :, ci:2 * ci] = taps
                rows = rows.reshape(co, 9 * 64)
            elif k == PK_CONV3_K_BF16:
                rows = w.permute(0, 2, 3, 1).reshape(w.shape[0], -1)       # [cout][(r,s,cin)]
            elif k == PK_CONV1_K_BF16:
                rows = w.reshape(w.shape[0], w.shape[1])                    # [cout][cin]
            elif k == PK_NIN_K_BF16:
                rows = w.t()                                               # W[in,out] -> [out][in]
            else:
                raise ValueError(f"unknown pack kind {k}")
            n, kk = rows.shape
            rs, ko = p["row_stride"], p["k_offset"]
            dst = b16[off // 2: off // 2 + n * rs].view(n, rs)
            dst[:, ko:ko + kk].copy_(rows.to(torch.bfloat16))
        return blob

    def load_state_dict(self, sd, device="cuda"):
        _lib.require_device()
        self.device = torch.device(device)
        self.blob = self.pack_state_dict(sd).to(self.device)
        _lib.check(self.lib.snrse_ncsnpp_set_weights(self.h, _lib.ptr(self.blob)), "set_weights")
        self._ws.clear()
        self.weights_generation += 1
        return self

    # ------------------------------------------------------------------ flat weight file (SURVEY 8f-2)
    FLAT_MAGIC = b"SNRSEW01"

    def export_flat(self, sd, path):
        """Write a reference-format state dict as the flat, kernel-ready weight file: 8-byte magic, 8-byte little-endian
        header length, a JSON header (network config, blob size, sha256 of the blob, the parameter table: name, pack
        kind, byte offset, row stride, k offset) and the packed blob exactly as the kernels read it (3x3 / 1x1 / NIN
        weights bf16 K-major with the fused Conv_1|Conv_2 rows concatenated, fp32 biases / GroupNorm affine / Dense_0
        block).  `load_flat` uploads the blob with one copy and no per-tensor work."""
        import hashlib
        import json
        blob = self.pack_state_dict(sd)
        raw = blob.numpy().tobytes()
        header = dict(format="snrse_b200 packed NCSN++ weights", version=1, config={k: list(v) if isinstance(v, tuple) else v
                                                                                  for k, v in self.cfg.items()},
                      weight_bytes=len(raw), sha256=hashlib.sha256(raw).hexdigest(), params=self.param_table())
        hj = json.dumps(header).encode()
        with open(path, "wb") as f:
            f.write(self.FLAT_MAGIC)
            f.write(len(hj).to_bytes(8, "little"))
            f.write(hj)
            f.write(raw)
        return header

    @classmethod
    def read_flat(cls, path):
        """-> (header dict, packed blob as a uint8 host tensor); verifies magic, size and checksum."""
        import hashlib
        import json
        with open(path, "rb") as f:
            if f.read(8) != cls.FLAT_MAGIC:
                raise ValueError(f"{path}: not a snrse_b200 flat weight file")
            n = int.from_bytes(f.read(8), "little")
            header = json.loads(f.read(n).decode())
            raw = f.read()
        if len(raw) != header["weight_bytes"] or hashlib.sha256(raw).hexdigest() != header["sha256"]:
            raise ValueError(f"{path}: weight blob is truncated or corrupt")
        return header, torch.frombuffer(bytearray(raw), dtype=torch.uint8)

    def load_flat(self, path, device="cuda"):
        """Upload a file written by `export_flat` (must match this engine's configuration and parameter table)."""
        header, blob = self.read_flat(path)
        cfg = {k: list(v) if isinstance(v, tuple) else v for k, v in self.cfg.items()}
        if header["config"] != cfg or header["weight_bytes"] != self.weight_bytes or header["params"] != self.param_table():
            raise ValueError(f"{path}: written for another network configuration / library layout")
        _lib.require_device()
        self.device = torch.device(device)
        self.blob = blob.to(self.device)
        _lib.check(self.lib.snrse_ncsnpp_set_weights(self.h, _lib.ptr(self.blob)), "set_weights")
        self._ws.clear()
        self.weights_generation += 1
        return self

    # ------------------------------------------------------------------ plans
    def workspace_bytes(self, B, F, T, flags=0):
        n = int(self.lib.snrse_ncsnpp_plan_bytes(self.h, B, F, T, flags))
        if n < 0:
            _lib.check(1, "plan")
        return n

    def reserve(self, nbytes):
        """One shared activation arena of `nbytes` for every plan created from now on (instead of one buffer per
        (B,F,T) bucket).  Forwards of one engine run on one stream, so all buckets can live in the same memory: a sweep
        over many utterance lengths then needs the LARGEST bucket's workspace, not the sum over buckets."""
        self._arena = torch.empty(int(nbytes) + 1024, dtype=torch.uint8, device=self.device)
        return self

    def prepare(self, B, F, T, flags=0):
        key = (B, F, T)
        cur = self._ws.get(key)
        if cur is not None and cur[1] == flags:
            return
        if self.blob is None:
            raise RuntimeError("load_state_dict() first")
        n = self.workspace_bytes(B, F, T, flags)
        arena = getattr(self, "_arena", None)
        ws = arena if (arena is not None and arena.numel() >= n + 1024) else torch.empty(n + 1024, dtype=torch.uint8, device=self.device)
        base = ws.data_ptr()
        aligned = (base + 1023) // 1024 * 1024
        _lib.check(self.lib.snrse_ncsnpp_plan_bind(self.h, B, F, T, c_void_p(aligned), n), "plan_bind")
        self._ws[key] = (ws, flags)

    def forward(self, x, y, t, mode=MODE_RAW, out=None, flags=0):
        """x, y: complex64 [B,F,T] (or [B,1,F,T]); t: float32 [B].  Enqueues on the current stream."""
        assert x.is_cuda and x.dtype == torch.complex64 and y.dtype == torch.complex64
        shape = x.shape
        B, F, T = shape[0], shape[-2], shape[-1]
        self.prepare(B, F, T, flags)
        x = x.contiguous()
        y = y.contiguous()
        t = t.to(torch.float32).reshape(-1).contiguous()
        assert t.numel() == B
        if out is None:
            out = torch.empty_like(x)
        _lib.check(self.lib.snrse_ncsnpp_forward(self.h, B, F, T, _lib.ptr(x), _lib.ptr(y), _lib.ptr(t), _lib.ptr(out),
                                                 mode, _lib.stream_ptr()), "ncsnpp_forward")
        return out

    def read_tap(self, B, F, T, module_idx):
        dims = (c_int64 * 4)()
        cap = B * 512 * F * T
        buf = torch.empty(cap, dtype=torch.float32, device=self.device)
        _lib.check(self.lib.snrse_ncsnpp_read_tap(self.h, B, F, T, module_idx, _lib.ptr(buf), cap, dims,
                                                  _lib.stream_ptr()), "read_tap")
        b, c, h, w = (int(d) for d in dims)
        return buf[: b * c * h * w].view(b, c, h, w).clone()

    def profile_forward(self, x, y, t, mode=MODE_RAW, flags=0):
        """Eager forward with CUDA events between launch groups (measurement only).
        Returns a list of dict(kind, flops, bytes, ms); kind 1 = implicit-GEMM convolution."""
        from ctypes import c_double, c_float
        B, F, T = x.shape[0], x.shape[-2], x.shape[-1]
        self.prepare(B, F, T, flags)
        n = self.num_launch_groups(B, F, T)
        kinds, fl, by, ms = (c_int * n)(), (c_double * n)(), (c_double * n)(), (c_float * n)()
        cnt = c_int()
        out = torch.empty_like(x)
        t = t.to(torch.float32).reshape(-1).contiguous()
        _lib.check(self.lib.snrse_ncsnpp_profile_forward(self.h, B, F, T, _lib.ptr(x.contiguous()), _lib.ptr(y.contiguous()),
                                                         _lib.ptr(t), _lib.ptr(out), mode, _lib.stream_ptr(), n, kinds,
                                                         fl, by, ms, byref(cnt)), "profile_forward")
        return [dict(kind=kinds[i], flops=fl[i], bytes=by[i], ms=ms[i]) for i in range(cnt.value)]

    def conv_rows(self, B, F, T, flags=0, num_sms=148):
        """Every convolution the (B,F,T) plan records, with its operand views and its plan for num_sms SMs
        (snrse_ncsnpp_dbg_convs; no device needed): a numpy structured array with the fields CONV_ROW_FIELDS."""
        import numpy as np
        dtype = np.dtype([(f, np.float32 if f == "scale" else np.int32) for f in CONV_ROW_FIELDS])
        n = c_int()
        _lib.check(self.lib.snrse_ncsnpp_dbg_convs(self.h, B, F, T, flags, num_sms, None, 0, byref(n)), "dbg_convs")
        rows = np.zeros(n.value, dtype)
        _lib.check(self.lib.snrse_ncsnpp_dbg_convs(self.h, B, F, T, flags, num_sms, rows.ctypes.data, n.value, byref(n)),
                   "dbg_convs")
        return rows

    def num_launch_groups(self, B, F, T):
        return int(self.lib.snrse_ncsnpp_num_launch_groups(self.h, B, F, T))
