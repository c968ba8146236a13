"""`ScoreModel` (inference API; mirror of sgmse-bbed/sgmse/model.py:22-30,43-134,481-634,702-839).

Same constructor / `load_from_checkpoint` / `eval(no_ema)` / `forward(x,t,y)` / `enhance(x,y,...)` /
`get_pc_sampler` / `get_ode_sampler` / `to_audio` contract as the reference, but the whole
sebridge_v3 branch of `enhance` runs on the GPU without a host round trip: peak -> SNR estimate ->
t snap / norm factor (device scalars) -> STFT+transform -> X_T -> preconditioned NCSN++ -> iSTFT.
Training-time members (`_step`, losses, dataloaders) are out of scope (SURVEY 2.1).
"""
import os
import time
import warnings
from math import ceil

import numpy as np
import torch

from .. import ops
from ..engine import MODE_NEG, MODE_RAW, MODE_SEBRIDGE
from . import sampling
from ._checkpoint import CheckpointedModule
from .backbones import BackboneRegistry
from .data_module import SpecsDataModule
from .sdes import SDERegistry, axpby
from .snr_estimator import SNRModel
from .util.other import pad_spec, pad_spec_16, snr_dB  # noqa: F401

i_30 = np.arange(1, 30 + 1)
t_30 = (0.001 ** (1 / 7) + (i_30 - 1) / (30 - 1) * (1 ** (1 / 7) - 0.001 ** (1 / 7))) ** 7   # model.py:22-23

# The reference loads a module-global SNR estimator from a path relative to the CWD at import time
# (model.py:25-30).  Here it is resolved lazily on first use (same default path) or set explicitly.
SNR_ESTIMATOR_CKPT = './sgmse-bbed/sgmse/snr_estimator.ckpt'
snr_model = None


def set_snr_model(model):
    global snr_model
    snr_model = model


def get_snr_model():
    global snr_model
    if snr_model is None:
        if not os.path.exists(SNR_ESTIMATOR_CKPT):
            raise FileNotFoundError(f"SNR estimator checkpoint {SNR_ESTIMATOR_CKPT!r} not found "
                                    "(model.py:25-30 loads it relative to the working directory); "
                                    "call sgmse.model.set_snr_model(...) or pass oracle=True")
        snr_model = SNRModel.load_from_checkpoint(SNR_ESTIMATOR_CKPT, base_dir="", batch_size=1, num_workers=0)
        snr_model.eval()
    return snr_model


class ScoreModel(CheckpointedModule):
    frozen_params = ("all_modules.0.W",)   # GaussianFourierProjection.W has requires_grad=False (layerspp.py:37)

    @staticmethod
    def add_argparse_args(parser):
        parser.add_argument("--lr", type=float, default=1e-4)
        parser.add_argument("--ema_decay", type=float, default=0.999)
        parser.add_argument("--t_eps", type=float, default=0.03)
        parser.add_argument("--num_eval_files", type=int, default=10)
        parser.add_argument("--loss_type", type=str, default="mse")
        parser.add_argument("--loss_abs_exponent", type=float, default=0.5)
        return parser

    def __init__(self, backbone, sde, model_type='sebridge', snr_conditioned='false', fixed_snr=1.0, lr=1e-4,
                 ema_decay=0.999, t_eps=3e-2, loss_abs_exponent=0.5, num_eval_files=10, loss_type='mse',
                 data_module_cls=None, **kwargs):
        if snr_conditioned not in ('false', 'fixed', 'true'):
            raise ValueError(f"snr_conditioned must be the string 'true', 'false' or 'fixed' (got {snr_conditioned!r})")
        dnn_cls = BackboneRegistry.get_by_name(backbone)
        self.dnn = dnn_cls(**kwargs)
        if sde == 'bbve':   # model.py:70-76
            sde = 'bbed'
            kwargs['k'] = kwargs['sigma_max']
            del kwargs['sigma_max']
            del kwargs['sigma_min']
        sde_cls = SDERegistry.get_by_name(sde)
        self.sde = sde_cls(**kwargs)
        self.sigma_max = kwargs.get('sigma_max', None)
        self.model_type, self.snr_conditioned, self.fixed_snr = model_type, snr_conditioned, fixed_snr
        self.lr, self.ema_decay, self.t_eps = lr, ema_decay, t_eps
        self.loss_type, self.num_eval_files, self.loss_abs_exponent = loss_type, num_eval_files, loss_abs_exponent
        self._init_ckpt(ema_decay)
        data_module_cls = data_module_cls or SpecsDataModule
        self.data_module = data_module_cls(**kwargs, fixed_snr=self.fixed_snr, gpu=kwargs.get('gpus', 0) > 0)

    @classmethod
    def from_state_dict(cls, sd, **hparams):
        """Build directly from a reference-format state dict (no checkpoint file)."""
        m = cls(**hparams)
        m._error_loading_ema = True
        m.load_state_dict(sd)
        return m

    def _dnn_names(self):
        return list(self.dnn.param_shapes().keys())

    def export_flat(self, path):
        """Write the weights that are live now (EMA after `eval()`, raw after `eval(no_ema=True)` / `train()`) as the flat
        kernel-ready file of `NCSNppEngine.export_flat` (SURVEY 8f-2); `NCSNppEngine().load_flat(path)` uploads it."""
        return self.dnn.engine.export_flat({"dnn." + k: v for k, v in self.dnn.state_dict().items()}, path)

    # ------------------------------------------------------------------------------ network call
    def _head_mode(self):
        if self.snr_conditioned == 'false':
            if self.model_type == 'bbed':
                return MODE_NEG
            if self.model_type in ('sebridge', 'sebridge_v2'):
                return MODE_SEBRIDGE
        elif self.snr_conditioned == 'fixed':
            if self.model_type == 'sebridge_v3':
                return MODE_SEBRIDGE
            raise NotImplementedError("snr_conditioned='fixed' with sebridge_v2 (experimental preconditioning, "
                                      "model.py:507-514) is not implemented")
        elif self.snr_conditioned == 'true':
            if self.model_type in ('sebridge_v2', 'sebridge_v3'):
                return MODE_SEBRIDGE
        raise NotImplementedError(f"model_type={self.model_type!r} with snr_conditioned={self.snr_conditioned!r}")

    def forward(self, x, t, y, s=None):
        """x, y [B,1,F,T] complex64; t [B,1,1,1] (sebridge*) or [B] (bbed)  ->  [B,1,F,T]  (model.py:481-543)."""
        mode = self._head_mode()
        if mode == MODE_SEBRIDGE:
            if t.dim() != 4:
                raise IndexError("Dimension out of range (expected t of shape [B,1,1,1] for the sebridge heads, "
                                 "model.py:540)")
            t = t.squeeze(3).squeeze(2).squeeze(1)
        self.dnn._ensure_device_weights()
        dev = x.device
        xg = (x if x.is_cuda else x.cuda())[:, 0]
        yg = (y if y.is_cuda else y.cuda())[:, 0]
        out = self.dnn.engine.forward(xg, yg, t.to("cuda", torch.float32), mode=mode)
        return out[:, None].to(dev)

    __call__ = forward

    # ------------------------------------------------------------------------------ samplers
    def get_pc_sampler(self, predictor_name, corrector_name, y, Y_prior=None, N=None, minibatch=None,
                       timestep_type=None, **kwargs):
        N = self.sde.N if N is None else N
        sde = self.sde.copy()
        sde.N = N
        kwargs = {"eps": self.t_eps, **kwargs}
        if kwargs.get("graph", None) is not False:
            # captured loops are kept per model across sampler objects; they point into the packed weight blob and the
            # engine's activation arena, so a weight (re)load -- EMA swap, load_state_dict -- drops them.  The tag is the
            # engine's monotonically increasing weights generation (an address could be handed out again by the allocator)
            self.dnn._ensure_device_weights()
            tag = self.dnn.engine.weights_generation
            if self.__dict__.get("_pc_graph_tag") != tag:
                self.__dict__["_pc_graph_cache"], self.__dict__["_pc_graph_tag"] = {}, tag
            kwargs.setdefault("graph_cache", self.__dict__["_pc_graph_cache"])
        if minibatch is None:
            return sampling.get_pc_sampler(predictor_name, corrector_name, sde=sde, score_fn=self, Y=y,
                                           Y_prior=Y_prior, timestep_type=timestep_type, **kwargs)
        M = y.shape[0]

        def batched_sampling_fn():
            samples, ns = [], []
            for i in range(int(ceil(M / minibatch))):
                y_mini = y[i * minibatch:(i + 1) * minibatch]
                prior = None if Y_prior is None else Y_prior[i * minibatch:(i + 1) * minibatch]
                sample, n = sampling.get_pc_sampler(predictor_name, corrector_name, sde=sde, score_fn=self, Y=y_mini,
                                                    Y_prior=prior, **kwargs)()
                samples.append(sample)
                ns.append(n)
            return torch.cat(samples, dim=0), ns
        return batched_sampling_fn

    def get_ode_sampler(self, y, Y_prior=None, N=None, minibatch=None, timestep_type=None, **kwargs):
        N = self.sde.N if N is None else N
        sde = self.sde.copy()
        sde.N = N
        kwargs = {"eps": self.t_eps, **kwargs}
        if minibatch is None:
            return sampling.get_ode_sampler(sde, self, y=y, Y_prior=Y_prior, timestep_type=timestep_type, **kwargs)
        M = y.shape[0]

        def batched_sampling_fn():
            samples, ns = [], []
            for i in range(int(ceil(M / minibatch))):
                sample, n = sampling.get_ode_sampler(sde, self, y=y[i * minibatch:(i + 1) * minibatch], **kwargs)()
                samples.append(sample)
                ns.append(n)
            return torch.cat(samples, dim=0), ns
        return batched_sampling_fn

    # ------------------------------------------------------------------------------ transforms
    def to_audio(self, spec, length=None):
        return self._istft(self._backward_transform(spec), length)

    def _forward_transform(self, spec):
        return self.data_module.spec_fwd(spec)

    def _backward_transform(self, spec):
        return self.data_module.spec_back(spec)

    def _stft(self, sig):
        return self.data_module.stft(sig)

    def _istft(self, spec, length=None):
        return self.data_module.istft(spec, length)

    def calculate_snr_direct(self, s, n, fixed_snr):
        return (n / s) / (10 ** 0.25 * fixed_snr)

    def calculate_normfac_direct(self, s, n, fixed_snr):
        return (2.040166) * (0.240253 + 0.759747 * fixed_snr ** 2) ** 0.5 / ((1 + (n / s) ** 2) ** 0.5)

    def _spec_params(self):
        dm = self.data_module           # (kernel transform code 0 none / 1 exponent / 2 log, alpha, beta)
        if dm.transform_type == "none":
            return 0, 1.0, 1.0
        return dm.transform_code, float(dm.spec_abs_exponent), float(dm.spec_factor)

    # ------------------------------------------------------------------------------ enhancement
    def enhance_batch(self, y, lengths=None, oracle=False, noise_over_clean=None, noise=None, return_aux=False,
                      generator=None, keys=None, seed=0):
        """sebridge_v3 / snr_conditioned='true' enhancement of a padded batch, entirely on the GPU.

        y: [B, Lmax] float32 (host or device); lengths: optional [B] valid sample counts;
        noise_over_clean: [B] noise_rms/clean_rms when oracle=True; noise: optional explicit complex
        normal Z [B,1,256,Tpad], otherwise drawn from `generator` (a CUDA torch.Generator; default: torch's
        default CUDA generator).  Returns the enhanced batch [B, Lmax] on the GPU (zeros past each length).
        One pass = model.py:713-752,810-830 for every utterance, with no host synchronisation.

        keys: optional per-utterance 64-bit noise keys (int64 [B] or a list of ints, host or device; see
        `ops.key_tensor`) with `seed` (int in [0, 2^64)).  Then every utterance is enhanced as if alone: Z is the keyed
        noise of include/snrse_b200.h (a function of key, seed and element only) and the SNR estimate (oracle=False)
        covers the utterance's own 16-frame clusters (`SNRModel.estimate_batch`), so item b equals
        `enhance(None, y[b:b+1, :len_b], key=keys[b], seed=seed)` bit for bit whatever its row or batch.  Every
        utterance must pad to the batch's Tpad (64*ceil((1 + len//128)/64) frames): host lengths that do not raise
        ValueError, device lengths that do not make that item NaN.  keys cannot be combined with noise= or
        generator=.  return_aux then also holds the draw Z [B,1,256,Tpad]."""
        if not (self.snr_conditioned == 'true' and self.model_type == 'sebridge_v3'):
            raise NotImplementedError("enhance_batch implements the sebridge_v3 SNR-conditioned path")
        if keys is not None and (noise is not None or generator is not None):
            raise ValueError("enhance_batch: keys= draws the noise itself; it cannot be combined with noise= or generator=")
        self.dnn._ensure_device_weights()
        yd = (y if y.is_cuda else y.cuda()).to(torch.float32).contiguous()
        B, L = yd.shape
        ld = None if lengths is None else lengths.to("cuda", torch.int32).contiguous()
        tr, alpha, beta = self._spec_params()
        if keys is not None:
            kd = ops.key_tensor(keys, B).to(yd.device)
            if lengths is not None and not torch.as_tensor(lengths).is_cuda:
                tp = ops.padded_frames(L)
                own = [ops.padded_frames(int(n)) for n in torch.as_tensor(lengths).reshape(-1).tolist()]
                if any(t_ != tp for t_ in own):
                    raise ValueError(f"enhance_batch: with keys every utterance must pad to the batch's {tp} frames "
                                     f"(lengths {torch.as_tensor(lengths).tolist()} pad to {own})")
        if keys is not None and not oracle:
            ratio, est_aux = get_snr_model().estimate_batch(yd, lengths, return_aux=True)   # per file (:715-721)
            peak = est_aux["peak"]
        else:
            peak = ops.absmax(yd, ld)                                              # y.abs().max()  (:715,726)
            if oracle:
                ratio = torch.as_tensor(noise_over_clean, dtype=torch.float32).reshape(-1).to("cuda")
                if ratio.numel() == 1 and B > 1:
                    ratio = ratio.expand(B).contiguous()
            else:
                est = get_snr_model()
                feat = ops.stft(yd, ld, scale=peak, scale_is_divisor=True, transform=False, planar=True, pad_multiple=16)
                g = est.dnn.forward(feat)[:, 0].contiguous()                       # n/(s+n)  (:716-720)
                ratio = est.dnn.engine.noise_over_clean(g)                         # (:721)
        t, norm, idx = ops.v3_scalars(ratio, peak, self.fixed_snr)                # (:732-740)
        Y = ops.stft(yd, ld, scale=norm, scale_is_divisor=True, transform=tr, alpha=alpha, beta=beta)   # (:746-751)
        if keys is not None:                                                       # (:822-823), keyed Z
            ones = torch.ones(B, dtype=torch.float32, device=Y.device)
            _, X_T, Z = ops.lincomb_keyed(y=Y, b=ones, d=t * float(self.sigma_max), keys=kd, seed=seed, lengths=ld,
                                          want_mean=False, want_z=return_aux)
        else:
            Z = torch.randn_like(Y, generator=generator) if noise is None else noise.to("cuda").reshape(Y.shape).contiguous()
            X_T = axpby(y=Y, b=1.0, z=Z, d=t * float(self.sigma_max))             # (:822-823)
        sample = self.dnn.engine.forward(X_T, Y, t, mode=MODE_SEBRIDGE)           # (:824, 537-541)
        x_hat = ops.istft(sample, L, ld, scale=norm, transform=tr, alpha=alpha, beta=beta)   # (:828-830)
        if return_aux:
            aux = dict(t=t, t_index=idx, norm_factor=norm, Y=Y, X_T=X_T, sample=sample, ratio=ratio)
            if keys is not None:
                aux["Z"] = Z[:, None]
            return x_hat, aux
        return x_hat

    def enhance_snr_sweep(self, x, noise, snrs=range(0, 41, 5), oracle=True, noise_draws=None):
        """The SNR sweep of deep_eval.py:112-122 for one file as ONE batch: for every SNR in `snrs` the mixture
        y = x + noise * 10^(-SNR/20) is enhanced with clean_rms = 1, noise_rms = 10^((-SNR+5)/20) (oracle) or with the
        SNR estimator (oracle=False).  x, noise: [1, L] waveforms (clean, y - x).  Returns a list of 1-D float32 numpy
        arrays, one per SNR, equal to what `enhance` returns for each mixture on its own.
        noise_draws: optional explicit complex normal draws [len(snrs), 1, 256, Tpad]."""
        snrs = list(snrs)
        xd = (x if x.is_cuda else x.cuda()).to(torch.float32).reshape(1, -1)
        nd = (noise if noise.is_cuda else noise.cuda()).to(torch.float32).reshape(1, -1)
        gains = torch.tensor([10.0 ** (-s / 20.0) for s in snrs], dtype=torch.float32, device=xd.device)[:, None]
        y = xd + nd * gains                                                   # [len(snrs), L]
        ratios = [10.0 ** ((-s + 5) / 20.0) for s in snrs] if oracle else None
        out = self.enhance_batch(y, oracle=oracle, noise_over_clean=ratios, noise=noise_draws)
        out = out.detach().cpu().numpy()
        return [out[k] for k in range(len(snrs))]

    def enhance(self, x, y, sampler_type="pc", predictor="reverse_diffusion", corrector="ald", N=30,
                corrector_steps=1, snr=0.5, timeit=False, oracle=False, clean_rms=1, noise_rms=1, **kwargs):
        """One-call enhancement of noisy speech `y` [1,L] (model.py:702-839).  `x` (clean) is accepted for
        signature compatibility and unused.  Extra keyword `noise=` supplies the complex normal draw; `key=k, seed=s`
        (sebridge_v3) draw it as keyed noise instead, which is what `enhance_batch(..., keys=, seed=)` gives this file in
        any batch."""
        sr = 16000
        start = time.time()
        noise = kwargs.pop("noise", None)
        key, seed = kwargs.pop("key", None), kwargs.pop("seed", 0)
        if key is not None and not (self.snr_conditioned == 'true' and self.model_type == 'sebridge_v3'):
            raise NotImplementedError("key= (keyed noise) is implemented for the sebridge_v3 SNR-conditioned path")
        T_orig = y.size(1)
        nfe = 1
        if self.snr_conditioned == 'true' and self.model_type == 'sebridge_v3':
            ratio = None if not oracle else [noise_rms / clean_rms]
            x_hat = self.enhance_batch(y, oracle=oracle, noise_over_clean=ratio, noise=noise,
                                       keys=None if key is None else [key], seed=seed)
        elif self.snr_conditioned == 'fixed':
            raise NotImplementedError("snr fixed is only for experiment purpose, not real inference.")
        elif self.snr_conditioned == 'false':
            yd = (y if y.is_cuda else y.cuda()).to(torch.float32)
            norm = ops.absmax(yd)
            tr, alpha, beta = self._spec_params()
            Y = ops.stft(yd, scale=norm, scale_is_divisor=True, transform=tr, alpha=alpha, beta=beta)[:, None]
            if self.model_type == 'bbed':
                if sampler_type == "pc":
                    sampler = self.get_pc_sampler(predictor, corrector, Y, N=N, corrector_steps=corrector_steps,
                                                  snr=snr, intermediate=False, **kwargs)
                elif sampler_type == "ode":
                    sampler = self.get_ode_sampler(Y, N=N, **kwargs)
                else:
                    raise ValueError("{} is not a valid sampler type!".format(sampler_type))
                sample, nfe = sampler()
            elif self.model_type == 'sebridge':
                vec_t = torch.full((Y.shape[0], 1, 1, 1), 0.999, device=Y.device)
                sample = self(Y, vec_t, Y)
            elif self.model_type == 'sebridge_v2':
                vec_t = torch.full((Y.shape[0], 1, 1, 1), 0.999, device=Y.device)
                Z = torch.randn_like(Y) if noise is None else noise.to(Y.device)
                sample = self(axpby(y=Y, b=1.0, z=Z, d=float(self.sigma_max) * 0.999), vec_t, Y)
            else:
                raise NotImplementedError(self.model_type)
            x_hat = ops.istft(sample[:, 0].contiguous(), T_orig, scale=norm, transform=tr, alpha=alpha, beta=beta)
        else:
            raise NotImplementedError("sebridge_v2 with snr_conditioned='true' calls an undefined helper in the "
                                      "reference (model.py:795-796, noise_mag) and is not supported")
        x_hat = x_hat.squeeze().detach().cpu().numpy()    # the one device->host copy of the call
        end = time.time()
        if timeit:
            return x_hat, nfe, (end - start) / (len(x_hat) / sr)
        return x_hat
