"""`SNRModel` (inference half; mirror of sgmse-bbed/sgmse/snr_estimator.py:19-79,143-146)."""
import torch

from .. import ops
from ._checkpoint import CheckpointedModule
from .backbones.snrnet import SNRNet
from .data_module import SpecsDataModule


class SNRModel(CheckpointedModule):
    def __init__(self, backbone="snrnet", lr=1e-4, ema_decay=0.999, num_eval_files=10, loss_type='mse',
                 data_module_cls=None, **kwargs):
        self.dnn = SNRNet()
        self.lr, self.ema_decay, self.loss_type, self.num_eval_files = lr, ema_decay, loss_type, num_eval_files
        self._init_ckpt(ema_decay)
        data_module_cls = data_module_cls or SpecsDataModule
        self.data_module = data_module_cls(**kwargs, gpu=kwargs.get('gpus', 0) > 0)

    def _dnn_names(self):
        return list(self.dnn.state_dict().keys())

    def forward(self, y):
        return self.dnn(y)

    __call__ = forward

    def estimate_batch(self, y, lengths=None, return_aux=False):
        """Noise/clean ratio est_gt/(1-est_gt) of every utterance of a padded batch, each estimated as `enhance` estimates
        that file alone (model.py:715-721): y / max|y| over its own samples, STFT, features padded to its own multiple of
        16 frames, SNRNet over those clusters only.

        y: [B, L] float32, host or device; lengths: optional integer [B] valid sample counts, host or device (None: all
        L).  Returns float32 [B] on the device; with return_aux also dict(g = n/(s+n) [B], clusters = int32 [B],
        peak = max|y| over each item's samples [B]).
        Lengths given on the host are checked there (1 <= len <= L, else ValueError).  Nothing synchronises with the
        host, so with device-resident lengths the call can be captured in a CUDA graph."""
        yd = (y if y.is_cuda else y.cuda()).to(torch.float32).contiguous()
        if yd.dim() != 2:
            raise ValueError(f"estimate_batch: y must be [B, L] (got shape {tuple(yd.shape)})")
        B, L = yd.shape
        if lengths is None:
            ld = torch.full((B,), L, dtype=torch.int32, device=yd.device)
        else:
            lengths = torch.as_tensor(lengths)
            if lengths.dtype.is_floating_point or lengths.is_complex() or lengths.numel() != B:
                raise ValueError(f"estimate_batch: lengths must hold {B} integers (got {lengths.dtype}, "
                                 f"{lengths.numel()} elements)")
            if not lengths.is_cuda:
                bad = (lengths < 1) | (lengths > L)
                if bool(bad.any()):
                    raise ValueError(f"estimate_batch: lengths must lie in [1, {L}] (got {lengths[bad].tolist()})")
            ld = lengths.reshape(B).to(yd.device, torch.int32).contiguous()
        peak = ops.absmax(yd, ld)                                                            # (:715)
        feat = ops.stft(yd, ld, scale=peak, scale_is_divisor=True, transform=False, planar=True, pad_multiple=16)
        clusters = (ld // ops.HOP + 16) // 16                   # ceil(frames / 16), frames = 1 + len // 128  (:717)
        g = self.dnn.forward(feat, clusters)[:, 0].contiguous()                              # n/(s+n)  (:716-720)
        ratio = self.dnn.engine.noise_over_clean(g)                                          # (:721)
        if return_aux:
            return ratio, dict(g=g, clusters=clusters, peak=peak)
        return ratio

    def calculate_normfac_direct(self, s, n, fixed_snr):
        return (2.040166) * (0.240253 + 0.759747 * fixed_snr ** 2) ** 0.5 / ((1 + (n / s) ** 2) ** 0.5)
