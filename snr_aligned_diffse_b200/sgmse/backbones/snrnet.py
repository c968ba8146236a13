"""`SNRNet` backbone (mirror of sgmse-bbed/sgmse/backbones/snrnet.py:8-97)."""
import torch

from ...ops import SNRNetEngine
from .shared import BackboneRegistry


@BackboneRegistry.register("snrnet")
class SNRNet:
    @staticmethod
    def add_argparse_args(parser):
        return parser

    def __init__(self):
        self.engine = SNRNetEngine()
        self._sd = None
        self._dirty = True

    def load_state_dict(self, sd, strict=True):
        self._sd = {k: v.detach().to("cpu", torch.float32).clone() for k, v in sd.items()}
        self._dirty = True

    def state_dict(self):
        return dict(self._sd or {})

    def forward(self, x, clusters=None):
        """x [B,2,256,T] float32, T % 16 == 0 -> [B,1].  clusters: optional int32 [B], the number of valid 16-frame
        clusters of each item (see `SNRNetEngine.forward`); None runs every item over all T/16 clusters."""
        if self._sd is None:
            raise RuntimeError("SNRNet has no weights")
        if self._dirty:
            self.engine.load_state_dict({"dnn." + k: v for k, v in self._sd.items()}, "cuda")
            self._dirty = False
        dev = x.device
        xg = x if x.is_cuda else x.cuda()
        cg = None if clusters is None else clusters.to(xg.device, torch.int32)
        out = self.engine.forward(xg, cg)
        return out[:, None].to(dev)

    __call__ = forward
