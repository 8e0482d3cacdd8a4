"""Hand-over of the logit gradient between the criterion and the network's backward.

The soft-argmax backward (lib/core/integral_loss.py) can write the gradient w.r.t. the logits
straight in the form the final layer's backward consumes (split-fp16 planes + the bias
gradient, epb_softargmax_bwd_split) instead of an fp32 volume that would have to be read
twice more (amax + split) and once for the bias.  The model attaches a LogitGradSink to the
logits tensor it returns; the criterion fills it and hands autograd a zero-valued, zero-stride
token of the right shape; the network's backward takes the planes from the sink.  Anything that
does not fit (another layout, other consumers of the logits, a second backward) falls back to
the fp32 gradient -- the token is ZERO, so gradients of other consumers accumulated onto it
stay exact and the sink's contribution is added back (PoseResNet backward).
"""
import torch


class LogitGradSink:
    """nplanes: plane count of the split gradient the network's backward takes (2: hi + lo,
    1: hi only, the single-pass f16 mode)."""
    __slots__ = ("ptr", "shape", "nplanes", "planes", "sc", "dbias", "filled", "token")

    def __init__(self, logits_nchw_view, nplanes=2):
        t = logits_nchw_view
        self.ptr, self.shape = t.data_ptr(), tuple(t.shape)
        self.nplanes = nplanes
        self.planes = self.sc = self.dbias = None
        self.filled = False
        self.token = torch.zeros(1, device=t.device, dtype=torch.float32)

    def matches(self, t):
        return (not self.filled) and t.data_ptr() == self.ptr and tuple(t.shape) == self.shape

    def is_token(self, g):
        return g.data_ptr() == self.token.data_ptr() and all(s == 0 for s in g.stride())

    def dense(self):
        """The gradient the planes hold, fp32, in their NHWC layout."""
        g = self.planes[0].float()
        if self.nplanes == 2:
            g = g + self.planes[1].float()
        return g * self.sc[1]
