"""Integral (soft-argmax) joint-location losses -- host-side mirror of the
reference lib/core/integral_loss.py surface, computed by the fused sm_100a
kernels in libepb.so (epb_softargmax_fwd/bwd, epb_jointloss_fwd_bwd).

Same names / arguments / error behaviour as the reference:
  weighted_{mse,l1,smooth_l1}_loss (:7-47), softmax_integral_tensor (:71-86),
  L1/SmoothL1/L2JointLocationLoss (:93-160; ctor (num_joints, size_average,
  reduce, norm), forward(preds, gt_joints, gt_joints_vis)),
  generate_joint_location_label / reverse_joint_location_label (:170-185),
  get_joint_location_result (:187-207), get_label_func / get_result_func /
  merge_flip_func / get_merge_func (:209-220).
Deviation (documented): L2JointLocationLoss in the reference is broken
(self.output_3d undefined + stray print, :110-112); here it computes the
weighted MSE it was evidently meant to.
The logits may be NCHW-contiguous or the channels_last view PoseResNet returns;
both layouts are handled natively (no transposition pass).

Addition for the VOLUME=False head (pose3d_resnet.py:202-212 returns 2-D heat-maps and a
depth vector; BASELINE north_star "MSE heatmap loss + L1 3D loss fused into one kernel",
SURVEY 8(d) C2(ii)): HeatmapMSELoss / HeatmapJointLoss / heatmap_joint_loss over the single
launch epb_heatmap_joint_loss.  The reference ships no heat-map criterion (only the config
remnants LOSS.USE_TARGET_WEIGHT, lib/core/config.py:32-34); the arithmetic is
torch.nn.functional.mse_loss on the (weighted) maps.
"""
import numpy as np
import torch
import torch.nn as nn

from epipolarpose_b200 import ops as _ops

_KIND = {"mse": 0, "l1": 1, "smoothl1": 2}
_backend = [_ops]     # test hook: tests may swap in the CPU emulation of the C ABI


def _layout_of(preds, J=None, D=None):
    """0: NCHW contiguous, 1: channels_last (NHWC memory).  Otherwise copy.  The channels_last
    kernels read 4 depth bins per thread with one CTA row per pixel: D % 4 == 0 and
    J*D/4 <= 1024; other volumes take the NCHW kernels (any J/D/H/W, like the reference)."""
    if preds.is_contiguous():
        return preds, 0
    if preds.dim() == 4 and preds.permute(0, 2, 3, 1).is_contiguous() \
            and (D is None or (D % 4 == 0 and J * D // 4 <= 1024)):
        return preds, 1
    return preds.contiguous(), 0


def _storage(preds, layout):
    return preds if layout == 0 else preds.permute(0, 2, 3, 1)


class _SoftArgmaxFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, preds, J, D, H, W):
        ops = _backend[0]
        sink = getattr(preds, "_epb_logit_sink", None)     # attached by PoseResNet.forward (_sinks.py)
        preds, layout = _layout_of(preds, J, D)
        N = preds.shape[0]
        coords = torch.empty((N, J * 3), device=preds.device, dtype=torch.float32)
        lse = torch.empty((N * J * 2,), device=preds.device, dtype=torch.float32)
        ops.softargmax_fwd(_storage(preds, layout), layout, N, J, D, H, W, coords, lse)
        ctx.save_for_backward(preds, coords, lse)
        ctx.cfg = (layout, N, J, D, H, W)
        ctx.sink = sink if (sink is not None and layout == 1 and sink.matches(preds)) else None
        return coords

    @staticmethod
    def backward(ctx, dcoords):
        ops = _backend[0]
        preds, coords, lse = ctx.saved_tensors
        layout, N, J, D, H, W = ctx.cfg
        st = _storage(preds, layout)
        sink = ctx.sink
        if sink is not None and not sink.filled:
            # the gradient goes to the network's backward as split planes + bias gradient; autograd
            # carries a zero token (see _sinks.py)
            sink.planes = torch.empty((sink.nplanes,) + tuple(st.shape), device=st.device, dtype=torch.float16)
            sink.sc = torch.empty(2, device=st.device, dtype=torch.float32)
            sink.dbias = torch.empty(J * D, device=st.device, dtype=torch.float32)
            ops.softargmax_bwd_split(st, N, J, D, H, W, coords, lse, dcoords.contiguous(), sink.planes,
                                     sink.sc, sink.dbias,
                                     **({} if sink.nplanes == 2 else {"planes": sink.nplanes}))
            sink.filled = True
            return sink.token.expand(preds.shape), None, None, None, None
        dst = torch.empty_like(st)
        ops.softargmax_bwd(st, layout, N, J, D, H, W, coords, lse, dcoords.contiguous(), dst)
        dl = dst if layout == 0 else dst.permute(0, 3, 1, 2)
        return dl, None, None, None, None


def softmax_integral_tensor(preds, num_joints, output_3d, hm_width, hm_height, hm_depth):
    """reference :71-86.  preds [N, J*D, H, W] -> [N, J*3]."""
    assert output_3d, 'Not Implemented!'
    if preds.dtype != torch.float32:
        raise TypeError("softmax_integral_tensor expects float32 logits")
    assert preds.shape[1] == num_joints * hm_depth and preds.shape[2] == hm_height \
        and preds.shape[3] == hm_width
    return _SoftArgmaxFn.apply(preds, num_joints, hm_depth, hm_height, hm_width)


def _like(x, t, name):
    """target / weights as float32 tensors of x's shape: broadcast the way the reference's
    elementwise arithmetic does (integral_loss.py:12-14), raise where it would raise."""
    t = t.float()
    if t.shape != x.shape:
        try:
            t = torch.broadcast_to(t, x.shape)
        except RuntimeError as e:
            raise RuntimeError("%s of shape %s does not broadcast to the input's %s"
                               % (name, tuple(t.shape), tuple(x.shape))) from e
    return t.contiguous()


class _WeightedLossFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, inp, target, weights, kind, size_average, norm):
        ops = _backend[0]
        x = inp.contiguous()
        dx = torch.empty_like(x)
        loss = torch.empty((), device=x.device, dtype=torch.float32)
        div = float(len(inp)) if size_average else 1.0
        target, weights = _like(x, target, "target"), _like(x, weights, "weights")
        ops.jointloss(x, target, weights, x.numel(),
                      _KIND[kind], norm, div, loss, dx)
        ctx.save_for_backward(dx)
        return loss

    @staticmethod
    def backward(ctx, g):
        (dx,) = ctx.saved_tensors
        return dx * g, None, None, None, None, None


def weighted_mse_loss(input, target, weights, size_average, norm=False):
    return _WeightedLossFn.apply(input, target, weights, "mse", size_average, norm)


def weighted_l1_loss(input, target, weights, size_average, norm=False):
    return _WeightedLossFn.apply(input, target, weights, "l1", size_average, norm)


def weighted_smooth_l1_loss(input, target, weights, size_average, norm=False):
    return _WeightedLossFn.apply(input, target, weights, "smoothl1", size_average, norm)


def _assert_no_grad(tensor):
    assert not tensor.requires_grad, \
        "nn criterions don't compute the gradient w.r.t. targets - please " \
        "mark these tensors as not requiring gradients"


class _JointLocationLoss(nn.Module):
    _kind = None

    def __init__(self, num_joints, size_average=True, reduce=True, norm=False):
        super().__init__()
        self.size_average = size_average
        self.reduce = reduce
        self.num_joints = num_joints
        self.norm = norm

    def forward(self, preds, *args):
        gt_joints, gt_joints_vis = args[0], args[1]
        hm_width = preds.shape[-1]
        hm_height = preds.shape[-2]
        hm_depth = preds.shape[-3] // self.num_joints
        pred_jts = softmax_integral_tensor(preds, self.num_joints, True, hm_width, hm_height, hm_depth)
        _assert_no_grad(gt_joints)
        _assert_no_grad(gt_joints_vis)
        return _WeightedLossFn.apply(pred_jts, gt_joints, gt_joints_vis, self._kind,
                                     self.size_average, self.norm)


class L2JointLocationLoss(_JointLocationLoss):
    _kind = "mse"


class L1JointLocationLoss(_JointLocationLoss):
    _kind = "l1"


class SmoothL1JointLocationLoss(_JointLocationLoss):
    _kind = "smoothl1"


class _HeatmapJointLossFn(torch.autograd.Function):
    """total = hm_scale * mse(w_hm * hm, w_hm * target) + jt_scale * joint_loss(x, t, w)."""

    @staticmethod
    def forward(ctx, hm, target, hm_weight, x, t, w, kind, hm_scale, jt_scale, size_average):
        ops = _backend[0]
        if hm.dtype != torch.float32:
            raise TypeError("heat-map loss expects float32 heat-maps")
        if hm.shape != target.shape:
            raise ValueError("heat-map / target shape mismatch: %s vs %s"
                             % (tuple(hm.shape), tuple(target.shape)))
        N, J = hm.shape[0], hm.shape[1]
        R, HW = N * J, int(np.prod(hm.shape[2:]))
        h = hm.contiguous()
        if target.numel() != h.numel():
            raise ValueError("heat-map target has %d elements, the heat-maps %d" % (target.numel(), h.numel()))
        tg = target.contiguous().float()
        wh = None
        if hm_weight is not None:
            wh = hm_weight.reshape(-1).contiguous().float()
            if wh.numel() != R:
                raise ValueError("heat-map weight must have one entry per (sample, joint)")
        dhm = torch.empty_like(h)
        loss = torch.empty((3,), device=h.device, dtype=torch.float32)
        n, div = 0, 1.0
        xc = tc = wc = dx = None
        if x is not None:
            xc = x.contiguous()
            tc, wc = _like(xc, t, "gt_jts"), _like(xc, w, "jts_weight")
            n = xc.numel()
            div = float(len(x)) if size_average else 1.0
            dx = torch.empty_like(xc)
        ops.heatmap_joint_loss(h, tg, wh, R, HW, hm_scale, xc, tc, wc, n, _KIND[kind], div,
                               jt_scale, loss, dhm, dx)
        ctx.save_for_backward(dhm, dx if dx is not None else dhm.new_empty(0))
        ctx.has_x = x is not None
        return loss            # [loss_hm, loss_jt, total]; only `total` carries gradient

    @staticmethod
    def backward(ctx, g):
        dhm, dx = ctx.saved_tensors
        gt = g[2]
        return (dhm * gt, None, None, dx * gt if ctx.has_x else None, None, None, None, None,
                None, None)


def heatmap_joint_loss(heatmaps, hm_target, hm_weight=None, pred_jts=None, gt_jts=None,
                       jts_weight=None, kind="l1", hm_scale=1.0, jt_scale=1.0, size_average=True):
    """One fused launch.  heatmaps / hm_target [N, J, H, W] float32, hm_weight [N, J(,1)] or
    None, pred_jts / gt_jts / jts_weight [N, J*3] or None.
    Returns (total, parts): total = hm_scale*loss_hm + jt_scale*loss_jt (differentiable w.r.t.
    heatmaps and pred_jts), parts = tensor [loss_hm, loss_jt] (detached)."""
    if pred_jts is not None:
        _assert_no_grad(gt_jts)
        _assert_no_grad(jts_weight)
    _assert_no_grad(hm_target)
    out = _HeatmapJointLossFn.apply(heatmaps, hm_target, hm_weight, pred_jts, gt_jts, jts_weight,
                                    kind, float(hm_scale), float(jt_scale), size_average)
    return out[2], out[:2].detach()


class HeatmapMSELoss(nn.Module):
    """criterion(output [N,J,H,W], target [N,J,H,W], target_weight [N,J,1]) -> mean squared
    error of the (weighted, when use_target_weight) heat-maps."""

    def __init__(self, use_target_weight=False):
        super().__init__()
        self.use_target_weight = use_target_weight

    def forward(self, output, target, target_weight=None):
        w = target_weight if self.use_target_weight else None
        if self.use_target_weight and target_weight is None:
            raise ValueError("use_target_weight=True needs target_weight")
        return heatmap_joint_loss(output, target, w)[0]


class HeatmapJointLoss(nn.Module):
    """criterion((heatmaps, pred_jts), (hm_target, hm_weight), gt_joints, gt_joints_vis):
    heat-map MSE + jt_scale * L1 / SmoothL1 / MSE joint-location loss, one kernel launch.
    `last_parts` holds [loss_hm, loss_jt] of the most recent call."""

    def __init__(self, num_joints, kind="l1", hm_scale=1.0, jt_scale=1.0, size_average=True,
                 use_target_weight=True):
        super().__init__()
        if kind not in _KIND:
            raise ValueError("unknown joint loss kind %r" % (kind,))
        self.num_joints, self.kind = num_joints, kind
        self.hm_scale, self.jt_scale = hm_scale, jt_scale
        self.size_average, self.use_target_weight = size_average, use_target_weight
        self.last_parts = None

    def forward(self, preds, hm_target, gt_joints, gt_joints_vis, hm_weight=None):
        heatmaps, pred_jts = preds
        total, parts = heatmap_joint_loss(heatmaps, hm_target,
                                          hm_weight if self.use_target_weight else None,
                                          pred_jts, gt_joints, gt_joints_vis, self.kind,
                                          self.hm_scale, self.jt_scale, self.size_average)
        self.last_parts = parts
        return total


def get_loss_func(config):
    if config.loss_type == 'L1':
        return L1JointLocationLoss(config.output_3d)
    elif config.loss_type == 'L2':
        return L2JointLocationLoss(config.output_3d)
    assert 0, 'Error. Unknown heatmap type {}'.format(config.heatmap_type)


def generate_joint_location_label(patch_width, patch_height, joints, joints_vis):
    joints[:, 0] = joints[:, 0] / patch_width - 0.5
    joints[:, 1] = joints[:, 1] / patch_height - 0.5
    joints[:, 2] = joints[:, 2] / patch_width
    return joints.reshape((-1)), joints_vis.reshape((-1))


def reverse_joint_location_label(patch_width, patch_height, joints):
    joints = joints.reshape((joints.shape[0] // 3, 3))
    joints[:, 0] = (joints[:, 0] + 0.5) * patch_width
    joints[:, 1] = (joints[:, 1] + 0.5) * patch_height
    joints[:, 2] = joints[:, 2] * patch_width
    return joints


def get_joint_location_coords(preds):
    """Device-side half of get_joint_location_result: [N, J*3] float32 CUDA."""
    hm_width, hm_height = preds.shape[-1], preds.shape[-2]
    hm_depth = hm_width                       # reference :191-192 assumes D == W
    num_joints = preds.shape[1] // hm_depth
    with torch.no_grad():
        return softmax_integral_tensor(preds, num_joints, True, hm_width, hm_height, hm_depth)


def get_joint_location_result(patch_width, patch_height, preds):
    """reference :187-207 -> numpy float64 [N, J, 4] (x, y, z in patch px, score 1)."""
    coords = get_joint_location_coords(preds).detach().cpu().numpy().astype(float)
    coords = coords.reshape((coords.shape[0], coords.shape[1] // 3, 3))
    coords[:, :, 0] = (coords[:, :, 0] + 0.5) * patch_width
    coords[:, :, 1] = (coords[:, :, 1] + 0.5) * patch_height
    coords[:, :, 2] = coords[:, :, 2] * patch_width
    scores = np.ones((coords.shape[0], coords.shape[1], 1), dtype=float)
    return np.concatenate((coords, scores), axis=2)


def get_label_func():
    return generate_joint_location_label


def get_result_func():
    return get_joint_location_result


def merge_flip_func(a, b, flip_pair):
    return a


def get_merge_func(loss_config):
    return merge_flip_func
