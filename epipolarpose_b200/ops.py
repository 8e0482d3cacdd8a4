"""Thin torch-tensor wrappers over the libepb.so C ABI (include/epb.h).

torch is plumbing only here: it owns device memory and the current stream;
every op below is one or more hand-written sm_100a kernels.  Each wrapper
validates dtype / device / contiguity and raises on any failure -- there is no
CPU or eager fallback.  `launches` counts kernel launches issued through this
module (bench.py reports it as gpu_launches).
"""
import ctypes

import torch

from . import _lib
from ._lib import ConvGeom

launches = 0

# kernels launched per C-ABI call (for the gpu_launches accounting)
_KERNELS_PER_CALL = {
    "epb_softargmax_fwd": 2, "epb_bn_bwd_apply": 2, "epb_colsum": 3,
    "epb_split16_batch": 3, "epb_split16": 3, "epb_bn_bwd_apply_split": 2, "epb_conv16_wgrad": 2,
    "epb_bn_bwd_reduce_mx": 2, "epb_bn_bwd_split": 3, "epb_softargmax_bwd_split": 3,
    "epb_patch_sample": 2, "epb_patch_sample_occ": 2,
}


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t, dtype=torch.float32):
    if t is None:
        return None
    if not t.is_cuda:
        raise _lib.EpbError("tensor must live on a CUDA device (no CPU fallback)")
    if t.dtype != dtype:
        raise _lib.EpbError("expected dtype %s, got %s" % (dtype, t.dtype))
    if t.device.index != torch.cuda.current_device():
        # the stream handed to the C ABI is the CURRENT device's; a tensor of another device
        # would be dereferenced by a kernel running on the wrong GPU
        raise _lib.EpbError("tensor lives on cuda:%d but the current device is cuda:%d (wrap the call in "
                            "torch.cuda.device(tensor.device))" % (t.device.index, torch.cuda.current_device()))
    if not t.is_contiguous():
        raise _lib.EpbError("tensor must be contiguous")
    return ctypes.c_void_p(t.data_ptr())


def _call(name, *args):
    global launches
    _lib.call(name, *args)
    launches += _KERNELS_PER_CALL.get(name, 1)


def device_check():
    _lib.call("epb_device_check")


# ------------------------------------------------------------------ conv family

def make_geom(N, Hi, Wi, Cin, Ho, Wo, Cout, Hp, Wp, os, ph, pw, is_, taps, Tw,
              in_relu=0, accumulate=0, precision=0):
    """taps: list of (dh, dw, wt)."""
    g = ConvGeom()
    g.N, g.Hi, g.Wi, g.Cin = N, Hi, Wi, Cin
    g.Ho, g.Wo, g.Cout = Ho, Wo, Cout
    g.Hp, g.Wp, g.os, g.ph, g.pw, g.is_ = Hp, Wp, os, ph, pw, is_
    g.T = len(taps)
    if g.T > _lib.EPB_MAX_TAPS:
        raise _lib.EpbError("too many taps")
    for i, (dh, dw, wt) in enumerate(taps):
        g.dh[i], g.dw[i], g.wt[i] = dh, dw, wt
    g.Tw = Tw
    g.in_relu, g.accumulate, g.precision = in_relu, accumulate, precision
    return g


def conv_fprop(g, x, w, out, in_scale=None, in_shift=None, bias=None, stats=None):
    _call("epb_conv_fprop", ctypes.byref(g), _p(x), _p(w), _p(in_scale), _p(in_shift),
          _p(bias), _p(out), _p(stats, torch.float64), _stream())


def conv_wgrad(g, x, dout, dw, in_scale=None, in_shift=None):
    _call("epb_conv_wgrad", ctypes.byref(g), _p(x), _p(dout), _p(in_scale), _p(in_shift),
          _p(dw), _stream())


def pack_weight(src, dst, A, B, kh, kw, swap, ypad, unpack=0):
    _call("epb_pack_weight", _p(src), _p(dst), A, B, kh, kw, swap, ypad, unpack, _stream())


class PackBatch:
    """A fixed list of pack / unpack jobs (epb_pack_job, include/epb.h) with its device table.
    jobs: (src, dst, A, B, T, swap, ypad, unpack, x_pitch) with src / dst tensors whose
    storage must stay where it is for the lifetime of the batch."""

    def __init__(self, jobs):
        import struct
        self.jobs = list(jobs)
        self.keep = [(j[0], j[1]) for j in self.jobs]
        blob, first = b"", 0
        for (src, dst, A, B, T, swap, ypad, unpack, xp) in self.jobs:
            X = B if swap else A
            blob += struct.pack("<QQ8iqq", src.data_ptr(), dst.data_ptr(), A, B, T, swap, ypad,
                                unpack, xp, 0, first, 0)
            first += (X * T * ypad + 1023) // 1024
        self.total_blocks = first
        dev = self.jobs[0][1].device
        self.table = torch.frombuffer(bytearray(blob), dtype=torch.uint8).to(dev)

    def pointers(self):
        return tuple((j[0].data_ptr(), j[1].data_ptr()) for j in self.jobs)


def pack_weight_batch(batch):
    _call("epb_pack_weight_batch", _p(batch.table, torch.uint8), len(batch.jobs), batch.total_blocks, _stream())


def im2col(x, col, N, Hi, Wi, pitch, C, kh, kw, stride, pad, Ho, Wo, Kpad):
    _call("epb_im2col", _p(x), _p(col), N, Hi, Wi, pitch, C, kh, kw, stride, pad, Ho, Wo, Kpad,
          _stream())


def nchw_to_nhwc(src, dst, N, C, H, W, Cpad):
    _call("epb_nchw_to_nhwc", _p(src), _p(dst), N, C, H, W, Cpad, _stream())


def nhwc_to_nchw(src, dst, N, C, H, W, Cpad):
    _call("epb_nhwc_to_nchw", _p(src), _p(dst), N, C, H, W, Cpad, _stream())


# ------------------------------------------------------------------ BN family

def channel_stats(x, M, C, stats):
    _call("epb_channel_stats", _p(x), M, C, _p(stats, torch.float64), _stream())


def bn_finalize(stats, M, C, gamma, beta, eps, momentum, running_mean, running_var,
                scale, shift, mean, invstd):
    _call("epb_bn_finalize", _p(stats, torch.float64), M, C, _p(gamma), _p(beta), eps, momentum,
          _p(running_mean), _p(running_var), _p(scale), _p(shift), _p(mean), _p(invstd), _stream())


def bn_eval_affine(C, gamma, beta, running_mean, running_var, eps, scale, shift):
    _call("epb_bn_eval_affine", C, _p(gamma), _p(beta), _p(running_mean), _p(running_var), eps,
          _p(scale), _p(shift), _stream())


def bn_act(x, scale, shift, r, rscale, rshift, relu, y, M, C):
    _call("epb_bn_act", _p(x), _p(scale), _p(shift), _p(r), _p(rscale), _p(rshift), int(relu),
          _p(y), M, C, _stream())


def bn_relu_maxpool(x, scale, shift, y, argidx, N, H, W, C):
    _call("epb_bn_relu_maxpool", _p(x), _p(scale), _p(shift), _p(y), _p(argidx, torch.uint8),
          N, H, W, C, _stream())


def maxpool_bwd(dy, argidx, dx, N, H, W, C):
    _call("epb_maxpool_bwd", _p(dy), _p(argidx, torch.uint8), _p(dx), N, H, W, C, _stream())


def bn_bwd_reduce(dy, x, y_out, scale, shift, mean, invstd, relu, M, C, sums):
    _call("epb_bn_bwd_reduce", _p(dy), _p(x), _p(y_out), _p(scale), _p(shift), _p(mean),
          _p(invstd), int(relu), M, C, _p(sums, torch.float64), _stream())


def bn_bwd_apply(dy, x, y_out, scale, shift, mean, invstd, gamma, relu, sums, M, C, dx,
                 dgamma, dbeta):
    _call("epb_bn_bwd_apply", _p(dy), _p(x), _p(y_out), _p(scale), _p(shift), _p(mean),
          _p(invstd), _p(gamma), int(relu), _p(sums, torch.float64), M, C, _p(dx), _p(dgamma),
          _p(dbeta), _stream())


def add_masked(a, b, mask_src, dx, n):
    _call("epb_add_masked", _p(a), _p(b), _p(mask_src), _p(dx), n, _stream())


def avgpool(x, y, N, HW, C):
    _call("epb_avgpool", _p(x), _p(y), N, HW, C, _stream())


def avgpool_bwd(dy, dx, N, HW, C, accumulate):
    _call("epb_avgpool_bwd", _p(dy), _p(dx), N, HW, C, int(accumulate), _stream())


def colsum(x, M, C, out):
    _call("epb_colsum", _p(x), M, C, _p(out), _stream())


# ------------------------------------------------------------------ split-fp16 ("f16x3") family
# A split tensor is a torch.float16 tensor [2, ...] (hi plane, lo plane) plus a device
# float32[2] = (s, 1/s).  `planes=1` selects the single-pass layout [1, ...] (hi plane only,
# include/epb.h): producers write the hi plane alone, readers and GEMMs read it alone.

_H = torch.float16


def act_scale(stats, scale, shift, M, C, stats2, scale2, shift2, res_sc, sc):
    _call("epb_act_scale", _p(stats, torch.float64), _p(scale), _p(shift), M, C,
          _p(stats2, torch.float64), _p(scale2), _p(shift2), _p(res_sc), _p(sc), _stream())


def bn_finalize_scale(stats, M, C, gamma, beta, eps, momentum, running_mean, running_var, scale, shift,
                      mean, invstd, stats2, scale2, shift2, res_sc, sc):
    _call("epb_bn_finalize_scale", _p(stats, torch.float64), M, C, _p(gamma), _p(beta), eps, momentum,
          _p(running_mean), _p(running_var), _p(scale), _p(shift), _p(mean), _p(invstd),
          _p(stats2, torch.float64), _p(scale2), _p(shift2), _p(res_sc), _p(sc), _stream())


def bn_act_split(x, scale, shift, r, rscale, rshift, r_split, r_sc, relu, M, C, y, y_sc, mask_bits=None,
                 planes=2):
    _call("epb_bn_act_split", _p(x), _p(scale), _p(shift), _p(r), _p(rscale), _p(rshift),
          _p(r_split, _H), _p(r_sc), int(relu), M, C, _p(y, _H), _p(y_sc), _p(mask_bits, torch.uint8),
          planes, _stream())


def bn_relu_maxpool_split(x, scale, shift, y, y_sc, argidx, N, H, W, C, planes=2):
    _call("epb_bn_relu_maxpool_split", _p(x), _p(scale), _p(shift), _p(y, _H), _p(y_sc),
          _p(argidx, torch.uint8), N, H, W, C, planes, _stream())


def im2col_split(img, col, col_sc, N, C, Hi, Wi, kh, kw, stride, pad, Ho, Wo, Kpad, planes=2):
    _call("epb_im2col_split", _p(img), _p(col, _H), _p(col_sc), N, C, Hi, Wi, kh, kw, stride, pad,
          Ho, Wo, Kpad, planes, _stream())


class SplitBatch:
    """A fixed list of fp32 -> split conversions (epb_split_job) with its device table.
    jobs: (src fp32 [n], dst fp16 [planes][n], sc fp32 [2]); the tensors must stay where they are."""

    def __init__(self, jobs, planes=2):
        import struct
        self.jobs = list(jobs)
        self.planes = planes
        blob, first = b"", 0
        for (src, dst, sc) in self.jobs:
            n = src.numel()
            assert dst.numel() == planes * n and dst.dtype == _H and sc.numel() == 2
            blob += struct.pack("<QQQqq", src.data_ptr(), dst.data_ptr(), sc.data_ptr(), n, first)
            first += (n + 2047) // 2048
        self.total_blocks = first
        dev = self.jobs[0][1].device
        self.table = torch.frombuffer(bytearray(blob), dtype=torch.uint8).to(dev)
        self.amax = torch.zeros(len(self.jobs), dtype=torch.int32, device=dev)


def split16(src, dst, sc, amax_ws, planes=2):
    _call("epb_split16", _p(src), src.numel(), _p(dst, _H), _p(sc), _p(amax_ws, torch.int32), planes,
          _stream())


def split16_batch(batch):
    _call("epb_split16_batch", _p(batch.table, torch.uint8), len(batch.jobs), batch.total_blocks,
          _p(batch.amax, torch.int32), batch.planes, _stream())


def conv16_fprop(g, x, x_sc, w, w_sc, out, bias=None, stats=None, planes=2):
    _call("epb_conv16_fprop", ctypes.byref(g), _p(x, _H), _p(x_sc), _p(w, _H), _p(w_sc), _p(bias),
          _p(out), _p(stats, torch.float64), planes, _stream())


def conv16_wgrad(g, x, x_sc, dout, dout_sc, dw, ws, planes=2):
    _call("epb_conv16_wgrad", ctypes.byref(g), _p(x, _H), _p(x_sc), _p(dout, _H), _p(dout_sc),
          _p(dw), _p(ws), ws.numel() if ws is not None else 0, planes, _stream())


def bn_bwd_reduce_mx(dy, x, mask_hi, scale, shift, mean, invstd, relu, M, C, sums, maxes):
    _call("epb_bn_bwd_reduce_mx", _p(dy), _p(x), _p(mask_hi, _H), _p(scale), _p(shift), _p(mean),
          _p(invstd), int(relu), M, C, _p(sums, torch.float64), _p(maxes), _stream())


def bn_bwd_apply_split(dy, x, mask_hi, scale, shift, mean, invstd, gamma, relu, sums, maxes, M, C,
                       dz, dz_sc, dy_masked, dgamma, dbeta, planes=2):
    _call("epb_bn_bwd_apply_split", _p(dy), _p(x), _p(mask_hi, _H), _p(scale), _p(shift), _p(mean),
          _p(invstd), _p(gamma), int(relu), _p(sums, torch.float64), _p(maxes), M, C, _p(dz, _H),
          _p(dz_sc), _p(dy_masked), _p(dgamma), _p(dbeta), planes, _stream())


def bn_bwd_split(dy, x, mask_hi, scale, shift, mean, invstd, gamma, relu, M, C, dz, dz_sc, dy_masked,
                 dgamma, dbeta, mask_bits=None, planes=2):
    _call("epb_bn_bwd_split", _p(dy), _p(x), _p(mask_hi, _H), _p(mask_bits, torch.uint8), _p(scale),
          _p(shift), _p(mean),
          _p(invstd), _p(gamma), int(relu), M, C, _p(dz, _H), _p(dz_sc), _p(dy_masked), _p(dgamma),
          _p(dbeta), planes, _stream())


def avgpool_split(x, x_sc, y, N, HW, C, planes=2):
    _call("epb_avgpool_split", _p(x, _H), _p(x_sc), _p(y), N, HW, C, planes, _stream())


# ------------------------------------------------------------------ decode / loss

def softargmax_fwd(logits, layout, N, J, D, H, W, coords, lse):
    _call("epb_softargmax_fwd", _p(logits), layout, N, J, D, H, W, _p(coords), _p(lse), _stream())


def softargmax_bwd(logits, layout, N, J, D, H, W, coords, lse, dcoords, dlogits):
    _call("epb_softargmax_bwd", _p(logits), layout, N, J, D, H, W, _p(coords), _p(lse),
          _p(dcoords), _p(dlogits), _stream())


def jointloss(x, t, w, n, kind, norm, div, loss, dx):
    _call("epb_jointloss_fwd_bwd", _p(x), _p(t), _p(w), n, kind, int(norm), float(div),
          _p(loss), _p(dx), _stream())


def heatmap_joint_loss(hm, target, hm_weight, R, HW, hm_scale, x, t, w, n, kind, div, jt_scale,
                       loss, dhm, dx):
    _call("epb_heatmap_joint_loss", _p(hm), _p(target), _p(hm_weight), R, HW, float(hm_scale),
          _p(x), _p(t), _p(w), n, kind, float(div), float(jt_scale), _p(loss), _p(dhm), _p(dx),
          _stream())


def argmax2d(hm, NJ, H, W, idx, maxval, preds):
    _call("epb_argmax2d", _p(hm), NJ, H, W, _p(idx, torch.int32), _p(maxval), _p(preds), _stream())


def softargmax_bwd_split(logits, N, J, D, H, W, coords, lse, dcoords, dlogits16, sc, dbias, planes=2):
    _call("epb_softargmax_bwd_split", _p(logits), N, J, D, H, W, _p(coords), _p(lse), _p(dcoords),
          _p(dlogits16, _H), _p(sc), _p(dbias), planes, _stream())


def final_preds(hm, N, J, H, W, center, scale, post_process, preds, maxvals):
    _call("epb_final_preds", _p(hm), N, J, H, W, _p(center, torch.float64), _p(scale, torch.float64),
          int(bool(post_process)), _p(preds), _p(maxvals), _stream())


# ------------------------------------------------------------------ geometry (fp64)

def patch_to_image(coords, box, B, J, patch_w, patch_h, rect3d_w, kps):
    _call("epb_patch_to_image", _p(coords), _p(box, torch.float64), B, J, float(patch_w),
          float(patch_h), float(rect3d_w), _p(kps, torch.float64), _stream())


def triangulate(u1, u2, stride_u, P1, P2, NP, J, method, tol, X, status):
    _call("epb_triangulate", _p(u1, torch.float64), _p(u2, torch.float64), stride_u,
          _p(P1, torch.float64), _p(P2, torch.float64), NP, J, method, float(tol),
          _p(X, torch.float64), _p(status, torch.int32), _stream())


def add3(a, b, c, out, n):
    _call("epb_add3", _p(a), _p(b), _p(c), _p(out), n, _stream())


def mask_scale(x, mask, scale, out, n):
    _call("epb_mask_scale", _p(x), _p(mask, torch.uint8), float(scale), _p(out), n, _stream())


def patch_sample(img_base, img_off, img_hwp, box, flip, color, mean_std, B, patch_w, patch_h, out, trans):
    """mean_std: None or a sequence of 6 floats (mean RGB, std RGB) -- passed as a HOST array."""
    ms = None
    if mean_std is not None:
        ms = (ctypes.c_double * 6)(*[float(v) for v in mean_std])
    _call("epb_patch_sample", _p(img_base, torch.uint8), _p(img_off, torch.int64), _p(img_hwp, torch.int32),
          _p(box, torch.float64), _p(flip, torch.int32), _p(color), ms, B, patch_w, patch_h, _p(out),
          _p(trans, torch.float64), _stream())


def patch_sample_occ(img_base, img_off, img_hwp, box, flip, color, mean_std, B, patch_w, patch_h,
                     occ_base, occ_desc, occ_count, out, trans):
    ms = None
    if mean_std is not None:
        ms = (ctypes.c_double * 6)(*[float(v) for v in mean_std])
    _call("epb_patch_sample_occ", _p(img_base, torch.uint8), _p(img_off, torch.int64),
          _p(img_hwp, torch.int32), _p(box, torch.float64), _p(flip, torch.int32), _p(color), ms, B,
          patch_w, patch_h, _p(occ_base, torch.uint8), _p(occ_desc, torch.int64),
          _p(occ_count, torch.int32), _p(out), _p(trans, torch.float64), _stream())


def patch_joints(joints, box, trans, B, J, patch_w, patch_h, rect_3d_w, depth_in_image, label):
    _call("epb_patch_joints", _p(joints, torch.float64), _p(box, torch.float64), _p(trans, torch.float64),
          B, J, float(patch_w), float(patch_h), float(rect_3d_w), int(depth_in_image),
          _p(label, torch.float64), _stream())


def h36m_eval(pred, gt, cam, S, J, root, j14mask, pck_thr, metrics, per_joint, pck, poses):
    _call("epb_h36m_eval", _p(pred, torch.float64), _p(gt, torch.float64), _p(cam, torch.float64),
          S, J, root, int(j14mask), float(pck_thr), _p(metrics, torch.float64),
          _p(per_joint, torch.float64), _p(pck, torch.int32), _p(poses, torch.float64), _stream())


def triangulate_nview(u, stride_u, P, NT, V, J, X, status):
    _call("epb_triangulate_nview", _p(u, torch.float64), stride_u, _p(P, torch.float64), NT, V, J,
          _p(X, torch.float64), _p(status, torch.int32), _stream())


def project_labels(X, cam, box, B, J, patch_w, patch_h, rect3d_w, label, weight):
    _call("epb_project_labels", _p(X, torch.float64), _p(cam, torch.float64),
          _p(box, torch.float64), B, J, float(patch_w), float(patch_h), float(rect3d_w),
          _p(label), _p(weight), _stream())


# ------------------------------------------------------------------ optimiser
def sumsq(x, n, total):
    _call("epb_sumsq", _p(x), n, _p(total, torch.float64), _stream())


def clip_scale(x, n, total, max_norm):
    _call("epb_clip_scale", _p(x), n, _p(total, torch.float64), float(max_norm), _stream())


def adam_step(param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay, step,
              grad_scale=1.0):
    _call("epb_adam_step", _p(param), _p(grad), _p(exp_avg), _p(exp_avg_sq), n, lr, beta1, beta2,
          eps, weight_decay, step, grad_scale, _stream())


def sgd_step(param, grad, buf, n, lr, momentum, weight_decay, nesterov, first_step,
             grad_scale=1.0):
    _call("epb_sgd_step", _p(param), _p(grad), _p(buf), n, lr, momentum, weight_decay,
          int(nesterov), int(first_step), grad_scale, _stream())


def adam_step_dev(param, grad, exp_avg, exp_avg_sq, n, hyper, step_dev):
    _call("epb_adam_step_dev", _p(param), _p(grad), _p(exp_avg), _p(exp_avg_sq), n, _p(hyper),
          _p(step_dev, torch.int32), _stream())


def sgd_step_dev(param, grad, buf, n, hyper, step_dev):
    _call("epb_sgd_step_dev", _p(param), _p(grad), _p(buf), n, _p(hyper),
          _p(step_dev, torch.int32), _stream())
