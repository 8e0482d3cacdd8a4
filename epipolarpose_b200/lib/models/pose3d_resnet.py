"""PoseResNet on the B200 engine -- host-side mirror of the reference
lib/models/pose3d_resnet.py surface: `get_pose_net(cfg, is_train, **kw)`
(:295-305), `PoseResNet(block, layers, cfg)` (:91-126), `BasicBlock`,
`Bottleneck`, `resnet_spec` (:288-292), `.init_weights(pretrained)` (:214-255),
`.load_pretrained_pose_model` (:257-286).

The module tree is a parameter CONTAINER only: it reproduces the reference's
state_dict keys / shapes / default initialisation (Conv2d [O,I,kh,kw],
ConvTranspose2d [I,O,kh,kw], BatchNorm2d weight/bias/running_*/num_batches_tracked)
so checkpoints interchange, but no torch.nn forward is ever executed: forward
and backward run in epipolarpose_b200.net.Engine on hand-written sm_100a kernels
(libepb.so).  There is no CPU / eager fallback; a non-CUDA input raises.
"""
import logging
import os
from collections import OrderedDict

import torch
import torch.nn as nn

from epipolarpose_b200 import net as _net
from epipolarpose_b200 import net16 as _net16
from epipolarpose_b200 import _sinks

BN_MOMENTUM = 0.1
logger = logging.getLogger(__name__)

# f16x3: split-fp16 operands, three kind::f16 tensor passes (net16.Engine16); plans with
# channel counts outside whole 64-element TMA boxes keep the 3xTF32 engine.
# f16: the same engine on the hi planes alone, one kind::f16 pass (TF32-class operands); its
# fall-back for such plans is the single-pass TF32 engine.
_PRECISIONS = {"fp32": 0, "tf32": 1, "tf32x3": 3, "f16x3": 4, "f16": 5}
_SPLIT_PLANES = {4: 2, 5: 1}           # Engine16 plane count of the split precisions
_FALLBACK = {4: 3, 5: 1}               # net.Engine precision when net16 does not take the plan
DEFAULT_PRECISION = "f16x3"


def _no_forward(self, *a, **k):
    raise RuntimeError("parameter container: compute runs in epipolarpose_b200.net.Engine")


class _Conv(nn.Conv2d):
    forward = _no_forward


class _Deconv(nn.ConvTranspose2d):
    forward = _no_forward


class _BN(nn.BatchNorm2d):
    forward = _no_forward


class _Linear(nn.Linear):
    forward = _no_forward


class _ReLU(nn.Module):          # keeps deconv_layers.{2,5,8} index slots (no params)
    forward = _no_forward


class BasicBlock(nn.Module):
    """Parameter container for reference :19-47."""
    expansion = 1

    def __init__(self, inplanes, planes, stride=1, downsample=None):
        super().__init__()
        self.conv1 = _Conv(inplanes, planes, 3, stride, 1, bias=False)
        self.bn1 = _BN(planes, momentum=BN_MOMENTUM)
        self.conv2 = _Conv(planes, planes, 3, 1, 1, bias=False)
        self.bn2 = _BN(planes, momentum=BN_MOMENTUM)
        self.downsample = downsample
        self.stride = stride

    forward = _no_forward


class Bottleneck(nn.Module):
    """Parameter container for reference :50-88."""
    expansion = 4

    def __init__(self, inplanes, planes, stride=1, downsample=None):
        super().__init__()
        self.conv1 = _Conv(inplanes, planes, 1, bias=False)
        self.bn1 = _BN(planes, momentum=BN_MOMENTUM)
        self.conv2 = _Conv(planes, planes, 3, stride, 1, bias=False)
        self.bn2 = _BN(planes, momentum=BN_MOMENTUM)
        self.conv3 = _Conv(planes, planes * 4, 1, bias=False)
        self.bn3 = _BN(planes * 4, momentum=BN_MOMENTUM)
        self.downsample = downsample
        self.stride = stride

    forward = _no_forward


class _PoseNetFn(torch.autograd.Function):
    """autograd bridge: one node for the whole network."""

    @staticmethod
    def forward(ctx, module, x, grad_mode, *flat_params):
        names = module._param_names
        params = dict(zip(names, flat_params))
        for k, b in module.named_buffers():
            params[k] = b
        need_grad = grad_mode and any(p.requires_grad for p in flat_params)
        eng = module._engine()
        logits, depth, saved = eng.forward(x, params, training=module.training, save=need_grad)
        ctx.module, ctx.saved_state, ctx.params = module, saved, params
        ctx.has_depth = depth is not None
        fin = module._plan.final
        N, Ho, Wo, Cp = logits.shape
        ctx.sink = module._last_sink = None
        if module.volume:
            out = logits.permute(0, 3, 1, 2)          # NCHW view, channels_last memory
            if Cp != fin.cout:
                out = out[:, :fin.cout]
            elif need_grad and module.training and module.fused_head_gradient \
                    and getattr(eng, "takes_logit_sink", lambda: False)():
                # the criterion may hand the logit gradient over as split planes (_sinks.py)
                ctx.sink = module._last_sink = _sinks.LogitGradSink(out, eng.planes)
            return out
        hm = torch.empty((N, fin.cout, Ho, Wo), device=x.device, dtype=torch.float32)
        eng.ops.nhwc_to_nchw(logits, hm, N, fin.cout, Ho, Wo, Cp)
        return hm, depth.reshape(N, -1)

    @staticmethod
    def backward(ctx, *gouts):
        module, S, params = ctx.module, ctx.saved_state, ctx.params
        if S is None:
            raise RuntimeError("backward through a forward that ran without grad")
        if not module.training:
            raise RuntimeError("backward in eval() mode is not supported (reference trains in train())")
        eng = module._engine()
        ops = eng.ops
        fin = module._plan.final
        g0 = gouts[0]
        N, Ho, Wo = S["N"], g0.shape[2], g0.shape[3]
        sink, head = getattr(ctx, "sink", None), None
        if sink is not None and sink.filled:
            if sink.is_token(g0):
                head = sink                             # the whole gradient is in the sink
            else:
                # the logits had other consumers too: their (fp32) gradients accumulated onto the
                # zero token; add the sink's share back and take the fp32 route
                g0 = g0 + sink.dense().permute(0, 3, 1, 2)
        nhwc = g0.permute(0, 2, 3, 1)
        if head is not None:
            dlogits = None
        elif fin.cout_p == fin.cout and nhwc.is_contiguous():
            dlogits = nhwc                              # zero-copy (channels_last gradient)
        else:
            dlogits = torch.zeros((N, Ho, Wo, fin.cout_p), device=g0.device, dtype=torch.float32)
            ops.nchw_to_nhwc(g0.contiguous(), dlogits, N, fin.cout, Ho, Wo, fin.cout_p)
        ddepth = None
        if ctx.has_depth and len(gouts) > 1 and gouts[1] is not None:
            ddepth = gouts[1].contiguous()
        # one flat gradient buffer in parameter order (single NCCL all-reduce, fused Adam)
        names = module._param_names
        sizes = [params[n].numel() for n in names]
        padded = [(s + 3) // 4 * 4 for s in sizes]
        # The engine writes into a PERSISTENT staging buffer (its batched gradient unpack and
        # scratch tables are keyed on these addresses); autograd gets a fresh copy every step,
        # so accumulating into / keeping p.grad across steps stays correct.
        stage = getattr(module, "_grad_stage", None)
        if stage is None or stage[0].device != g0.device or stage[0].numel() != sum(padded):
            sflat = torch.zeros(sum(padded), device=g0.device, dtype=torch.float32)
            sgrads, off = {}, 0
            for n, s, ps in zip(names, sizes, padded):
                sgrads[n] = sflat[off:off + s].view(params[n].shape)
                off += ps
            stage = module._grad_stage = (sflat, sgrads)
        sflat, sgrads = stage
        sflat.zero_()
        # pure data parallel over view-tuples: the flat gradient is all-reduced in FIVE stage
        # slices (net.STAGES), each issued as soon as the backward pass has completed it, so
        # all but the last (stem + layer1, < 1 MB) overlap the remaining backward kernels
        import torch.distributed as dist
        works = []
        on_stage = None
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1 \
                and module.allreduce_grads:
            bounds = getattr(module, "_stage_bounds", None)
            if bounds is None:
                bounds, off = {}, 0
                for n, ps in zip(names, padded):
                    k = _net.stage_of(n)
                    a, b = bounds.get(k, (off, off))
                    bounds[k] = (min(a, off), max(b, off + ps))
                    off += ps
                module._stage_bounds = bounds

            def on_stage(k):
                if k in bounds:
                    a, b = bounds[k]
                    works.append(dist.all_reduce(sflat[a:b], op=dist.ReduceOp.AVG, async_op=True))
        if head is not None:
            eng.backward(S, None, ddepth, params, sgrads, on_stage=on_stage, head=head)
        else:
            eng.backward(S, dlogits, ddepth, params, sgrads, on_stage=on_stage)
        if sink is not None:
            sink.planes = sink.sc = sink.dbias = None       # the planes are as large as the logits: let them go
            module._last_sink = None
        for w_ in works:
            w_.wait()                                   # the current stream waits for the collectives
        flat = sflat.clone()
        grads, off = {}, 0
        for n, s, ps in zip(names, sizes, padded):
            grads[n] = flat[off:off + s].view(params[n].shape)
            off += ps
        ctx.saved_state = None
        return (None, None, None) + tuple(grads[n] if params[n].requires_grad else None for n in names)


class PoseResNet(nn.Module):

    def __init__(self, block, layers, cfg, **kwargs):
        super().__init__()
        extra = cfg.MODEL.EXTRA
        self.inplanes = 64
        self.deconv_with_bias = extra.DECONV_WITH_BIAS
        self.volume = cfg.MODEL.VOLUME
        self.allreduce_grads = kwargs.get("allreduce_grads", True)
        # set by the training loops (lib/core/function.py) for the duration of their forward: the
        # criterion may then pass the logit gradient to backward() as split planes (_sinks.py)
        self.fused_head_gradient = False
        prec = kwargs.get("precision", getattr(cfg.MODEL, "PRECISION", None)) or \
            os.environ.get("EPB_PRECISION", DEFAULT_PRECISION)
        self.precision = _PRECISIONS[os.environ.get("EPB_PRECISION", prec)]
        self.conv1 = _Conv(3, 64, 7, 2, 3, bias=False)
        self.bn1 = _BN(64, momentum=BN_MOMENTUM)
        self.layer1 = self._make_layer(block, 64, layers[0])
        self.layer2 = self._make_layer(block, 128, layers[1], stride=2)
        self.layer3 = self._make_layer(block, 256, layers[2], stride=2)
        self.layer4 = self._make_layer(block, 512, layers[3], stride=2)
        self.deconv_layers = self._make_deconv_layer(extra.NUM_DECONV_LAYERS,
                                                     extra.NUM_DECONV_FILTERS,
                                                     extra.NUM_DECONV_KERNELS)
        out_ch = cfg.MODEL.NUM_JOINTS * cfg.MODEL.DEPTH_RES if self.volume else cfg.MODEL.NUM_JOINTS
        k = extra.FINAL_CONV_KERNEL
        self.final_layer = _Conv(extra.NUM_DECONV_FILTERS[-1], out_ch, k, 1, 1 if k == 3 else 0)
        if not self.volume:
            self.depth_fc = _Linear(2048, cfg.MODEL.NUM_JOINTS * cfg.MODEL.DEPTH_RES)
        kind = "bottleneck" if block.expansion == 4 else "basic"
        num_layers = [n for n, (kk, ll) in _net.RESNET_SPEC.items()
                      if kk == kind and list(ll) == list(layers)]
        if not num_layers:
            raise ValueError("unsupported layer spec %r" % (layers,))
        self._plan = _net.PoseNetPlan(
            num_layers=num_layers[0], num_joints=cfg.MODEL.NUM_JOINTS, volume=self.volume,
            depth_res=cfg.MODEL.DEPTH_RES, image_size=tuple(int(v) for v in cfg.MODEL.IMAGE_SIZE),
            deconv_filters=tuple(extra.NUM_DECONV_FILTERS),
            deconv_kernels=tuple(extra.NUM_DECONV_KERNELS),
            deconv_with_bias=extra.DECONV_WITH_BIAS, final_kernel=k)
        self._param_names = [n for n, _ in self.named_parameters()]
        self._eng = None
        self._ops = kwargs.get("ops")      # test hook (CPU emulation of the C ABI)

    # ---- containers (reference :128-183)
    def _make_layer(self, block, planes, blocks, stride=1):
        downsample = None
        if stride != 1 or self.inplanes != planes * block.expansion:
            downsample = nn.Sequential(
                _Conv(self.inplanes, planes * block.expansion, 1, stride, bias=False),
                _BN(planes * block.expansion, momentum=BN_MOMENTUM))
        mods = [block(self.inplanes, planes, stride, downsample)]
        self.inplanes = planes * block.expansion
        mods += [block(self.inplanes, planes) for _ in range(1, blocks)]
        return nn.Sequential(*mods)

    @staticmethod
    def _get_deconv_cfg(deconv_kernel, index=None):
        return {4: (4, 1, 0), 3: (3, 1, 1), 2: (2, 0, 0)}[deconv_kernel]

    def _make_deconv_layer(self, num_layers, num_filters, num_kernels):
        assert num_layers == len(num_filters), \
            'ERROR: num_deconv_layers is different len(num_deconv_filters)'
        assert num_layers == len(num_kernels), \
            'ERROR: num_deconv_layers is different len(num_deconv_filters)'
        mods = []
        for planes, kern in zip(num_filters, num_kernels):
            k, p, op = self._get_deconv_cfg(kern)
            mods += [_Deconv(self.inplanes, planes, k, 2, p, op, bias=self.deconv_with_bias),
                     _BN(planes, momentum=BN_MOMENTUM), _ReLU()]
            self.inplanes = planes
        return nn.Sequential(*mods)

    # ---- compute
    def _engine(self):
        if self._eng is None or self._eng_precision != self.precision:
            if self.precision in _SPLIT_PLANES and _net16.supported(self._plan):
                self._eng = _net16.Engine16(self._plan, ops=self._ops, planes=_SPLIT_PLANES[self.precision])
            else:
                self._eng = _net.Engine(self._plan, precision=_FALLBACK.get(self.precision, self.precision),
                                        ops=self._ops)
            self._eng_precision = self.precision
        return self._eng

    def forward(self, x):
        if self._ops is None and not x.is_cuda:
            raise RuntimeError("PoseResNet runs on sm_100a only (no CPU fallback); got a CPU tensor")
        if x.dtype != torch.float32:
            raise TypeError("expected float32 NCHW images")
        params = [p for _, p in self.named_parameters()]
        out = _PoseNetFn.apply(self, x.contiguous(), torch.is_grad_enabled(), *params)
        sink = getattr(self, "_last_sink", None)
        if sink is not None and isinstance(out, torch.Tensor) and sink.ptr == out.data_ptr():
            out._epb_logit_sink = sink        # read by the soft-argmax criterion (integral_loss.py)
        return out

    # ---- weights (reference :214-286)
    def init_weights(self, pretrained=''):
        if not os.path.isfile(pretrained):
            logger.error('=> imagenet pretrained model dose not exist')
            logger.error('=> please download it first')
            raise ValueError('imagenet pretrained model does not exist')
        for m in self.deconv_layers.modules():
            if isinstance(m, nn.ConvTranspose2d):
                nn.init.normal_(m.weight, std=0.001)
                if self.deconv_with_bias:
                    nn.init.constant_(m.bias, 0)
            elif isinstance(m, nn.BatchNorm2d):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0)
        nn.init.normal_(self.final_layer.weight, std=0.001)
        nn.init.constant_(self.final_layer.bias, 0)
        if 'mpii' in pretrained or 'coco' in pretrained:
            logger.info('=> loading pretrained pose model {}'.format(pretrained))
            self.load_pretrained_pose_model(pretrained)
        elif 'imagenet' in pretrained:
            logger.info('=> loading pretrained imagenet model {}'.format(pretrained))
            self.load_state_dict(torch.load(pretrained, map_location='cpu'), strict=False)

    def load_pretrained_pose_model(self, pretrained):
        loaded = torch.load(pretrained, map_location='cpu')
        if loaded and all('module' in k for k in loaded):       # DataParallel prefix
            loaded = OrderedDict((k[7:], v) for k, v in loaded.items())
        own = self.state_dict()
        keep = OrderedDict()
        for k, v in loaded.items():
            if k in own and own[k].shape != v.shape:
                logger.info('WARNING! There is a mismatch in => %s (%s, %s)' % (k, own[k].size(), v.size()))
                continue
            if k not in own:
                logger.info('%s not in model_dict' % k)
            keep[k] = v
        self.load_state_dict(keep, strict=False)


resnet_spec = {18: (BasicBlock, [2, 2, 2, 2]),
               34: (BasicBlock, [3, 4, 6, 3]),
               50: (Bottleneck, [3, 4, 6, 3]),
               101: (Bottleneck, [3, 4, 23, 3]),
               152: (Bottleneck, [3, 8, 36, 3])}


def get_pose_net(cfg, is_train, **kwargs):
    block_class, layers = resnet_spec[cfg.MODEL.EXTRA.NUM_LAYERS]
    model = PoseResNet(block_class, layers, cfg, **kwargs)
    if is_train and cfg.MODEL.INIT_WEIGHTS:
        model.init_weights(cfg.MODEL.PRETRAINED)
    return model
