"""PoseResNet forward / backward on the split-fp16 ("f16x3") tensor-core path.

Same network walk as net.Engine (reference lib/models/pose3d_resnet.py:91-212), different
data layout in HBM: every GEMM operand is materialised ONCE as two fp16 planes
(x * s = hi + lo, include/epb.h "split-fp16 operand family") by the kernel that produces it
-- the BatchNorm+ReLU(+residual) pass of each conv output, the BatchNorm-backward apply pass
of each gradient, the weight packer -- so that the conv kernels (csrc/conv16.cu,
csrc/wgrad16.cu) take both operands by TMA and run three kind::f16 tensor passes per k-step
at twice the TF32 rate, with fp32-grade results (a_lo*b_hi + a_hi*b_lo + a_hi*b_hi).

Kept per conv: the raw output z (fp32, for the BatchNorm backward) and the post-activation
split tensor (the next layer's operand).  Gradients w.r.t. activations stay fp32 (dgrad
epilogue output, accumulate target of the residual joins); gradients w.r.t. conv outputs
(dz) are split tensors with a per-tensor power-of-two scale derived on the device from the
BatchNorm-backward reductions; the fp32 logit gradient that enters the network's backward is
split once (amax + split).  Heads whose channel count is not a whole number of 64-channel blocks
(test-sized) keep their backward on the 3xTF32 kernels of net.Engine.

planes=1 is the single-pass "f16" mode: every split tensor is its hi plane alone (the TF32
operand class: 10 explicit mantissa bits, power-of-two scale as above), the GEMMs issue one
kind::f16 pass per k-step, no lo plane is ever written, and the fp32-operand layers run
single-pass TF32 instead of 3xTF32.
"""
import os

import torch

from . import net as _net
from .net import BN_EPS, BN_MOMENTUM, Conv, _BNState

IMG_SCALE = 16.0          # static scale of the (normalised) input image planes
STEM_KPAD16 = 192         # 7*7*3 = 147 padded to whole 64-element k-blocks
WGRAD_WS_FLOATS = 48 << 20


def supported(plan):
    """True when every layer of the plan fits the split path (channel counts that are whole
    64-element TMA boxes); otherwise the model keeps the 3xTF32 engine."""
    convs = [c for c in plan.all_convs() if c is not plan.stem and c is not plan.final
             and c is not plan.fc]
    ok = all(c.cin % 64 == 0 and c.cout % 64 == 0 for c in convs)
    ok = ok and plan.final.cin % 64 == 0
    ok = ok and not any(c.bias for c, _ in plan.deconvs)
    return ok


class Engine16(_net.Engine):

    def __init__(self, plan, ops=None, planes=2):
        if planes not in (1, 2):
            raise ValueError("planes must be 1 (f16) or 2 (f16x3), got %r" % (planes,))
        # the few fp32-operand layers: 3xTF32 beside three f16 passes, TF32 beside one
        prec = 3 if planes == 2 else 1
        super().__init__(plan, precision=prec, ops=ops)
        self.tc_precision = prec
        self.planes = planes
        # plane count for the split-family calls; the two-plane calls pass none (the default)
        self._pk = {} if planes == 2 else {"planes": planes}
        # the fp32 packed weights are only read by the amax / split passes and the packed weight gradients
        # only written by plain stores: 1x1 layers use the parameter / gradient tensors themselves
        self.alias_1x1 = True
        self.stem_kpad = STEM_KPAD16
        self.stem_col = Conv("conv1", "conv", STEM_KPAD16, 64, 1, 1, 0)

    # geometry tables are shared with the fp32-operand kernels: their precision field is theirs
    def _geoms(self, conv, kind, N, H, W):
        f = conv.fprop_geoms if kind == "f" else conv.dgrad_geoms
        return f(self.ops, N, H, W, self.tc_precision)

    # ------------------------------------------------------------------ persistent state
    def _half(self, *shape):
        return torch.empty((self.planes,) + tuple(shape), device=self.dev, dtype=torch.float16)

    def _consts(self):
        st = getattr(self, "_cst", None)
        if st is None or st["dev"] != self.dev:
            st = {"dev": self.dev,
                  # the image patch matrix keeps a static scale: |pixel| <= 4094 representable
                  "img_sc": torch.tensor([IMG_SCALE, 1.0 / IMG_SCALE, 65504.0 / IMG_SCALE, 0.0],
                                         device=self.dev, dtype=torch.float32),
                  "ws": torch.empty(WGRAD_WS_FLOATS, device=self.dev, dtype=torch.float32),
                  "amax1": torch.zeros(1, device=self.dev, dtype=torch.int32)}
            self._cst = st
        return st

    def _split_weights(self, packed):
        """fp32 packed operands -> split operands {name: ((wf16, sc), (wd16, sc) | None)},
        all layers in ONE batched conversion (amax + split)."""
        ops, plan = self.ops, self.plan
        key = tuple(t.data_ptr() for pair in packed.values() for t in pair if t is not None)
        st = getattr(self, "_w16", None)
        if st is None or st["key"] != key:
            out, jobs = {}, []
            for name, pair in packed.items():
                ent = []
                for t in pair:
                    if t is None:
                        ent.append(None)
                        continue
                    h = torch.empty(self.planes * t.numel(), device=self.dev, dtype=torch.float16)
                    sc = torch.ones(2, device=self.dev, dtype=torch.float32)
                    jobs.append((t, h, sc))
                    ent.append((h, sc))
                out[name] = tuple(ent)
            st = {"key": key, "w": out, "batch": ops.SplitBatch(jobs, **self._pk)}
            self._w16 = st
        ops.split16_batch(st["batch"])
        return st["w"]

    # ------------------------------------------------------------------ conv helpers
    def _conv_fwd16(self, conv, x, x_sc, N, H, W, w16, bias=None, stats=None):
        ops = self.ops
        Ho, Wo = conv.out_hw(H, W)
        geoms = self._geoms(conv, "f", N, H, W)
        need_zero = any(g is None for g in geoms)
        out = (torch.zeros if need_zero else torch.empty)(
            (N, Ho, Wo, conv.cout_p), device=self.dev, dtype=torch.float32)
        for g in geoms:
            if g is None:
                continue
            g.in_relu, g.accumulate = 0, 0
            ops.conv16_fprop(g, x, x_sc, w16[0], w16[1], out, bias, stats, **self._pk)
        return out, Ho, Wo

    def _conv_dgrad16(self, conv, dz, dz_sc, N, H, W, wd16, accumulate_into=None):
        ops = self.ops
        geoms = self._geoms(conv, "d", N, H, W)
        if accumulate_into is not None:
            din = accumulate_into
        else:
            need_zero = any(g is None for g in geoms)
            din = (torch.zeros if need_zero else torch.empty)(
                (N, H, W, conv.cin_p), device=self.dev, dtype=torch.float32)
        for g in geoms:
            if g is None:
                continue
            g.in_relu = 0
            g.accumulate = 1 if accumulate_into is not None else 0
            ops.conv16_fprop(g, dz, dz_sc, wd16[0], wd16[1], din, None, None, **self._pk)
        return din

    def _conv_wgrad16(self, conv, x, x_sc, dz, dz_sc, N, H, W):
        """Weight gradient into the step's flat packed accumulator; on the side stream
        (nothing downstream consumes it before the optimiser)."""
        ops = self.ops
        dwp = self._gs["dwp"][conv.name]
        ws = self._consts()["ws"]

        def run():
            for g in self._geoms(conv, "f", N, H, W):
                if g is None:
                    continue
                g.in_relu, g.accumulate = 0, 0
                ops.conv16_wgrad(g, x, x_sc, dz, dz_sc, dwp, ws, **self._pk)

        side = getattr(self, "_side", None)
        if side is None:
            run()
            return
        main = torch.cuda.current_stream()
        side.wait_stream(main)
        self._keep.append((x, dz, dz_sc))
        with torch.cuda.stream(side):
            run()

    def _bn_bwd16(self, st, dy, z, mask_bits, relu, params, grads, dy_masked=None):
        """BatchNorm(+ReLU) backward -> (dz split, dz_sc).  Fills grads[name.weight/.bias].
        mask_bits: the block output's ReLU bit mask (bn_act_split), or None (mask from z)."""
        ops = self.ops
        C = st.C
        M = z.numel() // C
        dz = self._half(*z.shape)
        dz_sc = torch.empty(2, device=self.dev, dtype=torch.float32)
        ops.bn_bwd_split(dy, z, None, st.scale, st.shift, st.mean, st.invstd,
                         params[st.name + ".weight"], relu, M, C, dz, dz_sc, dy_masked,
                         grads[st.name + ".weight"], grads[st.name + ".bias"], mask_bits=mask_bits,
                         **self._pk)
        return dz, dz_sc

    # ------------------------------------------------------------------ forward
    def forward(self, x_nchw, params, training=True, save=True):
        ops, plan = self.ops, self.plan
        self.dev = x_nchw.device
        N, _, H, W = x_nchw.shape
        cst = self._consts()
        S = {"N": N, "H": H, "W": W, "bn": {}, "blocks": []}
        bns = plan.all_bns()
        offs, tot = {}, 0
        for name, C in bns:
            offs[name] = tot
            tot += 2 * C
        # batch statistics of every conv output: BatchNorm in train(), and in both modes the
        # bound that fixes the scale of the post-activation split tensor (epb_act_scale)
        stats_all = torch.zeros(tot, device=self.dev, dtype=torch.float64)
        scs = torch.empty((len(bns) + 1, 4), device=self.dev, dtype=torch.float32)
        sc_slot = [0]

        def new_sc():
            sc_slot[0] += 1
            return scs[sc_slot[0] - 1]

        def stats_of(name, C):
            return stats_all[offs[name]:offs[name] + 2 * C]

        def bn(name, C, M, sc=None, group2=(None, None, None), res_sc=None):
            """BatchNorm state of conv output `name`; with sc also the scale of its post-activation
            split tensor (train(): the same launch)."""
            if training:
                fused = None if sc is None else group2 + (res_sc, sc)
                st = self._bn_train(name, C, stats_of(name, C), M, params, None, act_scale=fused)
            else:
                st = self._bn_eval(name, C, params)
                if sc is not None:
                    ops.act_scale(stats_of(name, C), st.scale, st.shift, M, C, *group2, res_sc, sc)
            S["bn"][name] = st
            return st

        self._nbt_tick = []

        S["packed"] = self._pack_weights(params)
        S["w16"] = self._split_weights(S["packed"])

        def w16(conv):
            return S["w16"][conv.name][0]

        def bn_act(z, name, shape):
            """BatchNorm state of conv output z, its post-BatchNorm/ReLU split tensor and scale"""
            C = shape[-1]
            M = z.numel() // C
            sc = new_sc()
            st = bn(name, C, M, sc)
            a = self._half(*shape)
            ops.bn_act_split(z, st.scale, st.shift, None, None, None, None, None, 1, M, C, a, sc, **self._pk)
            return st, a, sc

        # ---- stem (pose3d_resnet.py:186-189): patch matrix -> 1x1 GEMM -> BN+ReLU+maxpool
        stem, scol, kpad = plan.stem, self.stem_col, self.stem_kpad
        H1, W1 = stem.out_hw(H, W)
        col = self._half(N, H1, W1, kpad)
        isc = cst["img_sc"]
        ops.im2col_split(x_nchw, col, isc, N, 3, H, W, 7, 7, 2, 3, H1, W1, kpad, **self._pk)
        z0, _, _ = self._conv_fwd16(scol, col, isc, N, H1, W1, w16(stem), stats=stats_of("bn1", 64))
        cur_sc = new_sc()
        b0 = bn("bn1", 64, N * H1 * W1, cur_sc)
        H2, W2 = (H1 + 2 - 3) // 2 + 1, (W1 + 2 - 3) // 2 + 1
        cur = self._half(N, H2, W2, 64)
        argidx = torch.empty((N, H2, W2, 64), device=self.dev, dtype=torch.uint8)
        ops.bn_relu_maxpool_split(z0, b0.scale, b0.shift, cur, cur_sc, argidx, N, H1, W1, 64, **self._pk)
        S["stem"] = (col, z0, argidx, H1, W1, H2, W2)
        h, w = H2, W2

        # ---- residual stages (:191-194)
        for blk in plan.blocks:
            rec = {"in": (cur, cur_sc), "h": h, "w": w, "z": [], "hw": [], "a": []}
            src, src_sc = cur, cur_sc
            hh, ww = h, w
            nconv = len(blk["convs"])
            for ci, conv in enumerate(blk["convs"]):
                bname, C = blk["bns"][ci]
                z, ho, wo = self._conv_fwd16(conv, src, src_sc, N, hh, ww, w16(conv),
                                             stats=stats_of(bname, C))
                rec["z"].append(z)
                rec["hw"].append((hh, ww))
                hh, ww = ho, wo
                if ci < nconv - 1:
                    _, src, src_sc = bn_act(z, bname, (N, hh, ww, conv.cout_p))
                    rec["a"].append((src, src_sc))
            lname = blk["bns"][-1][0]
            zl = rec["z"][-1]
            Cl = blk["convs"][-1].cout_p
            M = N * hh * ww
            out = self._half(N, hh, ww, Cl)
            out_sc = new_sc()
            # ReLU mask of the block output, one bit per element (read twice by the backward)
            obits = torch.empty(M * Cl // 8, device=self.dev, dtype=torch.uint8) if save else None
            if blk["down"]:
                dconv, (dname, dC) = blk["down"]
                zd, _, _ = self._conv_fwd16(dconv, cur, cur_sc, N, h, w, w16(dconv),
                                            stats=stats_of(dname, dC))
                dst = bn(dname, dC, M)
                rec["zd"] = zd
                last = bn(lname, Cl, M, out_sc, (stats_of(dname, dC), dst.scale, dst.shift))
                ops.bn_act_split(zl, last.scale, last.shift, zd, dst.scale, dst.shift, None, None,
                                 1, M, Cl, out, out_sc, obits, **self._pk)
            else:
                last = bn(lname, Cl, M, out_sc, res_sc=cur_sc)
                ops.bn_act_split(zl, last.scale, last.shift, None, None, None, cur, cur_sc, 1, M, Cl,
                                 out, out_sc, obits, **self._pk)
            rec["out"] = (out, out_sc)
            rec["mask"] = obits
            S["blocks"].append(rec)
            cur, cur_sc, h, w = out, out_sc, hh, ww

        S["trunk"] = (cur, cur_sc, h, w)
        # ---- deconv head (:198)
        src, src_sc = cur, cur_sc
        S["deconv"] = []
        zlast, stlast = None, None
        for conv, (bname, C) in plan.deconvs:
            z, ho, wo = self._conv_fwd16(conv, src, src_sc, N, h, w, w16(conv), stats=stats_of(bname, C))
            S["deconv"].append((src, src_sc, z, h, w))
            st, src, src_sc = bn_act(z, bname, (N, ho, wo, conv.cout_p))
            h, w = ho, wo
            zlast, stlast = z, st
        if zlast is None:
            raise RuntimeError("the split path expects at least one deconv layer")
        # ---- final 1x1 / 3x3 conv with bias (:199)
        fin = plan.final
        fbias = params[fin.name + ".bias"]
        if fin.cout_p != fin.cout:
            fb = torch.zeros(fin.cout_p, device=self.dev)
            fb[:fin.cout] = fbias
            fbias = fb
        logits, ho, wo = self._conv_fwd16(fin, src, src_sc, N, h, w, w16(fin), bias=fbias)
        # the final layer's backward: split operands when the head has whole 64-channel blocks,
        # else the fp32-operand kernels from (z, BatchNorm affine)
        S["final"] = (zlast, (stlast.scale, stlast.shift), h, w)
        S["final16"] = (src, src_sc)
        depth = None
        if plan.fc is not None:                 # :202-210
            tr, tr_sc, th, tw = S["trunk"]
            assert th == plan.pool_k and tw == plan.pool_k, "AvgPool(k) -> 1x1 expected"
            pooled = torch.empty((N, 1, 1, 2048), device=self.dev, dtype=torch.float32)
            ops.avgpool_split(tr, tr_sc, pooled, N, th * tw, 2048, **self._pk)
            depth, _, _ = self._conv_fwd(plan.fc, pooled, N, 1, 1, S["packed"][plan.fc.name][0],
                                         bias=params["depth_fc.bias"])
            S["fc"] = pooled
        tick, self._nbt_tick = self._nbt_tick, None
        if tick:
            torch._foreach_add_(tick, 1)        # num_batches_tracked of every BatchNorm: one launch
        return logits, depth, (S if save else None)

    # ------------------------------------------------------------------ backward
    def backward(self, S, dlogits, ddepth, params, grads, on_stage=None, head=None):
        """head: a filled _sinks.LogitGradSink (the criterion wrote the logit gradient as split planes
        + bias gradient) instead of the fp32 dlogits."""
        self._head = head
        try:
            super().backward(S, dlogits, ddepth, params, grads, on_stage=on_stage)
        finally:
            self._head = None

    def takes_logit_sink(self):
        fin = self.plan.final
        return self.plan.fc is None and fin.cout_p == fin.cout and fin.cout_p % 64 == 0

    def _backward(self, S, dlogits, ddepth, params, grads):
        ops, plan = self.ops, self.plan
        N = S["N"]

        def wd16(conv):
            return S["w16"][conv.name][1]

        # ---- final layer
        fin = plan.final
        src, aff, h, w = S["final"]
        Ho, Wo = fin.out_hw(h, w)
        gb = grads[fin.name + ".bias"]
        head = getattr(self, "_head", None)
        if head is not None:
            gb.copy_(head.dbias)                # column sums from the soft-argmax backward itself
        elif fin.cout_p != fin.cout:
            tmp = torch.empty(fin.cout_p, device=self.dev)
            ops.colsum(dlogits, N * Ho * Wo, fin.cout_p, tmp)
            gb.copy_(tmp[:fin.cout])
        else:
            ops.colsum(dlogits, N * Ho * Wo, fin.cout_p, gb)
        if fin.cout_p % 64 == 0:
            if head is not None:
                dl16, dl_sc = head.planes, head.sc
            else:
                # the fp32 logit gradient becomes a split operand (amax + split): data and weight
                # gradient on the split kernels like every other layer (deterministic)
                dl16 = self._half(N, Ho, Wo, fin.cout_p)
                dl_sc = torch.empty(2, device=self.dev, dtype=torch.float32)
                ops.split16(dlogits.reshape(-1), dl16.reshape(-1), dl_sc, self._consts()["amax1"], **self._pk)
            fsrc, fsrc_sc = S["final16"]
            self._conv_wgrad16(fin, fsrc, fsrc_sc, dl16, dl_sc, N, h, w)
            dcur = self._conv_dgrad16(fin, dl16, dl_sc, N, h, w, wd16(fin))
        else:
            # few output channels (test-sized heads): the fp32-operand kernels take the fp32 gradient
            self._conv_wgrad(fin, src, dlogits, N, h, w, grads[fin.name + ".weight"], affine=aff)
            dcur = self._conv_dgrad(fin, dlogits, N, h, w, S["packed"][fin.name][1])
        # ---- deconv head, reversed
        for (conv, (bname, C)), (dsrc, dsrc_sc, z, dh, dw) in zip(reversed(plan.deconvs),
                                                                  reversed(S["deconv"])):
            st = S["bn"][bname]
            dz, dsc = self._bn_bwd16(st, dcur, z, None, 1, params, grads)
            self._conv_wgrad16(conv, dsrc, dsrc_sc, dz, dsc, N, dh, dw)
            dcur = self._conv_dgrad16(conv, dz, dsc, N, dh, dw, wd16(conv))
        # ---- VOLUME=False depth head (fp32 operands)
        if plan.fc is not None and ddepth is not None:
            tr, tr_sc, th, tw = S["trunk"]
            dd = ddepth.reshape(N, 1, 1, -1).contiguous()
            ops.colsum(dd, N, plan.fc.cout_p, grads["depth_fc.bias"])
            self._conv_wgrad(plan.fc, S["fc"], dd, N, 1, 1, grads["depth_fc.weight"])
            dpool = self._conv_dgrad(plan.fc, dd, N, 1, 1, S["packed"][plan.fc.name][1])
            ops.avgpool_bwd(dpool, dcur, N, th * tw, 2048, 1)
        self._stage_done(0)                     # head (deconvs, final layer, depth_fc) complete
        # ---- residual stages, reversed
        prev_stage = None
        for blk, rec in zip(reversed(plan.blocks), reversed(S["blocks"])):
            sk = _net.stage_of(blk["name"])
            if prev_stage is not None and sk != prev_stage:
                self._stage_done(prev_stage)
            prev_stage = sk
            (out, _), (xin, xin_sc), h, w = rec["out"], rec["in"], rec["h"], rec["w"]
            nconv = len(blk["convs"])
            mask = rec["mask"]                  # ReLU bit mask of the block output
            down = blk["down"]
            if down:
                dconv, (dname, dC) = down
                dzd, dzd_sc = self._bn_bwd16(S["bn"][dname], dcur, rec["zd"], mask, 0, params, grads)
            g = dcur
            for ci in range(nconv - 1, -1, -1):
                conv = blk["convs"][ci]
                st = S["bn"][blk["bns"][ci][0]]
                z = rec["z"][ci]
                if ci == nconv - 1:
                    # identity blocks: the masked gradient also replaces dcur in place; conv1's
                    # data gradient then accumulates into it (the residual join, no extra pass)
                    dz, dsc = self._bn_bwd16(st, dcur, z, mask, 0, params, grads,
                                             dy_masked=None if down else dcur)
                else:
                    dz, dsc = self._bn_bwd16(st, g, z, None, 1, params, grads)
                hh, ww = rec["hw"][ci]
                xop, xop_sc = (xin, xin_sc) if ci == 0 else rec["a"][ci - 1]
                self._conv_wgrad16(conv, xop, xop_sc, dz, dsc, N, hh, ww)
                if ci == 0 and not down:
                    g = self._conv_dgrad16(conv, dz, dsc, N, hh, ww, wd16(conv), accumulate_into=dcur)
                else:
                    g = self._conv_dgrad16(conv, dz, dsc, N, hh, ww, wd16(conv))
            if down:
                self._conv_wgrad16(dconv, xin, xin_sc, dzd, dzd_sc, N, h, w)
                self._conv_dgrad16(dconv, dzd, dzd_sc, N, h, w, wd16(dconv), accumulate_into=g)
            dcur = g
        # ---- stem
        col, z0, argidx, H1, W1, H2, W2 = S["stem"]
        gpool = torch.empty((N, H1, W1, 64), device=self.dev, dtype=torch.float32)
        ops.maxpool_bwd(dcur, argidx, gpool, N, H1, W1, 64)
        dz0, dsc0 = self._bn_bwd16(S["bn"]["bn1"], gpool, z0, None, 1, params, grads)
        self._conv_wgrad16(self.stem_col, col, self._consts()["img_sc"], dz0, dsc0, N, H1, W1)
