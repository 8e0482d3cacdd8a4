"""GPU (-m gpu): the single-pass fp16 mode (MODEL.PRECISION: f16, include/epb.h "single-pass
layout": split tensors are their hi plane alone, [1][rows][C], one kind::f16 pass per k-step).

  * kernels: conv16 fprop / dgrad / accumulate / statistics and wgrad16 with planes=1 against a
    float64 torch convolution of the SAME operands (hi * 1/s), so the bar is the fp32
    accumulation noise of the tensor pipe (<= 5e-5 of the tensor's max), as in
    test_gpu_split16.py; layer shapes of the bench network (R50, 256x256 input, small batch);
  * producers: the hi plane a planes=1 call writes is bit-identical to the hi plane of the
    planes=2 call, and nothing is written past it (sentinel-filled buffers);
  * network: the C1 / C2 goldens, f16 against float64 with the single-pass TF32 engine's
    distance (same test, same inputs) as the yardstick -- both round operands to 10 explicit
    mantissa bits;
  * training: run-to-run determinism, CUDA-graph capture / replay, a falling loss."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import restate_net
from tests import emul_ops as em
from tests import golden_inputs as gi
from tests.conftest import relerr

pytestmark = pytest.mark.gpu

H16 = torch.float16
SENTINEL = 0x7E01          # an fp16 NaN no producer writes


@pytest.fixture(scope="module")
def dev():
    from epipolarpose_b200 import ops
    ops.device_check()
    return torch.device("cuda:0")


def _hi(v, s):
    """One-plane split tensor [1, ...] of v at scale s."""
    return (v * s).clamp(-65504, 65504).to(H16).unsqueeze(0)


def _pow2(v):
    return em._pow2_scale(float(v.abs().max()))


# ------------------------------------------------------------------ GEMM kernels
def _layer_cases():
    """(name, Conv, N, H, W): the conv shapes of the bench network (R50 at 256x256; batch 1-2)."""
    from epipolarpose_b200.net import Conv
    return [
        ("stem_col_192_64", Conv("a", "conv", 192, 64, 1, 1, 0), 1, 128, 128),
        ("l1_1x1_64_64", Conv("b", "conv", 64, 64, 1, 1, 0), 2, 64, 64),
        ("l1_3x3_64_64", Conv("c", "conv", 64, 64, 3, 1, 1), 2, 64, 64),
        ("l1_1x1_64_256", Conv("d", "conv", 64, 256, 1, 1, 0), 2, 64, 64),
        ("l2_1x1_256_128", Conv("e", "conv", 256, 128, 1, 1, 0), 2, 64, 64),
        ("l2_3x3_s2_128", Conv("f", "conv", 128, 128, 3, 2, 1), 2, 64, 64),
        ("l2_down_1x1_s2_256_512", Conv("g", "conv", 256, 512, 1, 2, 0), 2, 64, 64),
        ("l3_3x3_256", Conv("h", "conv", 256, 256, 3, 1, 1), 2, 16, 16),
        ("l4_3x3_512", Conv("i", "conv", 512, 512, 3, 1, 1), 2, 8, 8),
        ("l4_1x1_512_2048", Conv("j", "conv", 512, 2048, 1, 1, 0), 2, 8, 8),
        ("deconv1_2048_256", Conv("k", "deconv", 2048, 256, 4, 2, 1), 1, 8, 8),
        ("deconv3_256_256", Conv("l", "deconv", 256, 256, 4, 2, 1), 1, 32, 32),
        ("final_1x1_256_1024", Conv("m", "conv", 256, 1024, 1, 1, 0), 1, 32, 32),
    ]


CASES = _layer_cases()


def _sd_shape(conv):
    k = conv.k
    return (conv.cout, conv.cin, k, k) if conv.kind == "conv" else (conv.cin, conv.cout, k, k)


def _pack_hi(w_sd, conv, dgrad, s):
    """One-plane packed weight operand of the fprop (dgrad=False) or dgrad GEMM."""
    A, B = w_sd.shape[0], w_sd.shape[1]
    swap = (conv.kind == "conv") == dgrad       # epb.h epb_pack_weight table
    ypad = conv.cout_p if dgrad else conv.cin_p
    X = B if swap else A
    dst = torch.empty(X * conv.k * conv.k * ypad)
    em.pack_weight(w_sd, dst, A, B, conv.k, conv.k, int(swap), ypad)
    return _hi(dst, s).reshape(-1), (A, B, int(swap), ypad)


def _ref_fn(conv):
    if conv.kind == "conv":
        return lambda x, w: F.conv2d(x, w, stride=conv.stride, padding=conv.pad)
    return lambda x, w: F.conv_transpose2d(x, w, stride=conv.stride, padding=conv.pad,
                                           output_padding=conv.opad)


def _operands(conv, N, H, W):
    g = torch.Generator().manual_seed(100 + ord(conv.name))
    x = torch.relu(torch.randn((N, H, W, conv.cin), generator=g))
    sx = _pow2(x)
    x1 = _hi(x, sx)
    w = torch.randn(_sd_shape(conv), generator=g) * (2.0 / (conv.cin * conv.k * conv.k)) ** 0.5
    sw = _pow2(w)
    w_r = (w * sw).to(H16).float() / sw                 # the values the hi plane carries, exactly
    x_r = x1[0].double() / sx
    return x1, sx, w_r, sw, x_r


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_conv16_fprop_single_pass_vs_float64(dev, case):
    from epipolarpose_b200 import ops
    name, conv, N, H, W = case
    x1, sx, w_r, sw, x_r = _operands(conv, N, H, W)
    w1, _ = _pack_hi(w_r, conv, False, sw)
    ref = _ref_fn(conv)(x_r.permute(0, 3, 1, 2), w_r.double()).permute(0, 2, 3, 1)
    Ho, Wo = conv.out_hw(H, W)
    out = torch.zeros((N, Ho, Wo, conv.cout_p), device=dev)
    stats = torch.zeros(2 * conv.cout_p, dtype=torch.float64, device=dev)
    xs = torch.tensor([sx, 1.0 / sx], device=dev)
    wsc = torch.tensor([sw, 1.0 / sw], device=dev)
    xg, wg = x1.to(dev), w1.to(dev)
    for g in conv.fprop_geoms(ops, N, H, W, 1):
        if g is None:
            continue
        g.in_relu, g.accumulate = 0, 0
        ops.conv16_fprop(g, xg, xs, wg, wsc, out, None, stats, planes=1)
    torch.cuda.synchronize()
    e = relerr(out.cpu().numpy(), ref.numpy())
    r2 = ref.reshape(-1, conv.cout)
    st_ref = torch.cat([r2.sum(0), (r2 * r2).sum(0)])
    es = relerr(stats.cpu().numpy(), st_ref.numpy())
    print("%s: output %.2e, statistics %.2e" % (name, e, es))
    assert e <= 5e-5, "output relerr %.3e" % e
    assert es <= 1e-4, "statistics relerr %.3e" % es


@pytest.mark.parametrize("case", CASES[1:], ids=[c[0] for c in CASES[1:]])
@pytest.mark.parametrize("acc", [0, 1])
def test_conv16_dgrad_single_pass_vs_float64(dev, case, acc):
    from epipolarpose_b200 import ops
    name, conv, N, H, W = case
    _, _, w_r, sw, _ = _operands(conv, N, H, W)
    Ho, Wo = conv.out_hw(H, W)
    g = torch.Generator().manual_seed(11)
    dz = torch.randn((N, Ho, Wo, conv.cout), generator=g) * 3e-5
    sd = _pow2(dz)
    dz1 = _hi(dz, sd)
    wd1, _ = _pack_hi(w_r, conv, True, sw)
    x0 = torch.zeros((N, conv.cin, H, W), dtype=torch.float64, requires_grad=True)
    y = _ref_fn(conv)(x0, w_r.double())
    (dx_ref,) = torch.autograd.grad(y, x0, (dz1[0].double() / sd).permute(0, 3, 1, 2))
    dx_ref = dx_ref.permute(0, 2, 3, 1)
    init = torch.randn((N, H, W, conv.cin_p), generator=g) * float(dx_ref.abs().max()) if acc else \
        torch.zeros((N, H, W, conv.cin_p))
    din = init.to(dev)
    dzs = torch.tensor([sd, 1.0 / sd], device=dev)
    wsc = torch.tensor([sw, 1.0 / sw], device=dev)
    dzg, wg = dz1.to(dev), wd1.to(dev)
    for gm in conv.dgrad_geoms(ops, N, H, W, 1):
        if gm is None:
            continue
        gm.in_relu, gm.accumulate = 0, acc
        ops.conv16_fprop(gm, dzg, dzs, wg, wsc, din, None, None, planes=1)
    torch.cuda.synchronize()
    ref = dx_ref + init.double()
    e = relerr(din.cpu().numpy(), ref.numpy())
    print("%s acc=%d: %.2e" % (name, acc, e))
    assert e <= 5e-5, "dgrad relerr %.3e" % e


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_wgrad16_single_pass_vs_float64(dev, case):
    from epipolarpose_b200 import ops
    name, conv, N, H, W = case
    x1, sx, w_r, sw, x_r = _operands(conv, N, H, W)
    Ho, Wo = conv.out_hw(H, W)
    g = torch.Generator().manual_seed(12)
    dz = torch.randn((N, Ho, Wo, conv.cout), generator=g) * 3e-5
    sd = _pow2(dz)
    dz1 = _hi(dz, sd)
    w0 = w_r.double().requires_grad_(True)
    y = _ref_fn(conv)(x_r.permute(0, 3, 1, 2), w0)
    (dw_ref,) = torch.autograd.grad(y, w0, (dz1[0].double() / sd).permute(0, 3, 1, 2))
    _, (A, B, swap, ypad) = _pack_hi(w_r, conv, False, sw)
    X = B if swap else A
    dwp = torch.zeros(X * conv.k * conv.k * ypad, device=dev)
    ws = torch.empty(48 << 20, device=dev)
    xs = torch.tensor([sx, 1.0 / sx], device=dev)
    dzs = torch.tensor([sd, 1.0 / sd], device=dev)
    xg, dzg = x1.to(dev), dz1.to(dev)
    for gm in conv.fprop_geoms(ops, N, H, W, 1):
        if gm is None:
            continue
        gm.in_relu, gm.accumulate = 0, 0
        ops.conv16_wgrad(gm, xg, xs, dzg, dzs, dwp, ws, planes=1)
    torch.cuda.synchronize()
    dw = torch.empty(_sd_shape(conv))
    em.pack_weight(dwp.cpu(), dw, A, B, conv.k, conv.k, swap, ypad, unpack=1)
    e = relerr(dw.numpy(), dw_ref.numpy())
    print("%s: %.2e" % (name, e))
    assert e <= 5e-5, "wgrad relerr %.3e" % e


# ------------------------------------------------------------------ producers / readers
def _sentinel(n, dev):
    return torch.full((n,), SENTINEL, dtype=torch.int16, device=dev).view(H16)


def _check_one_plane(two, one, n):
    """hi plane identical, the would-be lo plane untouched"""
    two, one = two.reshape(-1).view(torch.int16), one.reshape(-1).view(torch.int16)
    assert torch.equal(one[:n], two[:n]), "hi planes differ"
    assert bool((one[n:] == SENTINEL).all()), "a planes=1 call wrote past the hi plane"


def test_producers_write_hi_plane_only(dev):
    from epipolarpose_b200 import ops
    g = torch.Generator().manual_seed(21)
    M, C = 4096, 256
    x = torch.randn((M, C), generator=g).to(dev)
    scale = (torch.rand(C, generator=g) + 0.5).to(dev)
    shift = torch.randn(C, generator=g).to(dev)
    r = torch.randn((M, C), generator=g).to(dev)
    sc = torch.tensor([1024.0, 1.0 / 1024, 0.0, 0.0], device=dev)
    n = M * C
    # bn_act_split: plain, fp32 residual with affine, mask bits
    for res in (None, r):
        a2, a1 = _sentinel(2 * n, dev), _sentinel(2 * n, dev)
        m2 = torch.empty(n // 8, dtype=torch.uint8, device=dev)
        m1 = torch.empty_like(m2)
        rs = (scale, shift) if res is not None else (None, None)
        ops.bn_act_split(x, scale, shift, res, *rs, None, None, 1, M, C, a2, sc, m2)
        ops.bn_act_split(x, scale, shift, res, *rs, None, None, 1, M, C, a1, sc, m1, planes=1)
        _check_one_plane(a2, a1, n)
        assert torch.equal(m1, m2)
    # bn_act_split with a one-plane split residual: y = relu(x*scale+shift + hi_r/s_r)
    r1 = _hi(r.cpu(), 1024.0).reshape(-1).to(dev)
    a1 = _sentinel(2 * n, dev)
    ops.bn_act_split(x, scale, shift, None, None, None, r1, sc, 1, M, C, a1, sc, planes=1)
    ref = torch.relu(x * scale + shift + r1.float().reshape(M, C) / 1024.0)
    assert relerr(a1[:n].view(M, C).float().cpu().numpy() / 1024.0, ref.cpu().numpy()) <= 1e-3
    assert bool((a1[n:].view(torch.int16) == SENTINEL).all())
    # stem: BatchNorm + ReLU + maxpool
    N, Hh, Ww, Cs = 2, 32, 32, 64
    z = torch.randn((N, Hh, Ww, Cs), generator=g).to(dev)
    np_ = N * 16 * 16 * Cs
    y2, y1 = _sentinel(2 * np_, dev), _sentinel(2 * np_, dev)
    ai2 = torch.empty(np_, dtype=torch.uint8, device=dev)
    ai1 = torch.empty_like(ai2)
    ops.bn_relu_maxpool_split(z, scale[:Cs], shift[:Cs], y2, sc, ai2, N, Hh, Ww, Cs)
    ops.bn_relu_maxpool_split(z, scale[:Cs], shift[:Cs], y1, sc, ai1, N, Hh, Ww, Cs, planes=1)
    _check_one_plane(y2, y1, np_)
    assert torch.equal(ai1, ai2)
    # patch matrix: the staged kernel (3 channels: the stem) and the per-element one (16 channels:
    # the input window no longer fits the staged kernel's shared memory)
    isc = torch.tensor([16.0, 1.0 / 16, 65504.0 / 16, 0.0], device=dev)
    for Ci, Hi, Kpad in ((3, 64, 192), (16, 32, 784)):
        img = torch.randn((1, Ci, Hi, Hi), generator=g).to(dev)
        Ho = (Hi + 6 - 7) // 2 + 1
        nc = Ho * Ho * Kpad
        c2, c1 = _sentinel(2 * nc, dev), _sentinel(2 * nc, dev)
        ops.im2col_split(img, c2, isc, 1, Ci, Hi, Hi, 7, 7, 2, 3, Ho, Ho, Kpad)
        ops.im2col_split(img, c1, isc, 1, Ci, Hi, Hi, 7, 7, 2, 3, Ho, Ho, Kpad, planes=1)
        _check_one_plane(c2, c1, nc)
    # fp32 -> split: one tensor, and a batch of two
    amax = torch.zeros(1, dtype=torch.int32, device=dev)
    s2, s1 = torch.empty(2, device=dev), torch.empty(2, device=dev)
    d2, d1 = _sentinel(2 * n, dev), _sentinel(2 * n, dev)
    ops.split16(x.reshape(-1), d2, s2, amax)
    ops.split16(x.reshape(-1), d1, s1, amax, planes=1)
    _check_one_plane(d2, d1, n)
    assert torch.equal(s1, s2)
    srcs = [x.reshape(-1)[:5000], r.reshape(-1)]
    outs = {}
    for planes in (2, 1):
        jobs = [(t, _sentinel(2 * t.numel(), dev), torch.empty(2, device=dev)) for t in srcs]
        batch = ops.SplitBatch([(t, d[:planes * t.numel()], sc_) for t, d, sc_ in jobs], planes=planes)
        ops.split16_batch(batch)
        outs[planes] = jobs
    for (t, d2_, sc2), (_, d1_, sc1) in zip(outs[2], outs[1]):
        _check_one_plane(d2_, d1_, t.numel())
        assert torch.equal(sc1, sc2)
    # BatchNorm backward apply pass; its mask_hi reader takes either layout
    mean, invstd = torch.randn(C, generator=g).to(dev), (torch.rand(C, generator=g) + 0.5).to(dev)
    gamma = torch.randn(C, generator=g).to(dev)
    dy = torch.randn((M, C), generator=g).to(dev)
    mask2 = _hi(torch.relu(r).cpu(), 1.0)[0]
    mask2 = torch.cat([mask2.reshape(-1), mask2.reshape(-1)]).to(dev)
    for mask_hi in (None, mask2):
        res = {}
        for planes, mh in ((2, mask_hi), (1, None if mask_hi is None else mask_hi[:n].clone())):
            dz = _sentinel(2 * n, dev)
            dsc = torch.empty(2, device=dev)
            dgm, dbt = torch.empty(C, device=dev), torch.empty(C, device=dev)
            kw = {} if planes == 2 else {"planes": 1}
            ops.bn_bwd_split(dy, x, mh, scale, shift, mean, invstd, gamma, 1, M, C, dz, dsc, None,
                             dgm, dbt, **kw)
            res[planes] = (dz, dsc, dgm, dbt)
        _check_one_plane(res[2][0], res[1][0], n)
        for a, b in zip(res[2][1:], res[1][1:]):
            assert torch.equal(a, b)


def test_softargmax_bwd_split_and_avgpool_one_plane(dev):
    from epipolarpose_b200 import ops
    g = torch.Generator().manual_seed(22)
    N, J, D, H, W = 2, 4, 16, 16, 16
    logits = torch.randn((N, H, W, J * D), generator=g).to(dev)
    coords = torch.empty(N * J * 3, device=dev)
    lse = torch.empty(N * J * 2, device=dev)
    ops.softargmax_fwd(logits, 1, N, J, D, H, W, coords, lse)
    dco = torch.randn(N * J * 3, generator=g).to(dev)
    n = N * H * W * J * D
    res = {}
    for planes in (2, 1):
        p = _sentinel(2 * n, dev)
        sc, db = torch.empty(2, device=dev), torch.empty(J * D, device=dev)
        kw = {} if planes == 2 else {"planes": 1}
        ops.softargmax_bwd_split(logits, N, J, D, H, W, coords, lse, dco, p, sc, db, **kw)
        res[planes] = (p, sc, db)
    _check_one_plane(res[2][0], res[1][0], n)
    assert torch.equal(res[1][1], res[2][1]) and torch.equal(res[1][2], res[2][2])
    # avgpool_split reads the hi plane alone
    Np, HW, C = 3, 64, 2048
    v = torch.relu(torch.randn((Np, HW, C), generator=g))
    x1 = _hi(v, 512.0)
    y = torch.empty((Np, C), device=dev)
    ops.avgpool_split(x1.to(dev), torch.tensor([512.0, 1.0 / 512], device=dev), y, Np, HW, C, planes=1)
    ref = (x1[0].double() / 512.0).mean(1)
    assert relerr(y.cpu().numpy(), ref.numpy()) <= 1e-6


# ------------------------------------------------------------------ network
def test_f16_selects_single_plane_engine(dev):
    from tests.test_gpu_sizes import _model
    c = gi.SIZE_CASES["c1"]
    model = _model(dev, c, "f16", train=False)
    eng = model._engine()
    assert type(eng).__name__ == "Engine16" and eng.planes == 1 and eng.precision == 1


def test_c1_eval_f16_vs_float64(golden, dev):
    from tests.test_gpu_sizes import _model
    c = gi.SIZE_CASES["c1"]
    g = golden("net_c1")
    mx = float(g["f64/out_max"])
    x = torch.from_numpy(gi.images(c["N"], c["HW"], c["seed"])).to(dev)
    err = {}
    for prec in ("tf32", "f16"):
        model = _model(dev, c, prec, train=False)
        with torch.no_grad():
            out = model(x)
        s = gi.sample_output(out.cpu().numpy())
        assert np.isfinite(s["out_sample"]).all()
        err[prec] = float(np.max(np.abs(s["out_sample"] - g["f64/out_sample"])) / mx)
        del model, out
    print("C1 heat-maps, distance from float64: f16 %.2e, tf32 %.2e" % (err["f16"], err["tf32"]))
    assert err["f16"] <= 2.0 * err["tf32"]


def test_c2_train_f16_vs_float64(golden, dev):
    from tests.test_gpu_sizes import _model
    c = gi.SIZE_CASES["c2"]
    g = golden("net_c2")
    x = torch.from_numpy(gi.images(c["N"], c["HW"], c["seed"])).to(dev)
    dist = {}
    for prec in ("tf32", "f16"):
        model = _model(dev, c, prec, train=True)
        out = model(x)
        s = gi.sample_output(out.detach().cpu().numpy())
        e_out = float(np.max(np.abs(s["out_sample"] - g["f64/out_sample"])) / float(g["f64/out_max"]))
        go = torch.from_numpy(gi.grad_like_big(out.shape, c["seed"] + 1)).to(dev)
        (out * go).sum().backward()
        rows = []
        for k, p in model.named_parameters():
            smp, tot = gi.sample_grad(p.grad.cpu().numpy())
            assert np.isfinite(tot).all() and np.isfinite(smp).all(), (prec, k)
            den = max(float(g["f64/gsum/" + k][2]), 1e-30)
            rows.append(float(np.max(np.abs(smp - g["f64/grad/" + k])) / den))
        assert len(rows) == 170
        dist[prec] = (e_out, np.median(rows), max(rows))
        del model, out
    print("C2, distance from float64 (heat-maps, gradient median, gradient max): f16 %.2e %.2e %.2e; "
          "tf32 %.2e %.2e %.2e" % (dist["f16"] + dist["tf32"]))
    f, t = dist["f16"], dist["tf32"]
    assert f[0] <= 2.0 * t[0]
    assert f[1] <= 2.0 * t[1]
    assert f[2] <= 2.0 * t[2]


# ------------------------------------------------------------------ training
def test_f16_backward_is_run_to_run_deterministic(dev):
    from tests.test_gpu_sizes import _model
    c = gi.SIZE_CASES["c2"]
    grads = []
    for rep in range(2):
        model = _model(dev, c, "f16", train=True)
        x = torch.from_numpy(gi.images(c["N"], c["HW"], c["seed"])).to(dev)
        out = model(x)
        go = torch.from_numpy(gi.grad_like_big(out.shape, c["seed"] + 1)).to(dev)
        (out * go).sum().backward()
        torch.cuda.synchronize()
        grads.append({k: p.grad.detach().clone() for k, p in model.named_parameters()})
        del model, out
    diff = [k for k in grads[0] if not torch.equal(grads[0][k], grads[1][k])]
    assert not diff, "%d tensors differ between two runs: %s" % (len(diff), diff[:5])


def _selfsup_model(dev, precision):
    import lib.models as models
    from oracle import refshim
    J, D, HW = 16, 64, 256
    cfg = refshim.make_cfg(num_layers=50, num_joints=J, volume=True, depth_res=D, image_size=(HW, HW))
    model = models.pose3d_resnet.get_pose_net(cfg, False, precision=precision)
    model.load_state_dict(restate_net.init_state(restate_net.param_shapes(50, J, True, D), 3,
                                                 scale_final=0.001))
    return model.to(dev).train(), J, D, HW


def test_f16_graphed_step_and_loss_falls(dev):
    """GraphedTrainStep captures and replays in f16 mode -- the online self-supervised step with
    the one-plane logit-gradient hand-over -- and 20 graphed Adam steps on a fixed batch with
    fixed labels lower the loss."""
    import lib.core.function as fn
    import lib.core.integral_loss as il
    import lib.utils.utils as U
    from tests.test_gpu_sizes import _ring_meta
    model, J, D, HW = _selfsup_model(dev, "f16")
    assert model._engine().planes == 1
    tuples = 2
    B = tuples * 4
    meta = {k: torch.from_numpy(v) for k, v in _ring_meta(tuples, 1073).items()}
    x = torch.from_numpy(gi.images(B, HW, 81)).to(dev)
    opt = U.FusedAdam(list(model.parameters()), lr=1e-3)
    online = fn.GraphedTrainStep(model, il.SmoothL1JointLocationLoss(J), opt, online=True,
                                 method="iterative")
    losses = [float(online(x, meta=meta)) for _ in range(4)]
    assert online.graph is not None
    assert all(np.isfinite(losses)), losses
    gt, wt = gi.labels(B, J, 82)
    label, weight = torch.from_numpy(gt).to(dev), torch.from_numpy(wt).to(dev)
    sup = fn.GraphedTrainStep(model, il.L1JointLocationLoss(J), opt)
    losses = [float(sup(x, label, weight)) for _ in range(20)]
    assert sup.graph is not None
    print("f16 graphed losses on a fixed batch:", " ".join("%.5f" % v for v in losses))
    assert all(np.isfinite(losses)), losses
    assert losses[-1] < 0.9 * losses[0], losses
    for k, p in model.named_parameters():
        assert torch.isfinite(p.detach()).all(), k
