"""CPU: host-side logic (network plan, geometry / tap tables, weight packing,
autograd wiring, optimiser, config, dataset, loops) through the torch-CPU
emulation of the C ABI (tests/emul_ops.py), and the C-ABI library itself
(loads; exports every symbol include/epb.h declares; refuses to compute
without a GPU)."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import refshim, restate, restate_net
from tests import emul_ops, golden_inputs as gi
from tests.conftest import ROOT, relerr


def test_c_abi_exports_match_header():
    from epipolarpose_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "epb.h")).read()
    declared = set(re.findall(r"\b(epb_[a-z0-9_]+)\s*\(", hdr)) - {"epb_conv_geom"}
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    L = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(L, name), name
    assert _lib.lib().epb_version() >= 100


def test_product_path_fails_loudly_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from epipolarpose_b200 import _lib, ops
    with pytest.raises(_lib.EpbError):
        ops.device_check()
    import lib.models as models
    cfg = refshim.make_cfg(num_layers=18, num_joints=2, depth_res=4, image_size=(32, 32))
    m = models.pose3d_resnet.get_pose_net(cfg, False)
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 3, 32, 32))            # no CPU fallback
    import lib.core.integral_loss as il
    with pytest.raises(_lib.EpbError):
        il.softmax_integral_tensor(torch.zeros(1, 8, 4, 4), 2, True, 4, 4, 4)


def test_config_parses_reference_yamls(tmp_path):
    from lib.core.config import config, update_config, reset_config, get_model_name, gen_config
    y = tmp_path / "exp.yaml"
    y.write_text("GPUS: '0'\nMODEL:\n  NUM_JOINTS: 16\n  VOLUME: true\n  EXTRA:\n    NUM_LAYERS: 50\n"
                 "LOSS:\n  FN: SmoothL1JointLocationLoss\nTRAIN:\n  LR_STEP:\n  - 90\n  - 120\n")
    reset_config()
    update_config(str(y))
    assert config.MODEL.NUM_JOINTS == 16 and config.TRAIN.LR_STEP == [90, 120]
    assert get_model_name(config)[0] == "pose3d_resnet_50"
    bad = tmp_path / "bad.yaml"
    bad.write_text("MODEL:\n  NOT_A_KEY: 1\n")
    with pytest.raises(ValueError):
        update_config(str(bad))
    bad.write_text("NOPE: 1\n")
    with pytest.raises(ValueError):
        update_config(str(bad))
    gen_config(str(tmp_path / "dump.yaml"))
    reset_config()


@pytest.mark.parametrize("layers,volume", [(18, True), (34, True), (50, False)])
def test_engine_matches_oracle_through_emulated_abi(layers, volume):
    """Whole-network forward + backward wiring (geometry tables, phase
    decomposition of stride-2 dgrad / deconv, packing, BN, residual merges)."""
    import lib.models as models
    J, D, HW, N = 3, 8, 64, 2
    cfg = refshim.make_cfg(num_layers=layers, num_joints=J, volume=volume, depth_res=D,
                           image_size=(HW, HW))
    shapes = restate_net.param_shapes(layers, J, volume, D)
    sd = restate_net.init_state(shapes, 9)
    m = models.pose3d_resnet.get_pose_net(cfg, False, ops=emul_ops)
    assert list(m.state_dict().keys()) == list(shapes.keys())
    m.load_state_dict(sd)
    m.train()
    x = torch.from_numpy(gi.images(N, HW, 9))
    p = {k: (v.double().clone().requires_grad_(True) if v.is_floating_point() and "running" not in k
             else (v.double() if v.is_floating_point() else v)) for k, v in sd.items()}
    ref = restate_net.forward(p, x.double(), num_layers=layers, volume=volume, image_size=(HW, HW))
    out = m(x)
    refs = ref if isinstance(ref, tuple) else (ref,)
    outs = out if isinstance(out, tuple) else (out,)
    gs = [torch.from_numpy(gi.grad_like(o.shape, 10 + i)) for i, o in enumerate(outs)]
    for o, r in zip(outs, refs):
        assert relerr(o.detach().numpy(), r.detach().numpy()) <= 2e-3
    sum((o * g).sum() for o, g in zip(outs, gs)).backward()
    sum((r * g.double()).sum() for r, g in zip(refs, gs)).backward()
    if layers != 50:      # R50 at 64x64 / batch 2 is chaotic in fp32 (2x2x2 BN statistics)
        for k, q in m.named_parameters():
            assert relerr(q.grad.numpy(), p[k].grad.numpy()) <= 5e-3, k
    assert int(m.state_dict()["bn1.num_batches_tracked"]) == 1


@pytest.mark.parametrize("dk,fk,db", [((3, 2, 4), 3, True), ((2, 3, 4), 1, False)])
def test_engine_uncommon_head_configs_emulated(dk, fk, db):
    """cfg.MODEL.EXTRA variants the bench never uses (reference pose3d_resnet.py:145-156,116-122):
    deconv kernels 3 -> (pad 1, output_padding 1) and 2 -> (0, 0), FINAL_CONV_KERNEL = 3,
    DECONV_WITH_BIAS -- geometry tables, packing and gradients through the emulated ABI."""
    import lib.models as models
    J, D, HW, N = 3, 8, 64, 2
    cfg = refshim.make_cfg(num_layers=18, num_joints=J, volume=True, depth_res=D, image_size=(HW, HW),
                           deconv_with_bias=db, final_kernel=fk)
    cfg.MODEL.EXTRA.NUM_DECONV_KERNELS = list(dk)
    shapes = restate_net.param_shapes(18, J, True, D, deconv_kernels=dk, deconv_with_bias=db, final_kernel=fk)
    sd = restate_net.init_state(shapes, 9)
    m = models.pose3d_resnet.get_pose_net(cfg, False, ops=emul_ops)
    assert list(m.state_dict().keys()) == list(shapes.keys())
    m.load_state_dict(sd)
    m.train()
    x = torch.from_numpy(gi.images(N, HW, 9))
    p = {k: (v.double().clone().requires_grad_(True) if v.is_floating_point() and "running" not in k
             else (v.double() if v.is_floating_point() else v)) for k, v in sd.items()}
    ref = restate_net.forward(p, x.double(), num_layers=18, volume=True, image_size=(HW, HW),
                              deconv_kernels=dk, final_kernel=fk)
    out = m(x)
    assert out.shape == ref.shape and relerr(out.detach().numpy(), ref.detach().numpy()) <= 1e-4
    g = torch.from_numpy(gi.grad_like(out.shape, 10))
    (out * g).sum().backward()
    (ref * g.double()).sum().backward()
    gmax = max(float(p[k].grad.abs().max()) for k, _ in m.named_parameters())
    for k, q in m.named_parameters():
        r = p[k].grad.numpy()
        # a bias in front of a training-mode BatchNorm has an exactly-zero gradient: absolute check
        assert np.max(np.abs(q.grad.numpy() - r)) <= 5e-3 * max(np.max(np.abs(r)), 1e-4 * gmax), k


@pytest.mark.parametrize("layers", [18, 34, 50, 101, 152])
def test_state_dict_surface_all_depths(layers):
    """get_pose_net for every entry of resnet_spec (reference pose3d_resnet.py:288-292): state_dict
    keys, order and shapes equal the oracle's table (pinned to the reference module for 18 / 50),
    VOLUME on and off; parameter counts of SURVEY section 8 (R50 34.27 M, R101 53.27 M)."""
    import lib.models as models
    for volume in (True, False):
        cfg = refshim.make_cfg(num_layers=layers, num_joints=17, volume=volume, depth_res=64, image_size=(256, 256))
        m = models.pose3d_resnet.get_pose_net(cfg, False, ops=emul_ops)
        shapes = restate_net.param_shapes(layers, 17, volume, 64)
        sd = m.state_dict()
        assert list(sd.keys()) == list(shapes.keys())
        assert all(tuple(sd[k].shape) == tuple(shapes[k]) for k in shapes)
    if layers in (50, 101):
        cfg = refshim.make_cfg(num_layers=layers, num_joints=17, volume=True, depth_res=64, image_size=(256, 256))
        n = sum(p.numel() for p in models.pose3d_resnet.get_pose_net(cfg, False, ops=emul_ops).parameters())
        assert abs(n / 1e6 - {50: 34.27, 101: 53.27}[layers]) < 0.01


def test_losses_and_decode_surface_emulated():
    import lib.core.integral_loss as il
    import lib.core.inference as inf
    il._backend[0] = emul_ops
    inf._backend[0] = emul_ops
    try:
        N, J, D = 2, 3, 8
        x = torch.from_numpy(gi.logits(N, J, D, D, D, 4, 2.0)).requires_grad_(True)
        gt, wt = gi.labels(N, J, 4)
        for cls, kind in ((il.L1JointLocationLoss, "l1"), (il.SmoothL1JointLocationLoss, "smoothl1"),
                          (il.L2JointLocationLoss, "mse")):
            for norm in (False, True):
                x.grad = None
                loss = cls(J, norm=norm)(x, torch.from_numpy(gt), torch.from_numpy(wt))
                loss.backward()
                c = restate.softmax_integral(x.detach().numpy(), J, D, D, D)
                rl, dc = restate.weighted_loss(kind, c, gt, wt, True, norm)
                assert abs(loss.item() - rl) <= 1e-5
                rg = restate.softmax_integral_grad(x.detach().numpy(), dc, J, D, D, D)
                assert relerr(x.grad.numpy(), rg) <= 1e-3
        with pytest.raises(AssertionError):
            il.L1JointLocationLoss(J)(x, torch.from_numpy(gt).requires_grad_(True), torch.from_numpy(wt))
        hm = gi.argmax_heatmaps()
        p, mv = inf.get_max_preds(hm)
        rp, rm, _ = restate.get_max_preds(hm)
        assert np.array_equal(p, rp) and np.array_equal(mv, rm)
        with pytest.raises(AssertionError):
            inf.get_max_preds(hm[0])
        # get_final_preds through the reference-shaped numpy API (emulated epb_final_preds)
        import types
        g = dict(np.load(os.path.join(ROOT, "tests", "golden", "final_preds.npz")))
        fh, fc, fs = gi.final_preds_case()
        for pp in (1, 0):
            cfg = types.SimpleNamespace(TEST=types.SimpleNamespace(POST_PROCESS=bool(pp)))
            fp, fm = inf.get_final_preds(cfg, fh.copy(), fc, fs)
            assert np.array_equal(fp, g["preds_pp%d" % pp]) and np.array_equal(fm, g["maxvals_pp%d" % pp])
    finally:
        il._backend[0] = __import__("epipolarpose_b200.ops", fromlist=["ops"])
        inf._backend[0] = il._backend[0]


def test_heatmap_joint_loss_oracle_and_surface_emulated():
    """oracle == torch autograd on F.mse_loss + the reference weighted loss; the Python surface
    (HeatmapMSELoss / HeatmapJointLoss) through the emulated C ABI == oracle."""
    import torch.nn.functional as F
    import lib.core.integral_loss as il
    hm, tgt, wh, x, t, w = gi.heatmap_case(3, 5, 16, 24, 71)
    for kind in ("l1", "smoothl1", "mse"):
        th = torch.from_numpy(hm).double().requires_grad_(True)
        tx = torch.from_numpy(x).double().requires_grad_(True)
        ww = torch.from_numpy(wh).double().reshape(3, 5, 1, 1)
        lh = F.mse_loss(th * ww, torch.from_numpy(tgt).double() * ww)
        d = tx - torch.from_numpy(t).double()
        l = {"l1": d.abs(), "mse": d * d,
             "smoothl1": torch.where(d.abs() < 1, 0.5 * d * d, d.abs() - 0.5)}[kind]
        lj = (l * torch.from_numpy(w).double()).sum() / len(x)
        (0.5 * lh + 3.0 * lj).backward()
        o_hm, o_jt, o_tot, o_dhm, o_dx = restate.heatmap_joint_loss(hm, tgt, wh, x, t, w, kind, 0.5, 3.0)
        assert abs(o_hm - lh.item()) <= 1e-12 and abs(o_jt - lj.item()) <= 1e-12
        assert np.allclose(o_dhm, th.grad.numpy(), rtol=0, atol=1e-14)
        assert np.allclose(o_dx, tx.grad.numpy(), rtol=0, atol=1e-14)
    il._backend[0] = emul_ops
    try:
        th = torch.from_numpy(hm).requires_grad_(True)
        tx = torch.from_numpy(x).requires_grad_(True)
        crit = il.HeatmapJointLoss(5, kind="smoothl1", hm_scale=0.5, jt_scale=3.0)
        tot = crit((th, tx), torch.from_numpy(tgt), torch.from_numpy(t), torch.from_numpy(w),
                   hm_weight=torch.from_numpy(wh))
        tot.backward()
        o_hm, o_jt, o_tot, o_dhm, o_dx = restate.heatmap_joint_loss(hm, tgt, wh, x, t, w, "smoothl1", 0.5, 3.0)
        assert abs(tot.item() - o_tot) <= 1e-5 * abs(o_tot)
        assert abs(crit.last_parts[0].item() - o_hm) <= 1e-5 * o_hm
        assert abs(crit.last_parts[1].item() - o_jt) <= 1e-5 * o_jt
        assert relerr(th.grad.numpy(), o_dhm) <= 1e-5 and relerr(tx.grad.numpy(), o_dx) <= 1e-5
        # heat-map loss alone == F.mse_loss (no weights)
        th2 = torch.from_numpy(hm).requires_grad_(True)
        l2 = il.HeatmapMSELoss()(th2, torch.from_numpy(tgt))
        assert abs(l2.item() - F.mse_loss(torch.from_numpy(hm), torch.from_numpy(tgt)).item()) <= 1e-6
        with pytest.raises(ValueError):
            il.HeatmapMSELoss(True)(th2, torch.from_numpy(tgt))
        with pytest.raises(ValueError):
            il.HeatmapMSELoss()(th2, torch.from_numpy(tgt[:, :2]))
    finally:
        il._backend[0] = __import__("epipolarpose_b200.ops", fromlist=["ops"])


def test_h36m_eval_surface_emulated():
    """lib/dataset/h36m_eval.evaluate_h36m through the emulated C ABI == oracle == reference
    golden values; argument validation as the reference's array indexing would fail."""
    import lib.dataset.h36m_eval as he
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "h36m_eval.npz")))
    pred, gt, pelvis, fl, c_p = gi.eval_case()
    he._backend[0] = emul_ops
    try:
        for mpii, tag in ((False, "h36m"), (True, "mpii")):
            p = pred[:, he.H36M_TO_MPII_PERM, :] if mpii else pred
            nv, perf, det = he.evaluate_h36m(p, gt, pelvis, fl, c_p, mpii_order=mpii, return_poses=True)
            assert [n for n, _ in nv] == he.METRIC_NAMES
            assert np.max(np.abs(np.array([v for _, v in nv]) - g[tag + "_values"])) <= 1e-8
            assert abs(perf - float(g[tag + "_mean"])) <= 1e-8
            o = restate.h36m_evaluate(p, gt, pelvis[:, 2], fl, c_p, mpii_order=mpii)
            assert np.max(np.abs(det["metrics"] - o["metrics"])) <= 1e-8
            assert np.array_equal(det["pck"], o["pck"])
            assert np.max(np.abs(det["poses"] - o["poses"])) <= 1e-8
        with pytest.raises(ValueError):
            he.evaluate_h36m(pred[:, :5], gt, pelvis, fl, c_p)
        nv, perf, det = he.evaluate_h36m(pred[:0], gt[:0], pelvis[:0], fl[:0], c_p[:0])
        assert perf == 0.0 and det["metrics"].shape == (0, 9)
    finally:
        he._backend[0] = __import__("epipolarpose_b200.ops", fromlist=["ops"])


@pytest.fixture(scope="module")
def host_geometry(tmp_path_factory):
    """tests/harness/host_geometry.cu: the __host__ __device__ bodies of csrc/geometry.cu built
    for the CPU with nvcc (same source and --fmad=false arithmetic as the kernels)."""
    import shutil
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    exe = str(tmp_path_factory.mktemp("harness") / "host_geometry")
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "--fmad=false", "-O1",
                        "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "harness", "host_geometry.cu")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr

    def run(args, *arrays):
        inp = b"".join(np.ascontiguousarray(a, dtype=np.float64).tobytes() for a in arrays)
        out = subprocess.run([exe] + [str(a) for a in args], input=inp, capture_output=True)
        assert out.returncode == 0, out.stderr
        return np.frombuffer(out.stdout, dtype=np.float64)
    return run


@pytest.mark.parametrize("mpii", [False, True])
def test_h36m_eval_kernel_body_on_host(host_geometry, mpii):
    """the per-sample body of h36m_eval_kernel, executed on the CPU, against the numpy oracle."""
    pred, gt, pelvis, fl, c_p = gi.eval_case(64, 17, 82)
    p = pred[:, restate.H36M_TO_MPII_PERM, :3] if mpii else pred[:, :, :3]
    g = gt[:, restate.H36M_TO_MPII_PERM, :] if mpii else gt
    S, J = p.shape[:2]
    cam = np.concatenate([fl, c_p, pelvis[:, 2:3]], 1)
    j14 = restate.J14_MPII if mpii else restate.J14_H36M
    a = host_geometry(["eval", S, J, 6 if mpii else 0, sum(1 << j for j in j14)], p, g, cam)
    met, pj, poses = a[:S * 9].reshape(S, 9), a[S * 9:S * 9 + S * J].reshape(S, J), a[S * 9 + S * J:].reshape(S, J, 9)
    o = restate.h36m_evaluate(p, gt, pelvis[:, 2], fl, c_p, mpii_order=mpii)
    assert np.max(np.abs(met - o["metrics"])) <= 1e-9
    assert np.max(np.abs(pj - o["per_joint"])) <= 1e-9
    assert np.max(np.abs(poses - o["poses"])) <= 1e-9


def test_polynomial_correction_kernel_body_on_host(host_geometry):
    """fundamental_from_P + correct_match of csrc/geometry.cu (Laguerre root finder, float64),
    executed on the CPU, against cv2.correctMatches outputs stored by the reference run."""
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "triangulation_poly.npz")))
    u1, u2, P1, P2, X = gi.triangulation_case()
    for i in range(len(u1)):
        N = len(u1[i])
        a = host_geometry(["correct", N], P1[i], P2[i], u1[i], u2[i])
        F, n1, n2 = a[:9].reshape(3, 3), a[9:9 + 2 * N].reshape(N, 2), a[9 + 2 * N:].reshape(N, 2)
        Fo = restate.fundamental_from_projections(P1[i], P2[i])
        assert np.max(np.abs(F - Fo)) <= 1e-12 * np.abs(Fo).max()
        assert np.max(np.abs(n1 - g["corrected_u1"][i])) <= 1e-9          # px
        assert np.max(np.abs(n2 - g["corrected_u2"][i])) <= 1e-9
    # exact projections are a fixed point of the correction
    u1e, u2e = gi.exact_projections(P1, P2, X)
    a = host_geometry(["correct", 17], P1[0], P2[0], u1e[0], u2e[0])
    assert np.max(np.abs(a[9:9 + 34].reshape(17, 2) - u1e[0])) <= 1e-8


def test_eight_point_kernel_body_on_host(host_geometry):
    """fundamental_8point of csrc/geometry.cu (Jacobi eigenvectors of the 9x9 normal matrix,
    rank-2 projection), executed on the CPU, against cv2.findFundamentalMat(FM_8POINT)."""
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "triangulation_8point.npz")))
    u1, u2, P1, P2, X = gi.triangulation_case()
    for i in range(len(u1)):
        a = host_geometry(["f8", len(u1[i])], u1[i], u2[i])
        assert a[0] == 1.0
        F = a[1:].reshape(3, 3)
        assert np.max(np.abs(F - g["f8"][i])) <= 1e-9 * np.abs(g["f8"][i]).max()
    a = host_geometry(["f8", 17], np.ones((17, 2)), np.ones((17, 2)))     # degenerate: no matrix
    assert a[0] == 0.0
    # identical cameras: F is exactly zero and the correction NaN for every match (the trigger
    # of the fallback, lib/utils/triangulation.py:213-215)
    a = host_geometry(["correct", 17], P1[0], P1[0], u1[0], u2[0])
    assert np.all(a[:9] == 0.0) and np.isnan(a[9:]).all()


MEAN = np.array([123.675, 116.280, 103.530])
STD = np.array([58.395, 57.120, 57.375])


@pytest.mark.parametrize("tag", list(gi.PATCH_CASES))
def test_input_pipeline_kernel_body_on_host(host_geometry, tag):
    """warp_pixel_u8 / finish_pixel / patch_affine_fwd / patch_joint of csrc/input.cu, executed on
    the CPU: patches BIT-EXACT against the unmodified get_single_patch_sample (cv2.warpAffine)."""
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "patch_sample.npz")))
    img, box, joints, vis, pw, ph, seed = gi.frame_case(tag)
    H, W = img.shape[:2]
    for aug in (False, True):
        k = tag + ("_aug" if aug else "")
        sc, rot, fl, c0, c1, c2 = g[k + "_aug"]
        a = host_geometry(["patch", H, W, pw, ph, int(fl), 17], np.array(list(box) + [sc, rot]),
                          np.array([c0, c1, c2]), np.concatenate([MEAN, STD]), np.array([2000.0 * sc]), joints,
                          img.astype(np.float64))
        patch = a[6:6 + 3 * ph * pw].reshape(3, ph, pw).astype(np.float32)
        assert np.array_equal(patch, g[k + "_patch"]), k
        assert np.max(np.abs(a[6 + 3 * ph * pw:] - g[k + "_label"])) <= 1e-12


def test_input_pipeline_surface_emulated(tmp_path):
    """get_single_patch_sample / generate_patch_batch_device of the mirror through the emulated ABI:
    reference return tuple, same RNG draws as the reference's do_augmentation, error behaviour."""
    import random
    import lib.utils.img_utils as iu
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "patch_sample.npz")))
    iu._backend[0] = emul_ops
    try:
        for tag in ("noise64", "edge48"):
            img, box, joints, vis, pw, ph, seed = gi.frame_case(tag)
            for aug in (False, True):
                k = tag + ("_aug" if aug else "")
                np.random.seed(seed); random.seed(seed)
                patch, label, weight, scale, rot = iu.get_single_patch_sample(
                    img, box[0], box[1], box[2], box[3], joints.copy(), vis.copy(), [], None, pw, ph, 2000.0,
                    2000.0, MEAN, STD, aug, None)
                assert (scale, rot) == (g[k + "_aug"][0], g[k + "_aug"][1])      # same draws as the reference
                assert patch.dtype == np.float32 and np.array_equal(patch, g[k + "_patch"])
                assert np.max(np.abs(label - g[k + "_label"])) <= 1e-12
                assert np.array_equal(weight, g[k + "_weight"])
        # batched entry point with frames of different sizes
        a, b = gi.frame_case("noise64"), gi.frame_case("edge48")
        out, trans, _ = iu.generate_patch_batch_device([a[0], b[0]], [a[1][0], b[1][0]], [a[1][1], b[1][1]],
                                                       [a[1][2], b[1][2]], [a[1][3], b[1][3]], 48, 48,
                                                       mean=MEAN, std=STD)
        assert np.array_equal(out[1].numpy(), g["edge48_patch"]) and out.shape == (2, 3, 48, 48)
        # occluder augmentation (augmentation.py:61-123) through the emulated epb_patch_sample_occ:
        # same draws / resizes as the unmodified reference, bit-exact patches
        go = dict(np.load(os.path.join(ROOT, "tests", "golden", "patch_occluders.npz")))
        occ = gi.occluder_set()
        for tag in ("noise64", "edge48"):
            img, box, joints, vis, pw, ph, seed = gi.frame_case(tag)
            for aug in (False, True):
                k = tag + ("_aug" if aug else "")
                np.random.seed(seed + 7); random.seed(seed + 7)
                patch, label, weight, scale, rot = iu.get_single_patch_sample(
                    img, box[0], box[1], box[2], box[3], joints.copy(), vis.copy(), [], None, pw, ph, 2000.0,
                    2000.0, MEAN, STD, aug, None, occluder=occ)
                assert np.array_equal(patch, go[k + "_patch"]), k
        with pytest.raises(ValueError):
            iu.generate_patch_batch_device([a[0].astype(np.float32)], [1], [1], [1], [1], 8, 8)
        with pytest.raises(IOError):
            iu.get_single_patch_sample(str(tmp_path / "missing.png"), 1, 1, 1, 1, a[2], a[3], [], None, 8, 8, 1, 1,
                                       None, None, False, None)
    finally:
        iu._backend[0] = __import__("epipolarpose_b200.ops", fromlist=["ops"])


@pytest.mark.parametrize("V", [2, 3, 4])
def test_nview_dlt_kernel_body_on_host(host_geometry, V):
    """dlt_nview<V> of csrc/geometry.cu (one-sided Jacobi on the 2V x 4 system), executed on the
    CPU, against the numpy-SVD oracle: <= 1e-6 mm with 3 px observation noise."""
    rng = np.random.default_rng(30 + V)
    R, T, f, c, P = restate.synthetic_cameras(rng, 4, 4)
    for t in range(4):
        X = rng.normal(0, 400, (17, 3))
        us = np.stack([restate.project(P[t, v], X) for v in range(V)]) + rng.normal(0, 3, (V, 17, 2))
        xo, _ = restate.linear_eigen_triangulation_nview(us, P[t, :V])
        xh = host_geometry(["nview", V, 17], us, P[t, :V]).reshape(17, 3)
        assert np.max(np.abs(xh - xo)) <= 1e-6


def _refiner_case(precision):
    from oracle import restate_refiner as rr
    from epipolarpose_b200.refiner import model as rmodel
    sd = rr.init_state(rr.param_shapes(128, 45, 45), 17)
    m = rmodel.LinearModelPG(linear_size=128, p_dropout=0.0, input_size=45, output_size=45, precision=precision)
    assert list(m.state_dict().keys()) == list(sd.keys())
    m.load_state_dict(sd)
    return rr, rmodel, sd, m


def test_refiner_surface_emulated():
    """epipolarpose_b200/refiner/model.py (reference names, state_dict, forward signature) over
    mlp.MLPEngine through the emulated C ABI: forward / backward / running statistics / eval against
    the golden vectors of the unmodified reference; dropout against the oracle with the same masks."""
    from epipolarpose_b200.refiner import model as rmodel
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "refiner.npz")))
    rmodel.LinearModelPG._backend[0] = emul_ops
    try:
        rr, _, sd, m = _refiner_case("fp32")
        x = torch.from_numpy(gi.grad_like((24, 45), 18)).requires_grad_(True)
        tgt = torch.from_numpy(gi.grad_like((24, 45), 19))
        m.train()
        p1, p2 = m(x)
        loss = torch.nn.functional.mse_loss(p1, tgt) + torch.nn.functional.mse_loss(p2, tgt)
        loss.backward()
        assert relerr(p1.detach().numpy(), g["p1"]) <= 1e-5 and relerr(p2.detach().numpy(), g["p2"]) <= 1e-5
        assert relerr(x.grad.numpy(), g["dx"]) <= 1e-4
        named = dict(m.named_parameters())
        for k in [k[5:] for k in g if k.startswith("grad/")]:
            assert relerr(named[k].grad.numpy(), g["grad/" + k]) <= 1e-4, k
        assert relerr(m.state_dict()["batch_norm1.running_var"].numpy(), g["batch_norm1.running_var"]) <= 1e-5
        assert int(m.state_dict()["batch_norm1.num_batches_tracked"]) == 1
        m.eval()
        with torch.no_grad():
            e1, e2 = m(x.detach())
        assert relerr(e1.numpy(), g["eval_p1"]) <= 1e-5 and relerr(e2.numpy(), g["eval_p2"]) <= 1e-5
        # dropout: the engine draws its keep masks with torch.rand; replay them through the oracle
        rr, _, sd, m = _refiner_case("fp32")
        m.p_dropout = 0.5
        m.train()
        torch.manual_seed(123)
        q1, q2 = m(x.detach())
        torch.manual_seed(123)
        masks = [(torch.rand(24, 128) >= 0.5) for _ in range(10)]
        o1, o2 = rr.forward(sd, x.detach(), training=True, masks=masks, p_dropout=0.5)
        assert relerr(q1.detach().numpy(), o1.numpy()) <= 1e-5 and relerr(q2.detach().numpy(), o2.numpy()) <= 1e-5
        # two forward passes alive at once: each backward uses its own record
        rr, _, sd, m = _refiner_case("fp32")
        m.train()
        xa = torch.from_numpy(gi.grad_like((24, 45), 18)).requires_grad_(True)
        xb = torch.from_numpy(gi.grad_like((24, 45), 21)).requires_grad_(True)
        a1, _ = m(xa)
        b1, _ = m(xb)
        a1.sum().backward()
        pa = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v) for k, v in sd.items()}
        xo = xa.detach().clone().requires_grad_(True)
        rr.forward(pa, xo, training=True)[0].sum().backward()
        assert relerr(xa.grad.numpy(), xo.grad.numpy()) <= 1e-4 and xb.grad is None
        with pytest.raises(NotImplementedError):
            rmodel.LinearModelPG(leaky=True)
        with pytest.raises(NotImplementedError):
            rmodel.LinearPG(64, bn=False)
    finally:
        rmodel.LinearModelPG._backend[0] = None


def test_fused_optimizers_match_torch():
    import lib.utils.utils as U
    U._backend[0] = emul_ops
    try:
        torch.manual_seed(0)
        for kind in ("adam", "sgd"):
            ps = [torch.nn.Parameter(torch.randn(s)) for s in ((7, 3), (64,), (5, 5, 3), (17,))]
            qs = [torch.nn.Parameter(p.detach().clone()) for p in ps]
            if kind == "adam":
                a, b = U.FusedAdam(ps, lr=1e-2), torch.optim.Adam(qs, lr=1e-2)
            else:
                a = U.FusedSGD(ps, lr=1e-2, momentum=0.9, weight_decay=1e-4, nesterov=True)
                b = torch.optim.SGD(qs, lr=1e-2, momentum=0.9, weight_decay=1e-4, nesterov=True)
            sched = torch.optim.lr_scheduler.MultiStepLR(a, [2], 0.1)
            schedb = torch.optim.lr_scheduler.MultiStepLR(b, [2], 0.1)
            for it in range(4):
                for p, q in zip(ps, qs):
                    g = torch.randn_like(p)
                    p.grad, q.grad = g.clone(), g.clone()
                a.step(); b.step(); sched.step(); schedb.step()
            for p, q in zip(ps, qs):
                assert relerr(p.detach().numpy(), q.detach().numpy()) <= 1e-5
    finally:
        U._backend[0] = __import__("epipolarpose_b200.ops", fromlist=["ops"])


def test_synthetic_dataset_contract_and_pairing():
    from lib.core.config import config, reset_config
    import lib.dataset as dataset
    reset_config()
    config.MODEL.NUM_JOINTS = 16
    ds = eval("dataset.synthetic_h36m")(cfg=config, root="", image_set="train", is_train=True)
    img, label, weight, meta = ds[5]
    assert img.shape == (3, 256, 256) and img.dtype == torch.float32
    assert label.shape == (48,) and weight.shape == (48,)
    for k in ("center_x", "center_y", "width", "height", "scale", "rot", "R", "T", "f", "c",
              "projection_matrix", "image"):
        assert k in meta
    P = restate.projection_matrix(meta["R"], meta["T"], meta["f"], meta["c"])
    assert np.allclose(P, meta["projection_matrix"])
    b = next(iter(ds.pair_batch_sampler(3)))
    half = len(b) // 2
    for i in range(half):                # halves pair neighbouring views of the same tuple
        a, c = ds.db[b[i]], ds.db[b[half + i]]
        assert a["tuple"] == c["tuple"] and (a["view"], c["view"]) in ((0, 1), (3, 2))
    assert len(ds.db) == len(ds)


def _ddp_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank),
                      WORLD_SIZE=str(world))
    import torch.distributed as dist
    dist.init_process_group("gloo", rank=rank, world_size=world)
    import lib.models as models
    cfg = refshim.make_cfg(num_layers=18, num_joints=2, volume=True, depth_res=4, image_size=(32, 32))
    m = models.pose3d_resnet.get_pose_net(cfg, False, ops=emul_ops)
    m.load_state_dict(restate_net.init_state(restate_net.param_shapes(18, 2, True, 4), 1))
    m.train()
    x = torch.from_numpy(gi.images(4, 32, 100))[2 * rank:2 * rank + 2]
    g = torch.from_numpy(gi.grad_like((4, 8, 8, 8), 101))[2 * rank:2 * rank + 2]
    import torch.distributed as d2
    orig = d2.all_reduce

    class _Done:
        def wait(self):
            return True

    def avg(t, op=None, async_op=False):          # gloo has no AVG: emulate with SUM / world
        orig(t)
        t /= world
        return _Done()
    d2.all_reduce = avg
    (m(x) * g).sum().backward()
    got = {k: p.grad.numpy().copy() for k, p in m.named_parameters()}
    # the semantics of nn.DataParallel over replicas (scripts/train.py:94,143): the all-reduced
    # gradient is the MEAN of the per-replica gradients, each with its own BatchNorm statistics
    # -- recomputed here on one process, replica by replica, without any collective
    ref = None
    for r in range(world):
        m1 = models.pose3d_resnet.get_pose_net(cfg, False, ops=emul_ops, allreduce_grads=False)
        m1.load_state_dict(restate_net.init_state(restate_net.param_shapes(18, 2, True, 4), 1))
        m1.train()
        xr = torch.from_numpy(gi.images(4, 32, 100))[2 * r:2 * r + 2]
        gr = torch.from_numpy(gi.grad_like((4, 8, 8, 8), 101))[2 * r:2 * r + 2]
        (m1(xr) * gr).sum().backward()
        cur = {k: p.grad.numpy().astype(np.float64) / world for k, p in m1.named_parameters()}
        ref = cur if ref is None else {k: ref[k] + cur[k] for k in ref}
    worst = max(float(np.max(np.abs(got[k] - ref[k])) / max(np.max(np.abs(ref[k])), 1e-30)) for k in got)
    q.put((rank, (got, worst)))
    dist.destroy_process_group()


def test_data_parallel_allreduce_world2_gloo():
    """Two ranks, each with its own half batch: after the stage-wise all-reduce in the model's
    backward both ranks hold identical gradients, equal to the mean of the per-replica gradients
    (per-replica BatchNorm statistics: the reference's nn.DataParallel semantics)."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 500)
    ps = [ctx.Process(target=_ddp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    res = dict(q.get(timeout=240) for _ in ps)
    for p in ps:
        p.join(60)
    for k in res[0][0]:
        assert np.array_equal(res[0][0][k], res[1][0][k]), k
    assert any(np.abs(v).max() > 0 for v in res[0][0].values())
    assert res[0][1] <= 1e-5 and res[1][1] <= 1e-5      # == mean of the per-replica gradients


def test_bench_reference_arm_cli():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                          "--steps", "1", "--warmup", "0", "--layers", "18", "--cpu-tuples", "1"],
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    import json
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0 and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0


# ------------------------------------------------------------------ split-fp16 engine (net16.Engine16)
def test_engine16_matches_oracle_through_emulated_abi():
    """The f16x3 engine walk (split operands, per-tensor scales from statistics, dynamic dz
    scales, in-place masked residual join, final-layer backward on the fp32-operand kernels)
    through the CPU emulation of the split family: forward and EVERY gradient against the
    float64 oracle, and .eval() against the unmodified reference's golden output."""
    import lib.models as models
    from epipolarpose_b200 import net16
    c = gi.NET_CASES["r18"]
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "net_r18.npz")))
    cfg = refshim.make_cfg(num_layers=18, num_joints=c["J"], volume=True, depth_res=c["D"],
                           image_size=(c["HW"], c["HW"]))
    shapes = restate_net.param_shapes(18, c["J"], True, c["D"])
    sd = restate_net.init_state(shapes, c["seed"])
    m = models.pose3d_resnet.get_pose_net(cfg, False, ops=emul_ops, precision="f16x3")
    m.load_state_dict(sd)
    m.train()
    assert isinstance(m._engine(), net16.Engine16)
    x = torch.from_numpy(gi.images(c["N"], c["HW"], c["seed"]))
    p = {k: (v.double().clone().requires_grad_(True) if v.is_floating_point() and "running" not in k
             else (v.double() if v.is_floating_point() else v)) for k, v in sd.items()}
    ref = restate_net.forward(p, x.double(), num_layers=18, volume=True, image_size=(c["HW"], c["HW"]))
    out = m(x)
    assert relerr(out.detach().numpy(), ref.detach().numpy()) <= 2e-5
    assert relerr(out.detach().numpy(), g["out0"]) <= 1e-4
    m.eval()
    with torch.no_grad():
        e = m(x)
    assert relerr(e.numpy(), g["eval_out0"]) <= 1e-4     # un-normalised activations: dynamic scales
    # gradients on the seed the 3xTF32 engine test uses (the golden r18 batch sits on a ReLU
    # flip: ONE unit that the float32 and float64 evaluations resolve differently moves trunk
    # gradients by 2-4e-3 -- the float32 oracle shows the same, see test_gpu_parity.py)
    sd = restate_net.init_state(shapes, 9)
    m.load_state_dict(sd)
    m.train()
    x = torch.from_numpy(gi.images(2, c["HW"], 9))
    p = {k: (v.double().clone().requires_grad_(True) if v.is_floating_point() and "running" not in k
             else (v.double() if v.is_floating_point() else v)) for k, v in sd.items()}
    ref = restate_net.forward(p, x.double(), num_layers=18, volume=True, image_size=(c["HW"], c["HW"]))
    out = m(x)
    assert relerr(out.detach().numpy(), ref.detach().numpy()) <= 2e-5
    go = torch.from_numpy(gi.grad_like(out.shape, 10))
    (out * go).sum().backward()
    (ref * go.double()).sum().backward()
    for k, q in m.named_parameters():
        assert relerr(q.grad.numpy(), p[k].grad.numpy()) <= 1e-4, k
    # a head with a whole 64-channel block (J*D = 64): the final layer's backward also runs on
    # the split kernels (the fp32 logit gradient is split by epb_split16)
    J2, D2 = 4, 16
    cfg2 = refshim.make_cfg(num_layers=18, num_joints=J2, volume=True, depth_res=D2, image_size=(64, 64))
    sd2 = restate_net.init_state(restate_net.param_shapes(18, J2, True, D2), 9)
    m2 = models.pose3d_resnet.get_pose_net(cfg2, False, ops=emul_ops, precision="f16x3")
    m2.load_state_dict(sd2)
    m2.train()
    p2 = {k: (v.double().clone().requires_grad_(True) if v.is_floating_point() and "running" not in k
              else (v.double() if v.is_floating_point() else v)) for k, v in sd2.items()}
    ref2 = restate_net.forward(p2, x.double(), num_layers=18, volume=True, image_size=(64, 64))
    out2 = m2(x)
    go2 = torch.from_numpy(gi.grad_like(out2.shape, 11))
    (out2 * go2).sum().backward()
    (ref2 * go2.double()).sum().backward()
    for k, q in m2.named_parameters():
        assert relerr(q.grad.numpy(), p2[k].grad.numpy()) <= 1e-4, k


def test_engine16_falls_back_when_channels_do_not_fit():
    import lib.models as models
    from epipolarpose_b200 import net, net16
    cfg = refshim.make_cfg(num_layers=18, num_joints=3, volume=True, depth_res=8, image_size=(64, 64))
    cfg.MODEL.EXTRA.NUM_DECONV_FILTERS = [96, 96, 96]      # not whole 64-channel TMA boxes
    m = models.pose3d_resnet.get_pose_net(cfg, False, ops=emul_ops, precision="f16x3")
    eng = m._engine()
    assert isinstance(eng, net.Engine) and not isinstance(eng, net16.Engine16) and eng.precision == 3


def test_fused_optimizers_interchange_with_torch_optim_and_survive_rematerialisation():
    """ADVICE r1: state_dict()/load_state_dict() in the torch.optim per-parameter layout (a
    reference checkpoint resumes bit-identically, and vice versa), and parameters that were
    re-materialised after the optimiser was built (model.cuda() / .to()) keep training."""
    import lib.utils.utils as U
    U._backend[0] = emul_ops
    torch.manual_seed(0)
    ws = [torch.randn(5, 3), torch.randn(7), torch.randn(2, 2, 3)]
    for fused_cls, torch_cls, kw in ((U.FusedAdam, torch.optim.Adam, dict(lr=1e-2)),
                                     (U.FusedSGD, torch.optim.SGD, dict(lr=1e-2, momentum=0.9))):
        pa = [torch.nn.Parameter(w.clone()) for w in ws]
        pb = [torch.nn.Parameter(w.clone()) for w in ws]
        oa, ob = fused_cls(pa, **kw), torch_cls(pb, **kw)

        def step(pairs, gs):
            for ps, o in pairs:
                for q, g_ in zip(ps, gs):
                    q.grad = g_.clone()
                o.step()
        for _ in range(3):
            step(((pa, oa), (pb, ob)), [torch.randn_like(w) for w in ws])
        assert max((a - b).abs().max().item() for a, b in zip(pa, pb)) <= 1e-7
        pc = [torch.nn.Parameter(q.detach().clone()) for q in pb]
        oc = fused_cls(pc, **kw)
        oc.load_state_dict(ob.state_dict())                       # torch checkpoint -> fused
        pd = [torch.nn.Parameter(q.detach().clone()) for q in pa]
        od = torch_cls(pd, **kw)
        od.load_state_dict(oa.state_dict())                       # fused checkpoint -> torch
        step(((pa, oa), (pb, ob), (pc, oc), (pd, od)), [torch.randn_like(w) for w in ws])
        assert max((a - b).abs().max().item() for a, b in zip(pc, pb)) <= 1e-7
        assert max((a - b).abs().max().item() for a, b in zip(pd, pa)) <= 1e-7
        for q in pa:
            q.data = q.data.clone()                               # what model.to(device) does
        step(((pa, oa), (pb, ob)), [torch.randn_like(w) for w in ws])
        assert max((a - b).abs().max().item() for a, b in zip(pa, pb)) <= 1e-6


def test_refiner_train_loop_and_checkpoint_interop_emulated(tmp_path, monkeypatch):
    """epipolarpose_b200/refiner/main.py train() / test() / save_ckpt (reference refiner/main.py:
    31-84, refiner/utils.py:18-36) through the emulated ABI: parameters after an epoch equal an
    independent loop built from the oracle network + torch.optim.Adam + torch's clip_grad_norm_
    + the reference's lr_decay; the checkpoint resumes in torch.optim.Adam (and back)."""
    import logging
    import types
    from oracle import restate_refiner as rr
    from epipolarpose_b200.refiner import main as rmain, model as rmodel, utils as rutils, data as rdata
    import lib.utils.utils as U
    monkeypatch.setattr(rmain, "_to_device", lambda t: t)     # the emulation computes on the host
    rmodel.LinearModelPG._backend[0] = emul_ops
    rutils._backend[0] = emul_ops
    U._backend[0] = emul_ops
    try:
        sd = rr.init_state(rr.param_shapes(128, 45, 45), 17)
        m = rmodel.LinearModelPG(linear_size=128, p_dropout=0.0, input_size=45, output_size=45, precision="fp32")
        m.load_state_dict(sd)
        ds = rdata.SyntheticPoses(is_train=True, n=96, seed=3)
        dl = torch.utils.data.DataLoader(ds, batch_size=32, shuffle=False)
        args = types.SimpleNamespace(lr=1e-3, lr_decay=2, lr_gamma=0.9)
        opt = U.FusedAdam(list(m.parameters()), lr=args.lr)
        crit = torch.nn.MSELoss(reduction='mean')
        step, lr_now = rmain.train(m, dl, opt, 0, args.lr, crit, args, logging.getLogger("t"))
        assert step == 3 and abs(lr_now - 1e-3 * 0.9 ** 1.0) < 1e-12      # decayed at steps 1 and 2
        # independent loop
        p = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v.clone())
             for k, v in sd.items()}
        plist = [v for k, v in p.items() if torch.is_tensor(v) and v.requires_grad]
        ro = torch.optim.Adam(plist, lr=args.lr)
        g = 0
        for inp, tar in dl:
            g += 1
            if g % args.lr_decay == 0 or g == 1:
                for pg in ro.param_groups:
                    pg['lr'] = args.lr * args.lr_gamma ** (g / args.lr_decay)
            o1, o2 = rr.forward(p, inp, training=True)
            ro.zero_grad()
            (torch.nn.functional.mse_loss(o1, tar) + torch.nn.functional.mse_loss(o2, tar)).backward()
            torch.nn.utils.clip_grad_norm_(plist, max_norm=1.)
            ro.step()
        for k, q in m.named_parameters():
            # Adam normalises by sqrt(v): a bias in front of a BatchNorm has a noise-only gradient
            # (exactly zero in exact arithmetic) that becomes +-lr steps of arbitrary sign
            a, b = q.detach().numpy(), p[k].detach().numpy()
            assert np.max(np.abs(a - b)) <= 2e-4 * np.max(np.abs(b)) + 3 * 1e-3 * (1 if k.endswith(".bias") else 0), k
        err = rmain.test(m, torch.utils.data.DataLoader(rdata.SyntheticPoses(False, n=64, seed=3), batch_size=32))
        assert np.isfinite(err) and err > 0
        # checkpoint: the reference's dictionary, optimizer state in the torch.optim layout
        rutils.save_ckpt({'epoch': 1, 'lr': lr_now, 'step': step, 'err': err, 'state_dict': m.state_dict(),
                          'optimizer': opt.state_dict()}, ckpt_path=str(tmp_path), is_best=True)
        ck = torch.load(str(tmp_path / 'best.pth.tar'), weights_only=False)
        m2 = rmodel.get_model(str(tmp_path / 'best.pth.tar'), linear_size=128, p_dropout=0.0, precision="fp32")
        for (k, a), (_, b) in zip(m.state_dict().items(), m2.state_dict().items()):
            assert torch.equal(a, b), k
        t_opt = torch.optim.Adam([torch.nn.Parameter(v.detach().clone()) for v in m.parameters()], lr=1e-3)
        t_opt.load_state_dict(ck['optimizer'])                  # loads into the reference's optimiser
        assert int(t_opt.state[t_opt.param_groups[0]['params'][0]]['step']) == 3
        opt2 = U.FusedAdam(list(m2.parameters()), lr=1e-3)
        opt2.load_state_dict(ro.state_dict())                   # and a torch.optim checkpoint into ours
        assert opt2.state['flat0']['step'] == 3
        # clip_grad_norm_ alone against torch
        ws = [torch.nn.Parameter(torch.randn(7, 5)), torch.nn.Parameter(torch.randn(11))]
        for w in ws:
            w.grad = torch.randn_like(w) * 3
        ref = [w.grad.clone() for w in ws]
        tn = torch.nn.utils.clip_grad_norm_([torch.nn.Parameter(r) for r in ref], 1.0)   # dummy: norm only
        want = [r * min(1.0, 1.0 / (float(torch.sqrt(sum((r ** 2).sum() for r in ref))) + 1e-6)) for r in ref]
        got_norm = rutils.clip_grad_norm_(ws, 1.0)
        assert abs(float(got_norm) - float(torch.sqrt(sum((r ** 2).sum() for r in ref)))) <= 1e-5
        for w, r in zip(ws, want):
            assert relerr(w.grad.numpy(), r.numpy()) <= 1e-6
    finally:
        real = __import__("epipolarpose_b200.ops", fromlist=["ops"])
        rmodel.LinearModelPG._backend[0] = None
        rutils._backend[0] = real
        U._backend[0] = real


def test_joint_loss_broadcasts_or_raises_like_the_reference():
    """ADVICE r1: target / weights smaller than the input must broadcast the way the reference's
    elementwise arithmetic does (integral_loss.py:12-14) or raise -- never be read out of bounds."""
    import lib.core.integral_loss as il
    il._backend[0] = emul_ops
    try:
        rng = np.random.default_rng(0)
        x = torch.from_numpy(rng.standard_normal((4, 15)).astype(np.float32)).requires_grad_(True)
        t = torch.from_numpy(rng.standard_normal((4, 15)).astype(np.float32))
        w_col = torch.from_numpy((rng.random((4, 1)) > 0.3).astype(np.float32))
        loss = il.weighted_l1_loss(x, t, w_col, True)
        ref = (torch.abs(x.detach() - t) * w_col).sum() / 4
        assert abs(loss.item() - ref.item()) <= 1e-6
        loss.backward()
        assert torch.allclose(x.grad, torch.sign(x.detach() - t) * w_col / 4, atol=1e-7)
        row = il.weighted_smooth_l1_loss(x, t[:1], torch.ones(15), False)       # [1,15] and [15] broadcast
        d = x.detach() - t[:1]
        ref = torch.where(d.abs() < 1, 0.5 * d * d, d.abs() - 0.5).sum()
        assert abs(row.item() - ref.item()) <= 1e-5 * ref.item()
        with pytest.raises(RuntimeError):
            il.weighted_l1_loss(x, t[:, :7], torch.ones(4, 15), True)
        with pytest.raises(RuntimeError):
            il.weighted_l1_loss(x, t, torch.ones(3, 15), True)
        hm, tg = torch.rand(4, 5, 8, 8), torch.rand(4, 5, 8, 8)
        with pytest.raises(ValueError):
            il.heatmap_joint_loss(hm, tg[:2])
        total, parts = il.heatmap_joint_loss(hm, tg, None, x.detach(), t, w_col)
        ref_jt = (torch.abs(x.detach() - t) * w_col).sum() / 4
        assert abs(parts[1].item() - ref_jt.item()) <= 1e-6 and torch.isfinite(total)
    finally:
        il._backend[0] = __import__("epipolarpose_b200.ops", fromlist=["ops"])


@pytest.mark.parametrize("extra_consumer", [False, True])
def test_logit_gradient_sink_equals_fp32_route_emulated(extra_consumer):
    """The criterion hands the logit gradient to the network's backward as split planes + bias gradient
    (_sinks.py, epb_softargmax_bwd_split).  Same parameter gradients as the fp32 route (sink detached);
    with a second consumer of the logits the zero token keeps autograd's accumulation exact."""
    import lib.models as models
    import lib.core.integral_loss as il
    from tools.bench_cfg import make_cfg
    il._backend[0] = emul_ops
    try:
        J, D = 4, 16
        cfg = make_cfg(num_layers=18, num_joints=J, volume=True, depth_res=D, image_size=(64, 64))
        grads = []
        for use_sink in (True, False):
            torch.manual_seed(0)
            m = models.pose3d_resnet.get_pose_net(cfg, False, precision="f16x3")
            m._ops = emul_ops
            m.train()
            assert getattr(m(torch.randn(2, 3, 64, 64)), "_epb_logit_sink", None) is None   # opt-in only
            m.fused_head_gradient = True        # what lib/core/function.py sets around its forward
            out = m(torch.randn(2, 3, 64, 64))
            sink = getattr(out, "_epb_logit_sink", None)
            assert sink is not None and type(m._engine()).__name__ == "Engine16"
            if not use_sink:
                del out._epb_logit_sink
            lab, wt = torch.rand(2, J * 3) - 0.5, torch.ones(2, J * 3)
            loss = il.L1JointLocationLoss(J)(out, lab, wt)
            if extra_consumer:
                loss = loss + 1e-3 * (out * out).mean()
            loss.backward()
            assert sink.filled == use_sink
            grads.append({n: p.grad.clone() for n, p in m.named_parameters()})
        worst = max(float((grads[0][k] - grads[1][k]).abs().max() / (grads[1][k].abs().max() + 1e-30))
                    for k in grads[0])
        assert worst <= 5e-6, worst
    finally:
        il._backend[0] = __import__("epipolarpose_b200.ops", fromlist=["ops"])
