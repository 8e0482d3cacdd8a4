#!/usr/bin/env python
"""Benchmark of the EpipolarPose training-loop hot path on B200.

Workload (BASELINE.json metric "multi-view samples/sec (4-view 256x256, bs32)"):
one STEP = one self-supervised training iteration over a per-GPU batch of 32
view-tuples x 4 views = 128 images of 256x256 (SURVEY.md section 8(d) config C4):
  PoseResNet-50 (VOLUME, 16 joints x 64 depth bins -> 1024 x 64 x 64 logits)
  forward -> soft-argmax -> patch->image affine -> two-view iterative-LS
  triangulation (pairs (0,1),(3,2)) -> re-projection to labels -> SmoothL1
  integral loss -> backward (dgrad + wgrad, BN) -> fused Adam
  (+ one NCCL all-reduce of the flat gradient when N > 1).
`value` = view-tuples/s with the step's inputs resident in HBM; `e2e` = the same
through the reference-shaped public API (lib.core.function.train_integral) with
pinned HOST batches, H2D copies and a loss read-back inside the timed region.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

--impl reference times the reference's CPU implementation of the same step
(oracle port: torch-CPU fp32 network + numpy/OpenCV-equivalent geometry) on the
box's host cores on a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "epipolarpose_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

TUPLES, VIEWS, HW, J, D = 32, 4, 256, 16, 64
WORKLOAD_TAG = "C4"
METRIC = "multi-view samples/sec (4-view 256x256, bs32)"
UNIT = "view-tuples/s"


def workload_name(layers=50):
    return ("%s: R%d pose3d_resnet VOLUME J%d D%d, %d tuples x %d views of %dx%d per GPU, " % (WORKLOAD_TAG, layers, J, D, TUPLES, VIEWS, HW, HW) +
            "self-supervised step (fwd, soft-argmax, iterative-LS triangulation, SmoothL1, bwd, Adam)")


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# ---------------------------------------------------------------------------- data
def conv_flops(plan, n_img, hw):
    """Algorithmic conv FLOPs of one training step (fwd + dgrad + wgrad; no dgrad
    for the stem), true channel counts: 2*M*K*N per GEMM."""
    fwd = 0
    first = None
    h = w = hw
    def f(conv, h, w):
        ho, wo = conv.out_hw(h, w)
        if conv.kind == "conv":
            m = ho * wo
        else:
            m = h * w          # each input pixel meets k*k taps
        return 2 * m * conv.k * conv.k * conv.cin * conv.cout, ho, wo
    fl, h, w = f(plan.stem, h, w)
    first = fl
    fwd += fl
    h, w = (h + 2 - 3) // 2 + 1, (w + 2 - 3) // 2 + 1
    for blk in plan.blocks:
        hh, ww = h, w
        for conv in blk["convs"]:
            fl, hh, ww = f(conv, hh, ww)
            fwd += fl
        if blk["down"]:
            fwd += f(blk["down"][0], h, w)[0]
        h, w = hh, ww
    for conv, _ in plan.deconvs:
        fl, h, w = f(conv, h, w)
        fwd += fl
    fwd += f(plan.final, h, w)[0]
    return n_img * (3 * fwd - first), n_img * fwd


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons with nvidia-smi during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False
        self.proc = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                 "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass
        sm, mx, reasons = [], 0.0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                    "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


DUMP_SAMPLE = 4_000_000      # float32 values of the model state kept by --dump-outputs (16 MB)


def dump_outputs(out_dir, loss, model):
    """What the last timed step handed its caller, as float32 .npy files in out_dir:
    loss.npy (the returned loss), final_layer.{weight,bias}.npy (the updated head in full)
    and state_sample.npy: a fixed sample (seed 0, sorted indices) of every floating-point
    state_dict entry -- parameters after the Adam update and BatchNorm running statistics --
    flattened and concatenated in state_dict order."""
    os.makedirs(out_dir, exist_ok=True)
    sd = model.state_dict()
    out = {"loss": loss.detach().float().reshape(1),
           "final_layer.weight": sd["final_layer.weight"], "final_layer.bias": sd["final_layer.bias"]}
    flat = torch.cat([v.detach().reshape(-1).float() for v in sd.values() if v.is_floating_point()])
    n = min(DUMP_SAMPLE, flat.numel())
    idx = np.sort(np.random.default_rng(0).choice(flat.numel(), n, replace=False))
    out["state_sample"] = flat[torch.from_numpy(idx).to(flat.device)]
    for name, v in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), v.detach().float().cpu().numpy())


# ---------------------------------------------------------------------------- GPU arm
def run_gpu(args):
    import torch.distributed as dist
    from epipolarpose_b200 import ops
    from tools.bench_cfg import make_cfg
    import lib.models as models
    import lib.core.integral_loss as il
    import lib.utils.img_utils as iu
    import lib.utils.utils as U
    import lib.core.function as fn
    from lib.core.config import config as gcfg, reset_config
    from lib.dataset.synthetic import ring_camera

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    ops.device_check()

    layers = args.layers
    cfg = make_cfg(num_layers=layers, num_joints=J, volume=True, depth_res=D,
                           image_size=(HW, HW))
    torch.manual_seed(0)                               # identical weights on every rank
    model = models.pose3d_resnet.get_pose_net(cfg, False, precision=args.precision)
    model = model.to(dev).train()
    criterion = il.SmoothL1JointLocationLoss(J).to(dev)
    opt = U.FusedAdam(list(model.parameters()), lr=1e-3)
    n_img = args.tuples * VIEWS

    # synthetic batch (rank-seeded): images + per-sample cameras / boxes
    rng = np.random.default_rng(1000 + rank)
    order = [(t, 0) for t in range(args.tuples)] + [(t, 3) for t in range(args.tuples)] + \
            [(t, 1) for t in range(args.tuples)] + [(t, 2) for t in range(args.tuples)]
    cams = {(t, v): ring_camera(rng, v) for t in range(args.tuples) for v in range(VIEWS)}
    meta = {"center_x": torch.tensor(500 + rng.uniform(-50, 50, n_img)),
            "center_y": torch.tensor(500 + rng.uniform(-50, 50, n_img)),
            "width": torch.tensor(800 + rng.uniform(-100, 100, n_img)),
            "height": torch.tensor(800 + rng.uniform(-100, 100, n_img)),
            "scale": torch.ones(n_img, dtype=torch.float64),
            "rot": torch.zeros(n_img, dtype=torch.float64),
            "R": torch.tensor(np.stack([cams[o][0] for o in order])),
            "T": torch.tensor(np.stack([cams[o][1] for o in order])),
            "f": torch.tensor(np.stack([cams[o][2] for o in order])),
            "c": torch.tensor(np.stack([cams[o][3] for o in order])),
            "projection_matrix": torch.tensor(np.stack([cams[o][4] for o in order]))}
    meta_dev = {k: v.to(dev) for k, v in meta.items()}
    g = torch.Generator().manual_seed(1000 + rank)
    host_batches = [torch.randn(n_img, 3, HW, HW, generator=g).pin_memory() for _ in range(2)]
    dev_batches = [b.to(dev) for b in host_batches]
    dummy_lab = torch.zeros(n_img, J * 3)

    conv_t = {"events": []}
    # the step, as the public loop runs it: CUDA-graph replay of forward / epipolar labels /
    # loss / backward (+ all-reduce) / Adam (lib.core.function.GraphedTrainStep)
    stepper = fn.GraphedTrainStep(model, criterion, opt, online=True, method="iterative")
    use_graph = not args.no_graph

    def step(x):
        if use_graph:
            return stepper(x, meta=meta_dev)
        return stepper.eager_step(x, None, None, iu.pack_meta(meta_dev, n_img, dev))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()          # nvidia-smi needs ~1 s to emit its first sample: start it
        time.sleep(1.0)          # before the (identical-load) warm-up steps
    for i in range(args.warmup):
        step(dev_batches[i % 2])
    barrier()
    if rank == 0:
        sampler.rows = []        # keep only samples taken from here on (timed region)
    l0 = ops.launches
    barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    h0 = time.perf_counter()
    for i in range(args.steps):
        loss = step(dev_batches[i % 2])       # 2 x 100 MB inputs + >25 GB activations >> 126 MB L2
    host_enqueue_ms = (time.perf_counter() - h0) * 1e3 / args.steps
    t1.record()
    barrier()
    ms = t0.elapsed_time(t1)
    clocks = sampler.finish() if rank == 0 else None
    if world > 1:
        tmax = torch.tensor([ms], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms = tmax.item()
    ms_step = ms / args.steps
    value = world * args.tuples / (ms_step / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, model)    # before the eager steps below move the weights

    # ---- dominant kernel family (conv GEMMs): CUDA events around every launch of the same
    # step, issued eagerly right after the timed region (events cannot be read back from
    # inside a replayed graph); the kernels and their arguments are identical
    orig_call = ops._call
    engine_kind = type(model._engine()).__name__
    ns = {"fp32": 0, "tf32": 1, "tf32x3": 3, "f16x3": 3}[args.precision]

    def kernel_class(name, g):
        """Name of the kernel template the C dispatcher picks for this call (csrc/conv*.cu)."""
        if name == "epb_conv16_fprop":
            if g.Cout <= 64:
                bn = 64
            elif g.Cout <= 128:
                bn = 128
            else:
                p256, p128 = (g.Cout + 255) // 256 * 256, (g.Cout + 127) // 128 * 128
                bn = 128 if p256 * 4 > p128 * 5 else 256
            return "conv16_kernel<%d>" % bn
        if name == "epb_conv16_wgrad":
            return "wgrad16_kernel<%d>" % (128 if g.Cout <= 128 else 256)
        kind = "fprop" if name == "epb_conv_fprop" else "wgrad"
        if ns == 0 or g.Cin % 32 or (kind == "fprop" and g.Cout % 32):
            return "conv_%s_simt" % kind
        if kind == "fprop":
            bn = 256 if g.Cout >= 256 else (128 if g.Cout >= 128 else 64)
            # wide tiles over more than one M tile run on CTA pairs (csrc/conv_tc.cu:epb_conv_fprop_tc)
            pair = bn == 256 and g.N * g.Hp * g.Wp > 128 and os.environ.get("EPB_CTA_PAIR", "1") != "0"
            return "conv_fprop_tc_%skernel<%d,%d>" % ("pair_" if pair else "", bn, ns)
        bn = 128 if g.Cin >= 128 else (64 if g.Cin >= 64 else 32)
        return "conv_wgrad_tc_kernel<%d,%d>" % (bn, g.precision if g.precision else ns)

    CONV_CALLS = ("epb_conv_fprop", "epb_conv_wgrad", "epb_conv16_fprop", "epb_conv16_wgrad")
    other_t = {}

    def timed_call(name, *a):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()                       # torch's CURRENT stream = the one the kernel uses
        orig_call(name, *a)
        e1.record()
        if name in CONV_CALLS:
            g = a[0]._obj
            flops = 2.0 * g.N * g.Hp * g.Wp * g.Cin * g.Cout * g.T
            conv_t["events"].append((e0, e1, kernel_class(name, g), flops))
        else:
            other_t.setdefault(name, []).append((e0, e1))

    geom_dev = iu.pack_meta(meta_dev, n_img, dev)
    os.environ["EPB_OVERLAP_WGRAD"] = "0"      # serialise wgrad with the rest: clean per-kernel times
    ops._call = timed_call
    l0 = ops.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    n_inst = min(args.steps, 3)
    for i in range(n_inst):
        stepper.eager_step(dev_batches[i % 2], None, None, geom_dev)   # waits / is waited on
    e1.record()                                                       # by the current stream
    barrier()
    launches = (ops.launches - l0) // n_inst
    eager_ms = e0.elapsed_time(e1) / n_inst
    conv_ms = sum(a.elapsed_time(b) for a, b, _, _ in conv_t["events"]) / n_inst
    n_conv_launch = len(conv_t["events"]) // n_inst
    per_class = {}
    for a, b, name, fl in conv_t["events"]:
        c = per_class.setdefault(name, [0, 0.0, 0.0])
        c[0] += 1
        c[1] += a.elapsed_time(b)
        c[2] += fl
    dom = max(per_class, key=lambda k: per_class[k][1])
    ops._call = orig_call
    other_ms = {k: round(sum(a.elapsed_time(b) for a, b in v) / n_inst, 3) for k, v in other_t.items()}
    os.environ.pop("EPB_OVERLAP_WGRAD", None)

    # ---- e2e through the public loop API with HOST batches (H2D + loss read-back)
    reset_config()
    gcfg.PRINT_FREQ = 1
    gcfg.TRAIN.ONLINE_TRIANGULATION = True
    gcfg.TRAIN.TRIANGULATION_METHOD = "iterative"
    gcfg.TRAIN.CUDA_GRAPH = use_graph
    import logging
    logging.getLogger("lib.core.function").setLevel(logging.WARNING)
    logging.getLogger("epipolarpose_b200.lib.core.function").setLevel(logging.WARNING)

    model._epb_graphed_step = stepper      # the loop reuses the graph captured above

    class Loader(list):
        dataset = None
    def loader(n):
        return Loader([(host_batches[i % 2], dummy_lab, dummy_lab, meta) for i in range(n)])
    fn.train_integral(gcfg, loader(1), model, criterion, opt, 0)
    barrier()
    w0 = time.perf_counter()
    fn.train_integral(gcfg, loader(args.steps), model, criterion, opt, 0)
    barrier()
    e2e_s = time.perf_counter() - w0
    if world > 1:
        tmax = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        e2e_s = tmax.item()
    e2e_value = world * args.tuples * args.steps / e2e_s

    def finish():
        # tear-down of NCCL communicators that are referenced by a live CUDA graph can
        # block at interpreter exit: flush and leave without running destructors
        sys.stdout.flush()
        sys.stderr.flush()
        torch.cuda.synchronize()
        if world > 1:
            os._exit(0)

    if rank != 0:
        finish()
        return
    peaks, which = measured_peaks()
    total_flops, _ = conv_flops(model._plan, n_img, HW)
    f16 = args.precision == "f16x3" and engine_kind == "Engine16"
    tf32_peak = peaks["bf16_tflops_sustained"] / 2.0        # TF32 rate = half the bf16 rate
    tensor_peak = peaks["bf16_tflops_sustained"] if f16 else tf32_peak   # peak of the tcgen05 kind used
    fam_achieved = total_flops / (conv_ms / 1e3) / 1e12 if conv_ms > 0 else 0.0
    d_n, d_ms, d_fl = per_class[dom]
    achieved = d_fl / (d_ms / 1e3) / 1e12        # padded-channel FLOPs of the dominant kernel's calls
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            traffic = json.load(f).get(dom)
    out = {
        "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_step, 3),
        "higher_is_better": True, "scaling": "strong" if args.strong else "weak", "vs_baseline": None,
        "dtype": {"fp32": "f32 (CUDA-core FFMA)", "tf32": "tf32 (tcgen05, f32 accumulate)",
                  "tf32x3": "tf32x3 (3-pass error-compensated tcgen05, f32 accumulate; f32 SIMT "
                            "where the tensor path does not take the shape)",
                  "f16x3": "f16x3 (fp32 operands split into two fp16 planes, 3-pass error-compensated "
                           "tcgen05 kind::f16, f32 accumulate: fp32-grade results)"}[args.precision],
        "data": "synthetic",
        "config": {"workload": workload_name(layers), "tuples_per_gpu": args.tuples,
                   "images_per_gpu": n_img, "parallelism": "dp%d" % world,
                   "l2_policy": "inputs+activations >> L2 (2 alternating 100 MB batches, >25 GB "
                                "activations per step); no explicit flush"},
        "clocks": clocks,
        "e2e": {"value": round(e2e_value, 3), "unit": UNIT,
                "h2d_bytes_per_step": int(host_batches[0].numel() * 4),
                "d2h_bytes_per_step": 4},
        "gpu_launches": int(launches) * args.steps, "gpu_launches_per_step": int(launches),
        "host_enqueue_ms_per_step": round(host_enqueue_ms, 2),
        "cuda_graph": bool(use_graph),
        "roofline": {"bound": "tensor", "kernel": dom,
                     "achieved": round(achieved, 3), "peak": round(tensor_peak, 1),
                     "unit": "TFLOP/s", "frac": round(achieved / tensor_peak, 5),
                     "traffic": traffic,
                     "peak_source": which + (" bf16_tflops_sustained (kind::f16)" if f16 else
                                             " bf16_tflops_sustained / 2 (tf32)"),
                     "note": "achieved counts algorithmic FLOPs (2MNK once); the 3-pass split executes "
                             "3x that on the tensor pipe (executed_frac); frac_vs_tf32_peak is the "
                             "round-1 denominator (tf32 rate) for comparison",
                     "executed_frac": round(3 * achieved / tensor_peak, 5) if ns == 3 else round(achieved / tensor_peak, 5),
                     "frac_vs_tf32_peak": round(achieved / tf32_peak, 5),
                     "whole_step": {"algorithmic_tflops": round(total_flops / (ms_step / 1e3) / 1e12, 2),
                                    "mfu_vs_kind_peak": round(total_flops / (ms_step / 1e3) / 1e12 / tensor_peak, 5),
                                    "mfu_vs_tf32_peak": round(total_flops / (ms_step / 1e3) / 1e12 / tf32_peak, 5)},
                     "non_conv_ms_per_step": other_ms,
                     "launches_per_step": d_n // n_inst,
                     "avg_launch_ms": round(d_ms / d_n, 4),
                     "share_of_step": round(d_ms / n_inst / ms_step, 4) if ms_step > 0 else None,
                     "conv_family": {"achieved": round(fam_achieved, 3), "launches_per_step": n_conv_launch,
                                     "share_of_step": round(conv_ms / ms_step, 4),
                                     "per_kernel_ms_per_step": {k: round(v[1] / n_inst, 3)
                                                                for k, v in sorted(per_class.items())}},
                     "measured": "CUDA events around each launch of %d eager step(s) run right "
                                 "after the timed region (eager step %.2f ms)" % (n_inst, eager_ms)},
    }
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_reference(steps=1, warmup=1, tuples=args.cpu_tuples, layers=layers)
    print(json.dumps(out))
    finish()


# ---------------------------------------------------------------------------- CPU arm
def pick_cpu_threads():
    """torch-CPU convolutions do not scale to every hardware thread of the box
    (128 threads were 100x SLOWER than 16 on the B200 hosts): time a small
    forward at a few thread counts and give the reference arm the fastest."""
    from oracle import restate_net
    ncpu = os.cpu_count() or 1
    sd = restate_net.init_state(restate_net.param_shapes(18, 2, True, 8), 0)
    x = torch.randn(4, 3, 128, 128)
    best, best_t = 1, float("inf")
    for th in sorted({min(ncpu, c) for c in (8, 16, 32, 64)}):
        torch.set_num_threads(th)
        with torch.no_grad():
            restate_net.forward(sd, x, num_layers=18, training=True)
            t0 = time.perf_counter()
            restate_net.forward(sd, x, num_layers=18, training=True)
            dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = th, dt
    return best


def cpu_reference(steps, warmup, tuples, layers=50):
    """The reference's CPU implementation of the step, restated (oracle port):
    torch-CPU fp32 PoseResNet fwd/bwd + Adam on all host threads, float64
    numpy geometry single-threaded as in the reference's Python loops."""
    from oracle import restate, restate_net
    from lib.dataset.synthetic import ring_camera
    cores = pick_cpu_threads()
    torch.set_num_threads(cores)
    n_img = tuples * VIEWS
    shapes = restate_net.param_shapes(layers, J, True, D)
    sd = restate_net.init_state(shapes, 0, scale_final=0.001)
    params = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v)
              for k, v in sd.items()}
    opt = torch.optim.Adam([p for p in params.values() if p.requires_grad], lr=1e-3)
    rng = np.random.default_rng(1000)
    order = [(t, 0) for t in range(tuples)] + [(t, 3) for t in range(tuples)] + \
            [(t, 1) for t in range(tuples)] + [(t, 2) for t in range(tuples)]
    cams = {(t, v): ring_camera(rng, v) for t in range(tuples) for v in range(VIEWS)}
    meta = {"center_x": 500 + rng.uniform(-50, 50, n_img), "center_y": 500 + rng.uniform(-50, 50, n_img),
            "width": 800 + rng.uniform(-100, 100, n_img), "height": 800 + rng.uniform(-100, 100, n_img),
            "scale": np.ones(n_img), "rot": np.zeros(n_img),
            "R": np.stack([cams[o][0] for o in order]), "T": np.stack([cams[o][1] for o in order]),
            "f": np.stack([cams[o][2] for o in order]), "c": np.stack([cams[o][3] for o in order]),
            "projection_matrix": np.stack([cams[o][4] for o in order])}
    x = torch.randn(n_img, 3, HW, HW)

    def one():
        opt.zero_grad()
        out = restate_net.forward(params, x, num_layers=layers, training=True, new_stats={})
        sm = torch.softmax(out.reshape(n_img, J, -1), 2).reshape(n_img, J, D, D, D)
        ar = torch.arange(D, dtype=torch.float32)
        c = torch.stack([(sm.sum((2, 3)) * ar).sum(2) / D - 0.5, (sm.sum((2, 4)) * ar).sum(2) / D - 0.5,
                         (sm.sum((3, 4)) * ar).sum(2) / D - 0.5], 2).reshape(n_img, J * 3)
        label, weight, _, _ = restate.self_supervision(c.detach().numpy(), meta, "iterative")
        d = c - torch.from_numpy(label)
        a = d.abs()
        loss = (torch.where(a < 1, 0.5 * d * d, a - 0.5) * torch.from_numpy(weight)).sum() / n_img
        loss.backward()
        opt.step()
        return loss.item()

    for _ in range(warmup):
        one()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    model_name, phys = "unknown", None
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.lower().startswith("model name"):
                    model_name = line.split(":", 1)[1].strip()
                    break
        import psutil
        phys = psutil.cpu_count(logical=False)
    except Exception:
        pass
    return {"value": round(tuples / dt, 4), "unit": UNIT, "cores": cores, "kind": "port",
            "cpu_model": model_name, "physical_cores": phys, "logical_cores": os.cpu_count(),
            "threads_used": cores,
            "sample": "%d step(s) of %d view-tuples (%d images) of the same workload, R%d, "
                      "%.1f s/step; cv2.solve restated with numpy.linalg, cv2.getAffineTransform as its 6x6 LU"
                      % (steps, tuples, n_img, layers, dt),
            "s_per_step": round(dt, 3)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    base = cpu_reference(steps=max(1, min(args.steps, 2)), warmup=min(args.warmup, 1),
                         tuples=args.cpu_tuples, layers=args.layers)
    out = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": UNIT,
           "n_gpus": world, "steps": max(1, min(args.steps, 2)), "warmup": min(args.warmup, 1),
           "ms_per_step": round(base["s_per_step"] * 1e3, 1), "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32 (CPU) / f64 geometry",
           "data": "synthetic",
           "config": {"workload": workload_name(args.layers), "bounded_sample": base["sample"]},
           "cpu_baseline": base,
           "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0,
                   "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


def main():
    global TUPLES, HW, J, D, WORKLOAD_TAG
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("EPB_PRECISION", "f16x3"),
                    choices=["fp32", "tf32", "tf32x3", "f16x3"])
    ap.add_argument("--layers", type=int, default=50)
    ap.add_argument("--tuples", type=int, default=TUPLES, help="view-tuples per GPU per step")
    ap.add_argument("--cpu-tuples", type=int, default=8, help="bounded CPU sample size (view-tuples)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="issue every kernel eagerly")
    ap.add_argument("--workload", default="c4", choices=["c4", "c5"],
                    help="c4 (default, the BASELINE metric config): R50 256x256 J16 D64, 32 tuples/GPU; "
                         "c5 (extra line, not the headline): R101 384x384 J17 D96, 16 tuples/GPU")
    ap.add_argument("--strong", action="store_true",
                    help="strong scaling: the tuples of ONE GPU's batch are divided among the ranks")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the loss and model state of the last one to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.workload == "c5":
        HW, J, D, WORKLOAD_TAG = 384, 17, 96, "C5"
        args.layers = 101
        if args.tuples == 32:
            args.tuples = 16
    if args.strong:
        world = int(os.environ.get("WORLD_SIZE", "1"))
        assert args.tuples % world == 0, "tuples must divide among the ranks"
        args.tuples //= world
    TUPLES = args.tuples
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
