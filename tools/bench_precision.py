#!/usr/bin/env python
"""Step time of the bench workload under several MODEL.PRECISION values, in ONE process.

The workload is bench.py's C4 step: PoseResNet-50 (VOLUME, J16 D64), 32 view-tuples x 4 views of
256x256 per GPU, forward -> soft-argmax -> iterative-LS online triangulation -> SmoothL1 ->
backward -> fused Adam, replayed as one CUDA graph (lib.core.function.GraphedTrainStep).  One
model per precision is built and warmed up (eager step, capture, replays); then the precisions
are timed in alternation over --rounds rounds of --steps steps each with CUDA events, so clock
and neighbour drift hits all of them alike.  Prints one JSON line: ms/step of every round, the
memory each precision's model + captured step added (peak allocated), and the card's name and
power limit read in the same run.

    python tools/bench_precision.py [--precisions f16x3,f16,tf32] [--rounds 3] [--steps 50]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "epipolarpose_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

TUPLES, VIEWS, HW, J, D, LAYERS = 32, 4, 256, 16, 64, 50


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                        "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power, clk = (q.stdout.strip().split(", ") + [None] * 3)[:3] if q.returncode == 0 else \
        (torch.cuda.get_device_name(), None, None)
    return {"name": name, "power_limit": power, "sm_max_clock": clk}


def meta_and_batches(dev, tuples):
    """bench.py's synthetic batch (rank 0): ring cameras, boxes, two alternating image batches."""
    from lib.dataset.synthetic import ring_camera
    n_img = tuples * VIEWS
    rng = np.random.default_rng(1000)
    order = [(t, 0) for t in range(tuples)] + [(t, 3) for t in range(tuples)] + \
            [(t, 1) for t in range(tuples)] + [(t, 2) for t in range(tuples)]
    cams = {(t, v): ring_camera(rng, v) for t in range(tuples) for v in range(VIEWS)}
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
    g = torch.Generator().manual_seed(1000)
    batches = [torch.randn(n_img, 3, HW, HW, generator=g).to(dev) for _ in range(2)]
    return {k: v.to(dev) for k, v in meta.items()}, batches


def build_step(precision, dev):
    import lib.models as models
    import lib.core.integral_loss as il
    import lib.utils.utils as U
    import lib.core.function as fn
    from tools.bench_cfg import make_cfg
    cfg = make_cfg(num_layers=LAYERS, num_joints=J, volume=True, depth_res=D, image_size=(HW, HW))
    torch.manual_seed(0)
    model = models.pose3d_resnet.get_pose_net(cfg, False, precision=precision).to(dev).train()
    opt = U.FusedAdam(list(model.parameters()), lr=1e-3)
    stepper = fn.GraphedTrainStep(model, il.SmoothL1JointLocationLoss(J).to(dev), opt, online=True,
                                  method="iterative")
    return model, stepper


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--precisions", default="f16x3,f16,tf32")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--tuples", type=int, default=TUPLES)
    args = ap.parse_args()
    if args.rounds < 1 or args.steps < 1 or args.warmup < 3:
        ap.error("--rounds and --steps must be >= 1, --warmup >= 3 (eager step, capture, replay)")
    from epipolarpose_b200 import ops
    ops.device_check()
    dev = torch.device("cuda", torch.cuda.current_device())
    precs = args.precisions.split(",")
    meta, batches = meta_and_batches(dev, args.tuples)
    steps, engines, mem = {}, {}, {}
    for p in precs:
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        model, stepper = build_step(p, dev)
        for i in range(args.warmup):
            stepper(batches[i % 2], meta=meta)
        torch.cuda.synchronize()
        mem[p] = round((torch.cuda.max_memory_allocated() - base) / 2 ** 30, 2)
        eng = model._engine()
        engines[p] = "%s(planes=%d)" % (type(eng).__name__, eng.planes) if hasattr(eng, "planes") else \
            "%s(precision=%d)" % (type(eng).__name__, eng.precision)
        steps[p] = stepper
    rounds = {p: [] for p in precs}
    for r in range(args.rounds):
        for p in precs[r % len(precs):] + precs[:r % len(precs)]:       # rotate the order per round
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for i in range(args.steps):
                loss = steps[p](batches[i % 2], meta=meta)
            e1.record()
            torch.cuda.synchronize()
            assert torch.isfinite(loss).all(), p
            rounds[p].append(round(e0.elapsed_time(e1) / args.steps, 3))
    out = {"workload": "C4: R%d pose3d_resnet VOLUME J%d D%d, %d tuples x %d views of %dx%d, graphed "
                       "online-triangulation step (bench.py)" % (LAYERS, J, D, args.tuples, VIEWS, HW, HW),
           "card": card(), "rounds": args.rounds, "steps_per_round": args.steps,
           "ms_per_step": rounds, "median_ms_per_step": {p: float(np.median(v)) for p, v in rounds.items()},
           "peak_mem_gib": mem, "engine": engines,
           "timing": "CUDA events around --steps graph replays per precision and round, alternating; "
                     "peak_mem_gib = max allocated while building + warming up that precision, minus "
                     "what was allocated before"}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
