"""The drop-in claim as a test: a training script that drives the mirror through the same
calls as the upstream EpipolarPose scripts/train.py (:66-188) -- update_config,
create_logger, get_pose_net, DataParallel, criterion / dataset looked up by name,
get_optimizer + MultiStepLR, train / validate / eval per epoch, checkpoints, final state --
runs one epoch with DATASET.DATASET: synthetic_h36m and reproduces what the UNMODIFIED
upstream script computed over the same mirror (tests/golden/make_golden_dropin.py):
the logged losses, the evaluation result and a fixed sample of the final state.  A scratch
tree is laid out as INTEGRATION.md section 1 says (<tmp>/lib -> epipolarpose_b200/lib).
The C ABI is replaced by its CPU emulation (tests/emul_ops.py) from a sitecustomize hook
that touches neither the script nor the mirror; `.cuda()` is a no-op there.
tests/test_gpu_parity.py::test_reference_script_flow replays the same call sequence on the
device."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.conftest import ROOT

YAML = """\
GPUS: '0'
DATA_DIR: ''
OUTPUT_DIR: '{out}'
LOG_DIR: '{out}/log'
WORKERS: 0
PRINT_FREQ: 1
EXP_NAME: dropin
DATASET:
  DATASET: synthetic_h36m
  ROOT: ''
  TRAIN_SET: train
  TEST_SET: valid
  SYNTHETIC_LEN: 8
MODEL:
  NAME: pose3d_resnet
  INIT_WEIGHTS: false
  PRETRAINED: ''
  IMAGE_SIZE: [64, 64]
  NUM_JOINTS: 4
  DEPTH_RES: 16
  VOLUME: true
  EXTRA:
    NUM_LAYERS: 18
    NUM_DECONV_LAYERS: 3
    NUM_DECONV_FILTERS: [256, 256, 256]
    NUM_DECONV_KERNELS: [4, 4, 4]
    FINAL_CONV_KERNEL: 1
    DECONV_WITH_BIAS: false
LOSS:
  FN: L1JointLocationLoss
  NORM: false
TRAIN:
  BATCH_SIZE: 4
  SHUFFLE: false
  BEGIN_EPOCH: 0
  END_EPOCH: 1
  OPTIMIZER: adam
  LR: 0.001
  LR_FACTOR: 0.1
  LR_STEP: [1]
  ONLINE_TRIANGULATION: false
TEST:
  BATCH_SIZE: 4
"""

SITECUSTOMIZE = """\
# test-only: route the C ABI to its CPU emulation and make .cuda() a no-op (no GPU here)
import sys
sys.path.insert(0, {root!r})
import torch
torch.nn.Module.cuda = lambda self, *a, **k: self
torch.Tensor.cuda = lambda self, *a, **k: self
import epipolarpose_b200.ops as _o
from tests import emul_ops as _e
for _n in dir(_e):
    if not _n.startswith("_") and callable(getattr(_e, _n)):
        setattr(_o, _n, getattr(_e, _n))
sys.path.insert(0, {tree!r})
import lib.core.integral_loss, lib.core.inference, lib.utils.img_utils, lib.utils.triangulation
import lib.dataset.h36m_eval, lib.utils.utils
for _mod in (lib.core.integral_loss, lib.core.inference, lib.utils.img_utils, lib.utils.triangulation,
             lib.dataset.h36m_eval, lib.utils.utils):
    _mod._backend[0] = _e                      # the mirrors' own test hook
import lib.models.pose3d_resnet as _m
_init = _m.PoseResNet.__init__
def _patched(self, *a, **k):
    k.setdefault("ops", _e)
    _init(self, *a, **k)
_m.PoseResNet.__init__ = _patched
# seeded weight initialisation, so that two runs of the script can be compared
import random, numpy
random.seed(0)
numpy.random.seed(0)
torch.manual_seed(0)
"""

# What a user's training script does with the mirror: the calls of the upstream
# scripts/train.py, in its order (the learning-rate schedule steps before each epoch there).
TRAIN_SCRIPT = """\
import argparse
import os
import sys
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import torch
import torch.utils.data
import lib.core.integral_loss as loss
import lib.dataset as dataset
import lib.models as models
from lib.core.config import config, update_config, get_model_name
from lib.core.function import train_integral, validate_integral, eval_integral
from lib.utils.utils import get_optimizer, save_checkpoint, create_logger

ap = argparse.ArgumentParser()
ap.add_argument("--cfg", required=True)
ap.add_argument("--workers", type=int, default=8)
args = ap.parse_args()
update_config(args.cfg)
if args.workers:
    config.WORKERS = args.workers
logger, out_dir = create_logger(config, args.cfg, "train")
model = models.pose3d_resnet.get_pose_net(config, is_train=True)
gpus = [int(i) for i in config.GPUS.split(",")]
model = torch.nn.DataParallel(model, device_ids=gpus).cuda()
criterion = eval("loss." + config.LOSS.FN)(num_joints=config.MODEL.NUM_JOINTS, norm=config.LOSS.NORM).cuda()
optimizer = get_optimizer(config, model)
schedule = torch.optim.lr_scheduler.MultiStepLR(optimizer, config.TRAIN.LR_STEP, config.TRAIN.LR_FACTOR)
ds = eval("dataset." + config.DATASET.DATASET)
train_set = ds(cfg=config, root=config.DATASET.ROOT, image_set=config.DATASET.TRAIN_SET, is_train=True)
valid_set = ds(cfg=config, root=config.DATASET.ROOT, image_set=config.DATASET.TEST_SET, is_train=False)
train_loader = torch.utils.data.DataLoader(train_set, batch_size=config.TRAIN.BATCH_SIZE * len(gpus),
                                           shuffle=config.TRAIN.SHUFFLE, num_workers=config.WORKERS,
                                           pin_memory=True)
valid_loader = torch.utils.data.DataLoader(valid_set, batch_size=config.TEST.BATCH_SIZE * len(gpus),
                                           shuffle=False, num_workers=config.WORKERS, pin_memory=True)
best_perf = 0.0
for epoch in range(config.TRAIN.BEGIN_EPOCH, config.TRAIN.END_EPOCH):
    schedule.step()
    train_integral(config, train_loader, model, criterion, optimizer, epoch)
    preds = validate_integral(valid_loader, model)
    perf = 500. - eval_integral(epoch, preds, valid_loader, out_dir, debug=config.DEBUG.DEBUG)
    best = perf > best_perf
    best_perf = max(perf, best_perf)
    logger.info("=> saving checkpoint to {}".format(out_dir))
    save_checkpoint({"epoch": epoch + 1, "model": get_model_name(config), "state_dict": model.state_dict(),
                     "perf": perf, "optimizer": optimizer.state_dict()}, best, out_dir)
final = os.path.join(out_dir, "final_state.pth.tar")
logger.info("saving final model state to {}".format(final))
torch.save(model.module.state_dict(), final)
"""

SAMPLE = 20000        # final-state values compared with the upstream script's run


def run_train_script(tmp_path, scripts):
    """Run <scripts>/train.py over the mirror (CPU emulation, seeded) in a scratch tree;
    returns (log text, final state dict, checkpoint dict)."""
    tree = tmp_path / "tree"
    tree.mkdir()
    os.symlink(scripts, tree / "scripts")
    os.symlink(os.path.join(ROOT, "epipolarpose_b200", "lib"), tree / "lib")    # the mirror as `lib`
    out = tmp_path / "output"
    cfg = tmp_path / "dropin.yaml"
    cfg.write_text(YAML.format(out=str(out)))
    inject = tmp_path / "inject"
    inject.mkdir()
    (inject / "sitecustomize.py").write_text(SITECUSTOMIZE.format(root=ROOT, tree=str(tree)))
    # devices hidden: the emulation computes on the host, also on a machine with a GPU
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([str(inject), ROOT]), PYTHONDONTWRITEBYTECODE="1",
               CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, str(tree / "scripts" / "train.py"), "--cfg", str(cfg), "--workers", "0"],
                       cwd=str(tree), env=env, capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-4000:])
    finals = [os.path.join(d, f) for d, _, fs in os.walk(str(out)) for f in fs if f == "final_state.pth.tar"]
    assert len(finals) == 1
    ck = [os.path.join(d, f) for d, _, fs in os.walk(str(out)) for f in fs if f == "checkpoint.pth.tar"]
    assert len(ck) == 1
    return (r.stdout + r.stderr, torch.load(finals[0], map_location="cpu"),
            torch.load(ck[0], map_location="cpu", weights_only=False))


def summarize(log, state, checkpoint):
    """The arrays compared between runs: logged per-iteration losses, the evaluation's
    perf, the state_dict keys and a fixed sample (seed 0) of its floating-point values."""
    flat = torch.cat([v.reshape(-1).double() for v in state.values() if v.is_floating_point()]).numpy()
    idx = np.sort(np.random.default_rng(0).choice(flat.size, SAMPLE, replace=False))
    return {"losses": np.array([float(v) for v in re.findall(r"\tLoss ([-0-9.e+]+) \(", log)]),
            "perf": np.float64(checkpoint["perf"]), "keys": np.array(list(state)),
            "sample_idx": idx, "sample": flat[idx].astype(np.float32)}


def test_train_script_flow_matches_reference_run(golden, tmp_path):
    scripts = tmp_path / "scripts"
    scripts.mkdir()
    (scripts / "train.py").write_text(TRAIN_SCRIPT)
    log, state, checkpoint = run_train_script(tmp_path, str(scripts))
    assert "Epoch: [0][0/" in log and "Loss" in log            # train_integral's log line
    assert "saving final model state" in log
    assert "conv1.weight" in state and "final_layer.bias" in state
    assert all(torch.isfinite(v).all() for v in state.values() if v.is_floating_point())
    assert {"epoch", "state_dict", "perf", "optimizer"} <= set(checkpoint)
    g = golden("dropin_train")
    s = summarize(log, state, checkpoint)
    assert list(s["keys"]) == list(g["keys"])
    assert s["losses"].shape == g["losses"].shape and np.max(np.abs(s["losses"] - g["losses"])) <= 2e-5
    assert abs(float(s["perf"]) - float(g["perf"])) <= 1e-3 * abs(float(g["perf"]))
    assert np.array_equal(s["sample_idx"], g["sample_idx"])
    # another CPU may round a near-zero gradient to the other sign: Adam then moves that weight the
    # other way, by at most one learning rate (1e-4 after the schedule's first step) per step
    d = np.abs(s["sample"] - g["sample"])
    assert d.max() <= 5e-4 and np.mean(d <= 1e-5) >= 0.99
