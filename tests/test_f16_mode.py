"""Host-side selection of the single-pass fp16 mode (MODEL.PRECISION: f16): the yaml value parses
and picks the split engine with one plane; a plan the split engine does not take falls back to
the single-pass TF32 engine, as f16x3 falls back to 3xTF32.  No GPU: the engines are only built."""
import os

import pytest

from oracle import refshim
from tests import emul_ops


@pytest.fixture
def no_env_precision(monkeypatch):
    monkeypatch.delenv("EPB_PRECISION", raising=False)


def test_yaml_precision_f16_selects_one_plane_engine16(tmp_path, no_env_precision):
    import lib.models as models
    from lib.core import config as C
    from epipolarpose_b200 import net16
    path = os.path.join(str(tmp_path), "f16.yaml")
    with open(path, "w") as f:
        f.write("MODEL:\n  PRECISION: f16\n  NUM_JOINTS: 16\n  IMAGE_SIZE: [256, 256]\n")
    try:
        C.update_config(path)
        assert C.config.MODEL.PRECISION == "f16"
        m = models.pose3d_resnet.get_pose_net(C.config, False, ops=emul_ops)
        eng = m._engine()
        assert isinstance(eng, net16.Engine16)
        assert eng.planes == 1
        assert eng.precision == 1 and eng.tc_precision == 1     # fp32-operand layers: single-pass TF32
    finally:
        C.reset_config()


def test_keyword_and_environment_select_f16(monkeypatch):
    import lib.models as models
    from epipolarpose_b200 import net16
    cfg = refshim.make_cfg(num_layers=18, num_joints=4, volume=True, depth_res=16, image_size=(64, 64))
    monkeypatch.delenv("EPB_PRECISION", raising=False)
    eng = models.pose3d_resnet.get_pose_net(cfg, False, ops=emul_ops, precision="f16")._engine()
    assert isinstance(eng, net16.Engine16) and eng.planes == 1
    eng = models.pose3d_resnet.get_pose_net(cfg, False, ops=emul_ops, precision="f16x3")._engine()
    assert isinstance(eng, net16.Engine16) and eng.planes == 2 and eng.precision == 3
    monkeypatch.setenv("EPB_PRECISION", "f16")
    eng = models.pose3d_resnet.get_pose_net(cfg, False, ops=emul_ops)._engine()
    assert isinstance(eng, net16.Engine16) and eng.planes == 1


def test_f16_falls_back_to_single_pass_tf32_when_channels_do_not_fit(no_env_precision):
    import lib.models as models
    from epipolarpose_b200 import net, net16
    cfg = refshim.make_cfg(num_layers=18, num_joints=3, volume=True, depth_res=8, image_size=(64, 64))
    cfg.MODEL.EXTRA.NUM_DECONV_FILTERS = [96, 96, 96]      # not whole 64-channel TMA boxes
    m = models.pose3d_resnet.get_pose_net(cfg, False, ops=emul_ops, precision="f16")
    eng = m._engine()
    assert isinstance(eng, net.Engine) and not isinstance(eng, net16.Engine16)
    assert eng.precision == 1


def test_engine16_rejects_other_plane_counts():
    from epipolarpose_b200 import net, net16
    plan = net.PoseNetPlan(18, 3, True, 8, (64, 64))
    with pytest.raises(ValueError):
        net16.Engine16(plan, ops=emul_ops, planes=3)
