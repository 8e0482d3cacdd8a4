"""Global experiment configuration -- host-side mirror of the reference's
lib/core/config.py surface (module-global `config`, `update_config`,
`update_dir`, `gen_config`, `get_model_name`), re-implemented without easydict
(absent here) and with yaml.safe_load (reference :173 uses the removed
yaml.load(f) form).  Field names / defaults follow reference config.py:8-139 so
the six experiments/*.yaml files parse unchanged; unknown keys raise
ValueError exactly like reference :167,184.

Extra keys (superset, all default-off): TRAIN.ONLINE_TRIANGULATION,
TRAIN.TRIANGULATION_METHOD, TRAIN.CUDA_GRAPH (default on), MODEL.PRECISION,
DATASET.SYNTHETIC_LEN.

MODEL.PRECISION (lib/models/pose3d_resnet.py; EPB_PRECISION overrides it): f16x3 (fp32-grade,
three fp16 tensor passes over hi/lo operand planes), f16 (one fp16 pass over the hi planes:
TF32-class operands, the fastest mode), tf32x3, tf32 (single pass), fp32.
"""
import os

import numpy as np
import yaml


class AttrDict(dict):
    """dict with attribute access; nested dicts are converted on assignment."""

    def __init__(self, d=None, **kw):
        super().__init__()
        for k, v in dict(d or {}, **kw).items():
            self[k] = v

    def __setitem__(self, k, v):
        if isinstance(v, dict) and not isinstance(v, AttrDict):
            v = AttrDict(v)
        super().__setitem__(k, v)

    def __setattr__(self, k, v):
        self[k] = v

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError:
            raise AttributeError(k)


_POSE_RESNET = dict(NUM_LAYERS=50, DECONV_WITH_BIAS=False, NUM_DECONV_LAYERS=3,
                    NUM_DECONV_FILTERS=[256, 256, 256], NUM_DECONV_KERNELS=[4, 4, 4],
                    FINAL_CONV_KERNEL=1, TARGET_TYPE='gaussian', HEATMAP_SIZE=[64, 64], SIGMA=2)

_DEFAULTS = dict(
    OUTPUT_DIR='', LOG_DIR='', DATA_DIR='', GPUS='0', WORKERS=8, PRINT_FREQ=20,
    EXP_NAME='default',
    CUDNN=dict(BENCHMARK=True, DETERMINISTIC=False, ENABLED=True),
    MODEL=dict(NAME='pose3d_resnet', INIT_WEIGHTS=True, PRETRAINED='', RESUME='', NUM_JOINTS=17,
               IMAGE_SIZE=[256, 256], DEPTH_RES=64, VOLUME=True, EXTRA=_POSE_RESNET,
               PRECISION='tf32x3'),
    LOSS=dict(USE_TARGET_WEIGHT=True, FN='L1JointLocationLoss', USE_SOFT=True, NORM=False,
              DEPTH_LAMBDA=1.),
    DATASET=dict(ROOT='', DATASET='mpii', TRAIN_SET='train', TEST_SET='valid', DATA_FORMAT='jpg',
                 HYBRID_JOINTS_TYPE='', SELECT_DATA=False, TRI=False, MPII_ORDER=False,
                 TRAIN_FRAME=32, VAL_FRAME=64, NUM_CAMS=4, DEPTH_RANGE=2000, FLIP=True,
                 SCALE_FACTOR=0.25, ROT_FACTOR=30, OCCLUSION=False, VOC='', BG_AUG=False,
                 Z_WEIGHT=1., SYNTHETIC_LEN=256),
    TRAIN=dict(LR_FACTOR=0.1, LR_STEP=[90, 110], LR=0.001, OPTIMIZER='adam', MOMENTUM=0.9,
               WD=0.0001, NESTEROV=False, GAMMA1=0.99, GAMMA2=0.0, BEGIN_EPOCH=0, END_EPOCH=140,
               RESUME=False, CHECKPOINT='', BATCH_SIZE=32, SHUFFLE=True,
               ONLINE_TRIANGULATION=False, TRIANGULATION_METHOD='iterative', CUDA_GRAPH=True),
    TEST=dict(BATCH_SIZE=32, FLIP_TEST=False, POST_PROCESS=True, SHIFT_HEATMAP=True,
              USE_GT_BBOX=False, OKS_THRE=0.5, IN_VIS_THRE=0.0, COCO_BBOX_FILE='', BBOX_THRE=1.0,
              MODEL_FILE='', IMAGE_THRE=0.0, NMS_THRE=1.0),
    DEBUG=dict(DEBUG=False, SAVE_BATCH_IMAGES_GT=False, SAVE_BATCH_IMAGES_PRED=False,
               SAVE_HEATMAPS_GT=False, SAVE_HEATMAPS_PRED=False, SAVE_3D=False),
)

config = AttrDict(_DEFAULTS)


def reset_config():
    """Restore defaults in place (the object identity of `config` is kept)."""
    config.clear()
    for k, v in AttrDict(_DEFAULTS).items():
        config[k] = v
    return config


def _as_pair(v):
    return np.array([v, v]) if isinstance(v, int) else np.array(v)


def _merge_section(name, values):
    section = config[name]
    if name == 'DATASET':
        for key in ('MEAN', 'STD'):
            if values.get(key):
                values[key] = np.array([eval(x) if isinstance(x, str) else x for x in values[key]])
    if name == 'MODEL':
        if 'EXTRA' in values and 'HEATMAP_SIZE' in values['EXTRA']:
            values['EXTRA']['HEATMAP_SIZE'] = _as_pair(values['EXTRA']['HEATMAP_SIZE'])
        if 'IMAGE_SIZE' in values:
            values['IMAGE_SIZE'] = _as_pair(values['IMAGE_SIZE'])
    for key, val in values.items():
        if key not in section:
            raise ValueError("{}.{} not exist in config.py".format(name, key))
        section[key] = val


def update_config(config_file):
    with open(config_file) as f:
        exp = yaml.safe_load(f) or {}
    for key, val in exp.items():
        if key not in config:
            raise ValueError("{} not exist in config.py".format(key))
        if isinstance(val, dict):
            _merge_section(key, val)
        else:
            config[key] = val


def gen_config(config_file):
    def plain(v):
        if isinstance(v, dict):
            return {k: plain(x) for k, x in v.items()}
        if isinstance(v, np.ndarray):
            return v.tolist()
        return v
    with open(config_file, 'w') as f:
        yaml.dump(plain(config), f, default_flow_style=False)


def update_dir(model_dir, log_dir, data_dir):
    if model_dir:
        config.OUTPUT_DIR = model_dir
    if log_dir:
        config.LOG_DIR = log_dir
    if data_dir:
        config.DATA_DIR = data_dir
    config.DATASET.ROOT = os.path.join(config.DATA_DIR, config.DATASET.ROOT)
    config.TEST.COCO_BBOX_FILE = os.path.join(config.DATA_DIR, config.TEST.COCO_BBOX_FILE)
    config.MODEL.PRETRAINED = os.path.join(config.DATA_DIR, config.MODEL.PRETRAINED)


def get_model_name(cfg):
    """(name, full_name) as reference config.py:211-249."""
    extra = cfg.MODEL.EXTRA
    base = cfg.MODEL.NAME
    h, w = cfg.MODEL.IMAGE_SIZE[1], cfg.MODEL.IMAGE_SIZE[0]
    name = '{}_{}'.format(base, extra.NUM_LAYERS)
    if base == 'pose_resnet':
        suffix = ''.join('d{}'.format(n) for n in extra.NUM_DECONV_FILTERS)
    elif base == 'pose3d_resnet':
        suffix = 'DR%s_S%s_DL%s' % (cfg.MODEL.DEPTH_RES, int(cfg.LOSS.USE_SOFT),
                                    int(cfg.LOSS.DEPTH_LAMBDA))
    else:
        raise ValueError('Unkown model: {}'.format(cfg.MODEL))
    full_name = '{}x{}_{}_{}'.format(h, w, name, suffix)
    print(name, full_name)
    return name, full_name


if __name__ == '__main__':
    import sys
    gen_config(sys.argv[1])
