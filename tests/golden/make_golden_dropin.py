"""Golden values for tests/test_dropin_train_script.py: the UNMODIFIED reference
scripts/train.py run over the mirror (CPU emulation of the C ABI, seeded) exactly as the
test runs its own training script; stores the logged losses, the evaluation result, the
final state's keys and a fixed sample of its values.  Needs a checkout of the reference
(EPB_REFERENCE_ROOT, see oracle/refshim.py):
    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden_dropin.py"""
import os
import pathlib
import sys
import tempfile

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), "..", ".."))
sys.path.insert(0, ROOT)
from oracle import refshim  # noqa: E402
from tests.test_dropin_train_script import run_train_script, summarize  # noqa: E402

assert refshim.available(), "reference tree not present at %s" % refshim.REF_ROOT
with tempfile.TemporaryDirectory() as tmp:
    out = summarize(*run_train_script(pathlib.Path(tmp), os.path.join(refshim.REF_ROOT, "scripts")))
np.savez_compressed(os.path.join(os.path.dirname(os.path.abspath(__file__)), "dropin_train.npz"), **out)
print({k: (v.shape, v.dtype) for k, v in out.items()}, out["losses"], out["perf"])
