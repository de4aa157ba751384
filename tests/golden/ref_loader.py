"""Load the UNMODIFIED reference (`$NIC_REFERENCE_DIR/image_compression.py`) in-process.

NIC_REFERENCE_DIR names the `Projects/` directory of a checkout of the reference project, which is not part of this
repository.  Used by `tests/golden/make_golden.py` to regenerate the fixtures; at test time only the tests that compare
with the reference's source import it, and they skip when NIC_REFERENCE_DIR is unset.  Recipe = SURVEY.md §8(c):
`runpy.run_path` with `NUM_EPOCHS=0`, no-op stubs for the two missing plotting/logging packages, and a
scratch cwd that holds the directories the script writes into.
"""
import os
import runpy
import sys
import tempfile
import types

REF = os.environ.get("NIC_REFERENCE_DIR", "")


def _stub_modules():
    tbx = types.ModuleType("tensorboardX")

    class SummaryWriter:  # no-op stand-in for tensorboardX.SummaryWriter
        def __init__(self, *a, **k):
            pass

        def add_scalar(self, *a, **k):
            pass

        def close(self):
            pass

    tbx.SummaryWriter = SummaryWriter
    sys.modules["tensorboardX"] = tbx
    mpl = types.ModuleType("matplotlib")
    plt = types.ModuleType("matplotlib.pyplot")
    for name in ("figure", "subplot", "imshow", "axis", "title", "show"):
        setattr(plt, name, lambda *a, **k: None)
    mpl.pyplot = plt
    sys.modules["matplotlib"] = mpl
    sys.modules["matplotlib.pyplot"] = plt


def load_reference(*overrides, npy=None):
    """Return the globals dict of image_compression.py executed with `KEY=VALUE` overrides.

    `npy`: optional uint8 ndarray saved as the IMAGE_PATH for 3-D configs.
    """
    import numpy as np

    if not REF or not os.path.exists(os.path.join(REF, "image_compression.py")):
        raise FileNotFoundError("set NIC_REFERENCE_DIR to the reference project's Projects/ directory")
    os.environ["PYTHONDONTWRITEBYTECODE"] = "1"
    sys.dont_write_bytecode = True
    _stub_modules()
    if REF not in sys.path:
        sys.path.insert(0, REF)
    for m in ("var2", "utils", "models", "fp_def"):
        sys.modules.pop(m, None)
    import utils as _ref_utils  # the reference's utils.py (REF is first on sys.path)

    # video I/O stub: utils.timelaps hard-codes 64 frames (utils.py:86-93) and is outside the hot path
    _ref_utils.timelaps = lambda *a, **k: None
    scratch = tempfile.mkdtemp(prefix="nicref_")
    for d in ("model", "feature_pyramid", "image", "printlog", "LUT"):
        os.makedirs(os.path.join(scratch, d), exist_ok=True)
    os.symlink(os.path.join(REF, "data"), os.path.join(scratch, "data"))
    args = ["image_compression.py", "NUM_EPOCHS=0", "TF_SHOW_RESULT=0"] + list(overrides)
    if npy is not None:
        path = os.path.join(scratch, "vol.npy")
        np.save(path, npy)
        args.append(f"IMAGE_PATH={path}")
    old_argv, old_cwd = sys.argv, os.getcwd()
    sys.argv = args
    os.chdir(scratch)
    try:
        g = runpy.run_path(os.path.join(REF, "image_compression.py"), run_name="ref")
    finally:
        sys.argv = old_argv
        os.chdir(old_cwd)
    g["__scratch__"] = scratch
    return g
