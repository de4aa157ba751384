"""INTEGRATION.md section 1.  The documented block, exec'd on its own, binds every hot-path name to this package (runs
everywhere).  The tests marked `needs_reference` check it against the REAL reference script, which is not part of this
repository: they run when NIC_REFERENCE_DIR names the reference's Projects/ directory and skip otherwise
(tests/test_gpu_round2.py::test_integration_import_swap_recipe_runs_the_script_flow covers the run-time side without it).

The reference's image_compression.py is executed up to line 346 (imports, configuration, its function definitions — nothing
that touches a device), the documented block is appended, and the resulting namespace is checked: every global name the
script's hot functions use resolves, the hot-path names are this package's, and their signatures take the reference's calls."""
import ast
import builtins
import inspect
import os
import re
import sys

import pytest

from ref_loader import REF  # tests/golden: $NIC_REFERENCE_DIR

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = "neural_image_compression_v2_b200"

needs_reference = pytest.mark.skipif(not REF or not os.path.exists(os.path.join(REF, "image_compression.py")),
                                     reason="needs the reference project's Projects/ directory in NIC_REFERENCE_DIR")

HOT = ["ColorDecoder", "create_decoder_input_2d", "create_decoder_input_3d", "create_decoder_input_3d_v2",
       "finally_decode_input_2d", "finally_decode_input_3d", "finally_decode_input_3d_v2", "create_pyramid", "create_pyramid_3d",
       "create_pyramid_mip_levels", "fp_quantize_clamp", "fp_all_quantize", "fp_savable", "fp_load", "fp_freeze", "quantize4fp",
       "save4fp", "load4fp", "quantize_to_bit", "calculate_psnr", "triangular_positional_encoding", "positional_encoding",
       "bits2dtype_torch", "bits2dtype_np"]
HOST_HELPERS = ("print_", "make_filename_by_seq", "safe_statistics", "quantize_from_bit_to_bit")


def _recipe_block():
    doc = open(os.path.join(ROOT, "INTEGRATION.md")).read()
    sec1 = doc[doc.index("## 1."):doc.index("## 2.")]
    return re.findall(r"```python\n(.*?)```", sec1, flags=re.S)[1]


def test_recipe_block_binds_the_hot_path_names_and_nothing_else():
    """The inserted block alone (the script's own globals absent, so var2 keeps its defaults): every hot-path name it binds
    is this package's, and it binds none of the host-side helpers the script keeps from the reference's utils."""
    ns = {"__name__": "recipe_block"}
    exec(compile(_recipe_block(), "INTEGRATION.md(section 1 block)", "exec"), ns)
    for name in HOT:
        assert name in ns and ns[name].__module__.startswith(PKG), (name, getattr(ns.get(name), "__module__", None))
    for name in HOST_HELPERS:
        assert name not in ns, name


def _namespace():
    import tempfile
    from ref_loader import _stub_modules                   # tensorboardX / matplotlib no-op stubs (tests/golden)
    _stub_modules()
    block = _recipe_block()
    src = open(os.path.join(REF, "image_compression.py"), encoding="utf-8").read().split("\n")
    assert src[349].startswith("decoder = ColorDecoder()"), "the recipe's insertion point (line 350) moved"
    text = "\n".join(src[:346]) + "\n" + block
    scratch = tempfile.mkdtemp(prefix="nicrecipe_")
    os.makedirs(os.path.join(scratch, "printlog"), exist_ok=True)
    old_argv, old_cwd, old_path = sys.argv, os.getcwd(), list(sys.path)
    saved = {m: sys.modules.pop(m, None) for m in ("var2", "utils", "models", "fp_def")}
    sys.argv = ["image_compression.py", "NUM_EPOCHS=0"]
    sys.path.insert(0, REF)
    os.chdir(scratch)
    sys.dont_write_bytecode = True
    ns = {"__name__": "ref_with_recipe"}
    try:
        exec(compile(text, "image_compression.py(+recipe)", "exec"), ns)
        ref_mods = {m: sys.modules[m] for m in ("utils", "models", "fp_def")}
    finally:
        sys.argv = old_argv
        os.chdir(old_cwd)
        sys.path[:] = old_path
        for m, v in saved.items():
            sys.modules.pop(m, None)
            if v is not None:
                sys.modules[m] = v
    return ns, ref_mods, src


@needs_reference
def test_recipe_shadows_the_hot_path_and_every_script_global_resolves():
    ns, ref_mods, src = _namespace()
    for name in HOT:
        assert ns[name].__module__.startswith(PKG), (name, ns[name].__module__)
    # host-side helpers stay the reference's own
    for name in HOST_HELPERS:
        assert not ns[name].__module__.startswith(PKG)
    # globals used by the script's functions: defined by line 346 + the block, or assigned at module level further down
    tree = ast.parse("\n".join(src))
    later = set()
    for node in tree.body:
        if node.lineno > 346:
            for sub in ast.walk(node):
                if isinstance(sub, ast.Name) and isinstance(sub.ctx, ast.Store):
                    later.add(sub.id)
    for fn in [n for n in tree.body if isinstance(n, ast.FunctionDef)]:
        if fn.name not in ("train_models", "decode_image", "process_images", "random_crop_dataset"):
            continue
        local = {a.arg for a in fn.args.args} | {s.id for s in ast.walk(fn) if isinstance(s, ast.Name) and isinstance(s.ctx, ast.Store)}
        used = {s.id for s in ast.walk(fn) if isinstance(s, ast.Name) and isinstance(s.ctx, ast.Load)}
        missing = [u for u in sorted(used - local) if u not in ns and u not in later and not hasattr(builtins, u)]
        assert not missing, (fn.name, missing)


@needs_reference
def test_shadowed_functions_accept_the_reference_signatures():
    """Same parameter names in the same order as the reference's functions (ours may append optional ones)."""
    ns, ref_mods, src = _namespace()
    tree = ast.parse("\n".join(src))
    script_defs = {n.name: [a.arg for a in n.args.args] for n in tree.body if isinstance(n, ast.FunctionDef)}
    checked = 0
    for name, obj in ns.items():
        if not callable(obj) or not getattr(obj, "__module__", "").startswith(PKG) or inspect.isclass(obj):
            continue
        ref_params = None
        for m in ref_mods.values():
            if hasattr(m, name) and inspect.isfunction(getattr(m, name)):
                ref_params = list(inspect.signature(getattr(m, name)).parameters)
        if name in script_defs:
            ref_params = script_defs[name]
        if ref_params is None:
            continue
        ours = inspect.signature(obj).parameters
        names = list(ours)
        assert names[:len(ref_params)] == ref_params, (name, names, ref_params)
        for extra in names[len(ref_params):]:
            assert ours[extra].default is not inspect.Parameter.empty, (name, extra)
        checked += 1
    assert checked >= 20, checked
