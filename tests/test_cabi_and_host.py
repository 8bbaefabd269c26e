"""CPU: the C-ABI library loads and exports every symbol include/*.h declares, the
Python mirrors validate their arguments, and -- with no CUDA device -- compute calls
fail loudly instead of falling back to a CPU path."""
import ctypes
import glob
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ms():
    sys.path.insert(0, ROOT)
    import __graft_entry__
    __graft_entry__.build()
    import msnets_b200
    return msnets_b200


def _declared_symbols():
    names = []
    for h in glob.glob(os.path.join(ROOT, "include", "*.h")):
        names += re.findall(r"MSN_API\s+[\w\s\*]+?\b(msn_\w+)\s*\(", open(h).read())
    return sorted(set(names))


def test_library_exports_every_declared_symbol(ms):
    from msnets_b200 import _lib
    declared = _declared_symbols()
    assert len(declared) >= 40
    out = subprocess.run(["nm", "-D", "--defined-only", _lib.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r"\bT (msn_\w+)", out))
    missing = [n for n in declared if n not in exported]
    assert not missing, "declared in include/ but not exported: %s" % missing
    cdll = ctypes.CDLL(_lib.LIB_PATH)
    for n in declared:
        getattr(cdll, n)
    # and the ctypes table binds exactly the declared surface
    assert sorted(_lib.EXPORTS) == declared


def test_sass_is_sm100_only(ms):
    from msnets_b200 import _lib
    out = subprocess.run(["cuobjdump", "--list-elf", _lib.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_params_and_shapes(ms):
    from msnets_b200 import cbmv
    p = cbmv.make_params(192)
    assert (p.censw, p.nccw, p.sadw, p.sobelw) == (11, 3, 5, 5)        # cbmv_generator.py:437-440
    assert abs(p.cens_sigma - 128.0) < 1e-6 and abs(p.ncc_sigma - 0.02) < 1e-7 and p.sad_sigma == 20000.0
    p = cbmv.make_params(96, board_h=10, board_w_left=10, board_w_right=10, left_only=False)
    assert cbmv.output_shape(8, 560, 980, p) == (8, 16, 96, 540, 960)
    d = cbmv.get_default_args_dict()
    assert d["ds_scale"] == 2 and d["board_h"] == 12 and d["cbmv_F"] == 8


def test_argument_validation(ms):
    from msnets_b200 import libfeatextract as fte
    from msnets_b200 import libmatchers as mtc
    img = np.zeros((20, 20), np.uint8)
    with pytest.raises(ValueError):
        mtc.census(img.astype(np.float64), img, 4, 11)       # the reference silently misreads this
    with pytest.raises(ValueError):
        mtc.census(img[:, ::2], img[:, ::2], 4, 11)          # non-contiguous
    with pytest.raises(ValueError):
        mtc.zsad(img, np.zeros((20, 21), np.uint8), 4, 5)
    with pytest.raises(ValueError):
        fte.swap_axes(np.zeros((4, 4), np.float32))
    with pytest.raises(ValueError):
        mtc.sadsob(img, img, 4, 5)                           # needs float32 images


def test_no_cpu_fallback(ms):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the fallback question does not arise")
    from msnets_b200 import MsnetsError, cbmv, libmatchers as mtc, regression
    img = np.zeros((32, 32), np.uint8)
    for call in (lambda: mtc.census(img, img, 4, 11), lambda: mtc.sobel(img),
                 lambda: cbmv.ms_features(img, img, 4),
                 lambda: regression.soft_argmin(np.zeros((1, 4, 2, 2), np.float32))):
        with pytest.raises(MsnetsError, match="no CPU fallback"):
            call()
    with pytest.raises(MsnetsError):
        regression.soft_argmin(torch.zeros(1, 4, 2, 2))


def test_install_dropin_registers_reference_import_names(ms):
    mtc, fte = ms.install_dropin()
    import importlib
    assert importlib.import_module("src.cpp.lib.libmatchers") is mtc
    assert importlib.import_module("src.cpp.lib.libfeatextract") is fte
    for name in ("census", "nccNister", "sadsob", "zsad", "sobel", "initthreads"):   # matchers.cpp:574-579
        assert callable(getattr(mtc, name))
    for name in ("get_cost", "get_right_cost", "swap_axes", "swap_axes_back", "generate_d_indices", "get_samples",
                 "extract_ratio", "extract_likelihood", "get_left_cost", "generate_labels"):  # featextract.cpp:541-553
        assert callable(getattr(fte, name))
    for k in [k for k in sys.modules if k == "src" or k.startswith("src.")]:
        del sys.modules[k]


def test_install_dropin_keeps_the_reference_package_importable(ms, tmp_path):
    """install_dropin() BEFORE the reference package is imported (INTEGRATION.md option A): the real
    `src` package must still import afterwards -- `from src.dataloader import cbmv_generator`
    (main_msnet.py's import chain) -- and see the CUDA mirrors.  No compute here (CPU suite).
    Without a copy of the reference package, a stand-in with its layout and imports (oracle/ref_glue.py)."""
    import types
    import warnings
    from oracle import ref_glue
    roots = [p for p in ("/root/reference", os.path.join(ROOT, "oracle", "_ref", "pyref"))
             if os.path.isfile(os.path.join(p, "src", "dataloader", "cbmv_generator.py"))]
    if not roots:
        roots = [ref_glue.write_standin_package(str(tmp_path))]
    saved = {k: v for k, v in sys.modules.items()
             if k == "src" or k.startswith("src.") or k.split(".")[0] in ("skimage", "matplotlib")}
    for k in saved:
        del sys.modules[k]
    sys.path.insert(0, roots[0])
    try:
        for name in ("skimage", "skimage.transform", "matplotlib", "matplotlib.pyplot", "matplotlib.image"):
            sys.modules[name] = types.ModuleType(name)
        sys.modules["skimage"].transform = sys.modules["skimage.transform"]
        sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
        sys.modules["matplotlib"].image = sys.modules["matplotlib.image"]
        mtc, fte = ms.install_dropin()
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            from src.dataloader import cbmv_generator
        assert cbmv_generator.mtc is mtc and cbmv_generator.fte is fte
        assert callable(cbmv_generator.get_costs) and callable(cbmv_generator.generate_test_cbmv)
    finally:
        sys.path.remove(roots[0])
        for k in [k for k in sys.modules
                  if k == "src" or k.startswith("src.") or k.split(".")[0] in ("skimage", "matplotlib")]:
            del sys.modules[k]
        sys.modules.update(saved)


def test_product_never_imports_oracle():
    """The oracle is test infrastructure: nothing under ms-nets_b200/ may reference it."""
    pkg = os.path.join(ROOT, "ms-nets_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert "ms_oracle" not in text.replace("oracle/ms_oracle.py", ""), f
                assert not re.search(r"^\s*(from|import)\s+oracle", text, re.M), f
