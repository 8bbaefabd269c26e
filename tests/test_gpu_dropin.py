"""The drop-in under the reference's OWN caller: the unmodified src/dataloader/cbmv_generator.py
(taken from /root/reference here, from the verbatim copy oracle/build_ref.py leaves under
oracle/_ref/pyref on the GPU box) runs with `src.cpp.lib.libmatchers` / `libfeatextract`
(cbmv_generator.py:16-17) resolved to the CUDA-backed mirrors, and its outputs are compared with
the golden vectors the same file produced over the reference C++ (tests/golden/make_golden.py).
Without either copy of that file, the oracle's restatement of the glue (oracle/ref_glue.py) calls
the CUDA mirrors instead, against the same golden vectors.

  get_costs               cbmv_generator.py:27    bit-exact (SHA-256 of every cost volume)
  extract_features_left   :258                    channels 0-3 bit-exact, AML in its stated class
                                                  (tests/_synth.py: <= 2e-6, rare degenerate rows <= 1.2e-5)
  extract_features_lr     :84                     the same against the oracle (golden: SHA only)
  generate_test_cbmv      :727  (ds_scale = 1)    on PNG files, against the stored samples
"""
import os
import sys
import tempfile
import types

import numpy as np
import pytest

from tests._synth import assert_aml_close, digest

pytestmark = pytest.mark.gpu
AML_ATOL = 2e-6
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ms():
    import msnets_b200
    assert msnets_b200.device_count() >= 1
    return msnets_b200


@pytest.fixture(scope="module")
def gen(ms):
    """The unmodified generator bound to the CUDA mirrors through oracle/ref_glue (private module
    namespace, sys.modules untouched afterwards); the oracle's restated glue when the file is absent."""
    from oracle import ref_glue
    g = ref_glue.load_generator(ms.libmatchers, ms.libfeatextract)
    if g is None:
        g = ref_glue.restated_generator(ms.libmatchers, ms.libfeatextract)
    assert g.mtc is ms.libmatchers and g.fte is ms.libfeatextract
    return g


@pytest.mark.parametrize("case", ["small_a", "small_b", "small_c", "medium_a", "medium_b"])
def test_reference_get_costs_and_features_over_cuda_mirrors(gen, oracle, golden_dir, case):
    g = np.load(os.path.join(golden_dir, case + ".npz"))
    H, W, D, seed, shift, border = [int(v) for v in g["meta"]]
    costs = gen.get_costs(g["L"], g["R"], D, 11, 3, 5, 5, border, border, border)      # cbmv_generator.py:27
    for c, key in zip(costs, ("cost_census", "cost_ncc", "cost_sobel", "cost_sad")):
        assert c.dtype == np.float32 and digest(c) == str(g["sha_" + key]), key
    f8 = gen.extract_features_left(*costs)                                            # :258
    assert f8.dtype == np.float32
    want8 = g["features_left"] if "features_left" in g.files else oracle.extract_features_left(*costs)
    assert np.array_equal(f8[:4], want8[:4])
    assert_aml_close(f8[4:], want8[4:])
    if "features_left" not in g.files:   # medium cases store the hash only: the oracle is pinned to it bit for bit
        assert digest(want8) == str(g["sha_features_left"])
    f16 = gen.extract_features_lr(*costs)                                             # :84
    want16 = oracle.extract_features_lr(*costs)
    assert digest(want16) == str(g["sha_features_lr"])
    for lo in (0, 8):
        assert np.array_equal(f16[lo:lo + 4], want16[lo:lo + 4])
        assert_aml_close(f16[lo + 4:lo + 8], want16[lo + 4:lo + 8])


@pytest.mark.parametrize("tag,left_only", [("left", True), ("lr", False)])
def test_reference_generate_test_cbmv_over_cuda_mirrors(gen, golden_dir, tag, left_only):
    """generate_test_cbmv (:727-861) reads two image files, pads, adds the 10 px border, calls
    get_costs + extract_features_*: run here exactly as main_msnet.py's test mode runs it, ds_scale = 1."""
    import cv2
    g = np.load(os.path.join(golden_dir, "test_cbmv.npz"))
    with tempfile.TemporaryDirectory() as td:
        fl, fr = os.path.join(td, "l.png"), os.path.join(td, "r.png")
        cv2.imwrite(fl, g["L"])
        cv2.imwrite(fr, g["R"])
        ad = gen.get_default_args_dict()
        ad["ds_scale"] = 1
        f, h, w, ch, cw = gen.generate_test_cbmv(fl, fr, encoder_ds=16, maxdisp=24, args_dict=ad,
                                                 is_left_only=left_only)
    f = f.numpy()
    assert [h, w, ch, cw] + list(f.shape) == g["meta_" + tag].tolist()
    sub, want = f.reshape(-1)[::5], g["sub_" + tag]
    C = f.shape[0]
    chan = (np.arange(f.size)[::5] // (f.size // C))
    exact = (chan % 8) < 4
    assert np.array_equal(sub[exact], want[exact])
    assert np.abs(sub - want).max() <= AML_ATOL


def test_install_dropin_then_import_unmodified_generator(ms, golden_dir, tmp_path):
    """INTEGRATION.md option A end to end: install_dropin() first, then the reference package is
    imported the way main_msnet.py does (`from src.dataloader import cbmv_generator`) and runs on the
    CUDA mirrors.  The reference checkout, or its copy under oracle/_ref/pyref; without either, a
    stand-in with its layout and imports over the restated glue (oracle/ref_glue.py)."""
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
            sys.modules[name] = types.ModuleType(name)     # absent from this image; plotting / rescale only
        sys.modules["skimage"].transform = sys.modules["skimage.transform"]
        sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
        sys.modules["matplotlib"].image = sys.modules["matplotlib.image"]
        mtc, fte = ms.install_dropin()
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            from src.dataloader import cbmv_generator
        assert cbmv_generator.mtc is mtc and cbmv_generator.fte is fte
        assert os.path.samefile(os.path.dirname(os.path.dirname(cbmv_generator.__file__)),
                                os.path.join(roots[0], "src"))
        g = np.load(os.path.join(golden_dir, "small_a.npz"))
        H, W, D, seed, shift, border = [int(v) for v in g["meta"]]
        costs = cbmv_generator.get_costs(g["L"], g["R"], D, 11, 3, 5, 5, border, border, border)
        f8 = cbmv_generator.extract_features_left(*costs)
        assert np.array_equal(f8[:4], g["features_left"][:4])
        assert np.abs(f8[4:] - g["features_left"][4:]).max() <= AML_ATOL
    finally:
        sys.path.remove(roots[0])
        for k in [k for k in sys.modules
                  if k == "src" or k.startswith("src.") or k.split(".")[0] in ("skimage", "matplotlib")]:
            del sys.modules[k]
        sys.modules.update(saved)
