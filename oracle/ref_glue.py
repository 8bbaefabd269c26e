"""TEST INFRASTRUCTURE ONLY -- imports the reference's UNMODIFIED NumPy glue
(src/dataloader/cbmv_generator.py: get_costs :27, extract_features_left :258,
extract_features_lr :84, generate_test_cbmv :727) and binds it to a chosen pair of native
modules:

    load_generator(mtc, fte)   the two objects that `import src.cpp.lib.libmatchers as mtc` /
                               `...libfeatextract as fte` (cbmv_generator.py:16-17) resolve to:
                               either oracle/_ref (the unmodified reference C++), for the CPU
                               baseline and the golden vectors, or the CUDA-backed mirrors
                               (msnets_b200.libmatchers / libfeatextract), for the drop-in tests.

The file is taken from /root/reference when that exists (this container) and otherwise from the
verbatim copy oracle/build_ref.py leaves under oracle/_ref/pyref/ (git-ignored; it travels to the
GPU box like the compiled reference).  The generator's other imports are stubbed: skimage and
matplotlib are absent from this image (only used by down_sampling_input and the plot helpers),
`..pfmutil` / `..funcs_utili` are the reference's PFM reader and plotting module.

Where neither copy exists, restated_generator() gives the oracle's restatement of the same glue behind
the same interface, and write_standin_package() a `src` package laid out like the reference's around it.

Only tests/, bench.py's cpu_baseline / reference legs and tests/golden/make_golden.py may import
this module.  The product package never does.
"""
import importlib.util
import os
import sys
import types
import warnings

_HERE = os.path.dirname(os.path.abspath(__file__))
_CANDIDATES = ["/root/reference/src/dataloader/cbmv_generator.py",
               os.path.join(_HERE, "_ref", "pyref", "src", "dataloader", "cbmv_generator.py")]
_counter = [0]


def generator_path():
    for p in _CANDIDATES:
        if os.path.isfile(p):
            return p
    return None


class _Stub(types.ModuleType):
    """Module whose every attribute is a no-op callable (plot helpers, PFM I/O)."""

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return lambda *a, **k: None


def _load_sibling(name, filename, gen_path):
    """The reference's own src/<filename> (pfmutil.py: the PFM reader generate_crop_train_cbmv needs), executed
    under the stubbed matplotlib; None when the file did not travel."""
    path = os.path.join(os.path.dirname(os.path.dirname(gen_path)), filename)
    if not os.path.isfile(path):
        return None
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        spec.loader.exec_module(mod)
    return mod


def load_generator(mtc, fte, rescale=None):
    """Executes the unmodified cbmv_generator.py in a private package namespace whose
    `src.cpp.lib.libmatchers` / `libfeatextract` are `mtc` / `fte`.  sys.modules is restored
    afterwards, so several bindings (reference C++, CUDA mirrors) can coexist in one process.
    `rescale`: a stand-in for skimage.transform.rescale (absent from this image), called with the
    reference's own keyword arguments -- oracle.ms_oracle.rescale_antialiased restates it over
    scipy.ndimage -- so that the ds_scale = 2 default of generate_test_cbmv / generate_crop_train_cbmv runs.
    Returns the module, or None when the file is not available."""
    path = generator_path()
    if path is None:
        return None
    _counter[0] += 1
    saved = {k: v for k, v in sys.modules.items()
             if k == "src" or k.startswith("src.") or k.split(".")[0] in ("skimage", "matplotlib")}
    for k in saved:
        del sys.modules[k]
    try:
        def pkg(name):
            m = types.ModuleType(name)
            m.__path__ = []
            sys.modules[name] = m
            return m
        src = pkg("src")
        pkg("src.cpp")
        lib = pkg("src.cpp.lib")
        pkg("src.dataloader")
        lib.libmatchers, lib.libfeatextract = mtc, fte
        sys.modules["src.cpp.lib.libmatchers"] = mtc
        sys.modules["src.cpp.lib.libfeatextract"] = fte
        for name in ("skimage", "skimage.transform", "matplotlib", "matplotlib.pyplot", "matplotlib.image"):
            if name not in sys.modules:
                sys.modules[name] = _Stub(name)
        sys.modules["skimage"].transform = sys.modules["skimage.transform"]
        sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
        sys.modules["matplotlib"].image = sys.modules["matplotlib.image"]
        if rescale is not None:
            def _rescale(image, scale, anti_aliasing=True, preserve_range=True, multichannel=False, mode="constant"):
                assert anti_aliasing and preserve_range and not multichannel and mode == "constant"
                return rescale(image, scale)
            sys.modules["skimage.transform"].rescale = _rescale
        sys.modules["src.funcs_utili"] = _Stub("src.funcs_utili")
        sys.modules["src.pfmutil"] = _load_sibling("src.pfmutil", "pfmutil.py", path) or _Stub("src.pfmutil")
        src.pfmutil, src.funcs_utili = sys.modules["src.pfmutil"], sys.modules["src.funcs_utili"]
        name = "src.dataloader.cbmv_generator"
        spec = importlib.util.spec_from_file_location(name, path)
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            spec.loader.exec_module(mod)
        mod.__msnets_binding__ = (mtc, fte)
        return mod
    finally:
        for k in [k for k in sys.modules
                  if k == "src" or k.startswith("src.") or k.split(".")[0] in ("skimage", "matplotlib")]:
            del sys.modules[k]
        sys.modules.update(saved)


def restated_generator(mtc, fte):
    """load_generator's interface over the oracle's restatement of the glue (ms_oracle.get_costs,
    extract_features_left / _lr, generate_test_cbmv), bound to `mtc` / `fte`.  The restatement is pinned
    to the reference's stored outputs by tests/test_oracle_golden.py.  It has no generate_crop_train_cbmv."""
    from oracle import ms_oracle as O

    def get_default_args_dict():     # cbmv_generator.py:434-462, the entries generate_test_cbmv reads
        return {"censw": 11, "nccw": 3, "sadw": 5, "sobelw": 5, "cens_sigma": 128.0, "ncc_sigma": 0.02,
                "sad_sigma": 20000.0, "sobel_sigma": 20000.0, "ds_scale": 2}

    def generate_test_cbmv(leftname, rightname, encoder_ds=64, maxdisp=192, args_dict=None, is_left_only=True):
        import cv2
        import torch
        imgl, imgr = cv2.imread(leftname, 0), cv2.imread(rightname, 0)
        f, h, w, ch, cw = O.generate_test_cbmv(imgl, imgr, encoder_ds, maxdisp, args_dict or get_default_args_dict(),
                                               is_left_only, mtc=mtc, fte=fte)
        return torch.from_numpy(f), h, w, ch, cw

    return types.SimpleNamespace(
        mtc=mtc, fte=fte, get_default_args_dict=get_default_args_dict, generate_test_cbmv=generate_test_cbmv,
        get_costs=lambda *a: O.get_costs(*a, mtc=mtc, fte=fte),
        extract_features_left=lambda *c: O.extract_features_left(*c, fte=fte),
        extract_features_lr=lambda *c: O.extract_features_lr(*c, fte=fte))


_STANDIN_GENERATOR = '''"""Stand-in for the reference's src/dataloader/cbmv_generator.py (oracle/ref_glue.py)."""
import src.cpp.lib.libmatchers as mtc
import src.cpp.lib.libfeatextract as fte
from oracle import ref_glue as _ref_glue

_g = _ref_glue.restated_generator(mtc, fte)
get_default_args_dict = _g.get_default_args_dict
get_costs = _g.get_costs
extract_features_left = _g.extract_features_left
extract_features_lr = _g.extract_features_lr
generate_test_cbmv = _g.generate_test_cbmv
'''


def write_standin_package(root):
    """Writes a package `src` under `root` laid out like the reference's: src/dataloader/cbmv_generator.py
    imports `src.cpp.lib.libmatchers` / `libfeatextract` as cbmv_generator.py:16-17 do and serves its
    functions from restated_generator().  Returns `root`, the directory to put on sys.path."""
    files = {("src", "__init__.py"): "", ("src", "cpp", "__init__.py"): "",
             ("src", "dataloader", "__init__.py"): "",
             ("src", "dataloader", "cbmv_generator.py"): _STANDIN_GENERATOR}
    for parts, text in files.items():
        path = os.path.join(root, *parts)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        with open(path, "w") as f:
            f.write(text)
    return root
