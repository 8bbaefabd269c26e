"""TEST INFRASTRUCTURE ONLY -- Python face of the CPU oracle.

* ctypes bindings to oracle/libms_oracle.so (the C restatement, ms_oracle.c);
* NumPy restatements of the reference's glue:
    get_costs             -> src/dataloader/cbmv_generator.py:27-79
    extract_features_left -> src/dataloader/cbmv_generator.py:258-308
    extract_features_lr   -> src/dataloader/cbmv_generator.py:84-254
    generate_test_cbmv    -> src/dataloader/cbmv_generator.py:727-861 (ds_scale = 1 branch)
    WTA pictures          -> main_msnet.py:444-448 (np.argmin over D)
    soft-argmin           -> src/models/gcnet_3dcnn.py:127-141
* definitions for the north-star items that have NO reference code (SURVEY.md
  section 0.3 / 8a row 14): second-min / peak-ratio confidence, left-right
  consistency mask, concat / difference 4D volume.  Those are "parity unpinned"
  by the reference: this file is their only definition.
* load_ref(): the UNMODIFIED reference compiled into oracle/_ref (build_ref.py).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / reference
legs may import this module.  The product package never does.
"""
import ctypes
import importlib.util
import os
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libms_oracle.so")
FILL = np.float32(2147483648.0)  # float(RAND_MAX), matchers.cpp:65

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.isfile(_LIB_PATH):
            sys.path.insert(0, _HERE)
            import build_oracle
            build_oracle.build(verbose=False)
        L = ctypes.CDLL(_LIB_PATH)
        u8p = ctypes.POINTER(ctypes.c_uint8)
        f32p = ctypes.POINTER(ctypes.c_float)
        ci, cl, cf = ctypes.c_int, ctypes.c_long, ctypes.c_float
        for name in ("orc_census", "orc_ncc", "orc_zsad"):
            getattr(L, name).argtypes = [u8p, u8p, ci, ci, ci, ci, f32p]
        L.orc_sobel.argtypes = [u8p, ci, ci, f32p]
        L.orc_sadsob.argtypes = [f32p, f32p, ci, ci, ci, ci, f32p]
        L.orc_swap_axes.argtypes = [f32p, ci, ci, ci, f32p]
        L.orc_swap_axes_back.argtypes = [f32p, ci, ci, ci, f32p]
        L.orc_get_right_cost.argtypes = [f32p, ci, ci, ci, f32p]
        L.orc_get_left_cost.argtypes = [f32p, ci, ci, ci, f32p]
        L.orc_aml.argtypes = [f32p, cl, ci, cf, f32p]
        L.orc_pkrn.argtypes = [f32p, cl, ci, cf, f32p]
        L.orc_soft_argmin.argtypes = [f32p, ci, ci, ci, ci, f32p]
        _lib = L
    return _lib


def _u8(a):
    a = np.ascontiguousarray(a)
    if a.dtype != np.uint8 or a.ndim != 2:
        raise ValueError("expected a C-contiguous uint8 [H,W] image")
    return a


def _f32(a):
    a = np.ascontiguousarray(a)
    if a.dtype != np.float32:
        raise ValueError("expected float32")
    return a


def _p(a, ct):
    return a.ctypes.data_as(ctypes.POINTER(ct))


# ------------------------------------------------------------------ matchers
def census(left, right, ndisp, wsize):
    """matchers.cpp:232-353 -> float32 [H,W,D]."""
    l, r = _u8(left), _u8(right)
    H, W = l.shape
    out = np.empty((H, W, ndisp), np.float32)
    lib().orc_census(_p(l, ctypes.c_uint8), _p(r, ctypes.c_uint8), H, W, ndisp, wsize,
                     _p(out, ctypes.c_float))
    return out


def nccNister(left, right, ndisp, wsize):
    """matchers.cpp:47-228 -> float32 [D,H,W]."""
    l, r = _u8(left), _u8(right)
    H, W = l.shape
    out = np.empty((ndisp, H, W), np.float32)
    lib().orc_ncc(_p(l, ctypes.c_uint8), _p(r, ctypes.c_uint8), H, W, ndisp, wsize,
                  _p(out, ctypes.c_float))
    return out


def zsad(left, right, ndisp, wsize):
    """matchers.cpp:442-512 -> float32 [D,H,W]."""
    l, r = _u8(left), _u8(right)
    H, W = l.shape
    out = np.empty((ndisp, H, W), np.float32)
    lib().orc_zsad(_p(l, ctypes.c_uint8), _p(r, ctypes.c_uint8), H, W, ndisp, wsize,
                   _p(out, ctypes.c_float))
    return out


def sobel(img):
    """matchers.cpp:515-554 -> float32 [H,W]."""
    a = _u8(img)
    H, W = a.shape
    out = np.empty((H, W), np.float32)
    lib().orc_sobel(_p(a, ctypes.c_uint8), H, W, _p(out, ctypes.c_float))
    return out


def sadsob(left, right, ndisp, wsize):
    """matchers.cpp:356-438 -> float32 [D,H,W]."""
    l, r = _f32(left), _f32(right)
    H, W = l.shape
    out = np.empty((ndisp, H, W), np.float32)
    lib().orc_sadsob(_p(l, ctypes.c_float), _p(r, ctypes.c_float), H, W, ndisp, wsize,
                     _p(out, ctypes.c_float))
    return out


def initthreads():
    """matchers.cpp:556-563 returns THREADS_NUM_USED (paramSetting.hpp:11)."""
    return 8


# --------------------------------------------------------------- featextract
def swap_axes(cost):
    """featextract.cpp:49-76: [D,H,W] -> [H,W,D]."""
    c = _f32(cost)
    D, H, W = c.shape
    out = np.empty((H, W, D), np.float32)
    lib().orc_swap_axes(_p(c, ctypes.c_float), D, H, W, _p(out, ctypes.c_float))
    return out


def swap_axes_back(cost):
    """featextract.cpp:78-105: [H,W,D] -> [D,H,W]."""
    c = _f32(cost)
    H, W, D = c.shape
    out = np.empty((D, H, W), np.float32)
    lib().orc_swap_axes_back(_p(c, ctypes.c_float), H, W, D, _p(out, ctypes.c_float))
    return out


def get_right_cost(cost):
    """featextract.cpp:136-172."""
    c = _f32(cost)
    H, W, D = c.shape
    out = np.empty_like(c)
    lib().orc_get_right_cost(_p(c, ctypes.c_float), H, W, D, _p(out, ctypes.c_float))
    return out


def get_left_cost(cost):
    """featextract.cpp:464-499."""
    c = _f32(cost)
    H, W, D = c.shape
    out = np.empty_like(c)
    lib().orc_get_left_cost(_p(c, ctypes.c_float), H, W, D, _p(out, ctypes.c_float))
    return out


def extract_likelihood(cost, sigma):
    """featextract.cpp:415-462 (2-arg overload): AML over rows of [n,D]."""
    c = _f32(cost)
    n, D = c.shape
    out = np.empty_like(c)
    lib().orc_aml(_p(c, ctypes.c_float), n, D, float(sigma), _p(out, ctypes.c_float))
    return out


def extract_ratio(cost, e):
    """featextract.cpp:320-356 (2-arg overload): (min+e)/(c+e) over rows of [n,D]."""
    c = _f32(cost)
    n, D = c.shape
    out = np.empty_like(c)
    lib().orc_pkrn(_p(c, ctypes.c_float), n, D, float(e), _p(out, ctypes.c_float))
    return out


class _NS(object):
    """Tiny namespace so the oracle can be passed where (mtc, fte) modules go."""

    def __init__(self, **kw):
        self.__dict__.update(kw)


MTC = _NS(census=census, nccNister=nccNister, zsad=zsad, sobel=sobel, sadsob=sadsob,
          initthreads=initthreads)
FTE = _NS(swap_axes=swap_axes, swap_axes_back=swap_axes_back, get_right_cost=get_right_cost,
          get_left_cost=get_left_cost, extract_likelihood=extract_likelihood,
          extract_ratio=extract_ratio)


# ------------------------------------------------ NumPy glue (cbmv_generator)
def get_costs(iml, imr, maxdisp=192, censw=11, nccw=3, sadw=5, sobelw=5, board_h=10,
              board_w_left=10, board_w_right=0, mtc=MTC, fte=FTE):
    """cbmv_generator.py:27-79.  Returns (census, ncc, sobel, sad), each float32
    [h,w,D] C-contiguous after the border crop.  `mtc`/`fte` select who computes:
    the C oracle (default) or the compiled reference from load_ref()."""
    cen = mtc.census(iml, imr, maxdisp, censw).astype(np.float32)
    ncc = fte.swap_axes(mtc.nccNister(iml, imr, maxdisp, nccw).astype(np.float32))
    sad = fte.swap_axes(mtc.zsad(iml, imr, maxdisp, sadw).astype(np.float32))
    sob = fte.swap_axes(mtc.sadsob(mtc.sobel(iml), mtc.sobel(imr), maxdisp, sobelw)
                        .astype(np.float32))
    he = -board_h if board_h > 0 else None
    we = -board_w_right if board_w_right > 0 else None
    crop = lambda a: a[board_h:he, board_w_left:we, :].copy(order="C")
    return crop(cen), crop(ncc), crop(sob), crop(sad)


def _normalise4(census_c, ncc_c, sobel_c, sad_c):
    """cbmv_generator.py:283-287 (the same four lines at :210-213, :234-237)."""
    return (np.clip(census_c, 0., 120.) / 120.,
            (1 + np.clip(ncc_c, -1., 1.)) / 2,
            np.clip(sobel_c, 0., 2 ** 13) / float(2 ** 13),
            np.clip(sad_c, 0., 2 ** 13) / float(2 ** 13))


def extract_features_left(census_c, ncc_c, sobel_c, sad_c, cens_sigma=128.0, ncc_sigma=0.02,
                          sad_sigma=20000.0, sobel_sigma=20000.0, disp_image=None, fte=FTE):
    """cbmv_generator.py:258-308 -> float32 [8,D,h,w].  sobel_sigma is accepted
    and ignored, as in the reference (:298 uses sad_sigma for the sobel channel).
    The reference's float64 scratch (:281) holds float32 values exactly, so it is
    skipped here without changing any bit of the result."""
    h, w, D = census_c.shape
    flat = [np.reshape(a, [h * w, D]) for a in (census_c, ncc_c, sobel_c, sad_c)]
    feats = np.empty((8, h, w, D), np.float32)
    for k, v in enumerate(_normalise4(*flat)):
        feats[k] = np.reshape(v, [h, w, D])
    for k, (a, s) in enumerate(zip(flat, (cens_sigma, ncc_sigma, sad_sigma, sad_sigma))):
        feats[4 + k] = np.reshape(fte.extract_likelihood(a, s), [h, w, D])
    return np.ascontiguousarray(feats.transpose((0, 3, 1, 2)))


def extract_features_lr(census_c, ncc_c, sobel_c, sad_c, cens_sigma=128.0, ncc_sigma=0.02,
                        sad_sigma=20000.0, sobel_sigma=20000.0, disp_image=None, fte=FTE):
    """cbmv_generator.py:84-254 -> float32 [16,D,h,w] (left 0-7, right-view 8-15)."""
    h, w, D = census_c.shape
    left = (census_c, ncc_c, sobel_c, sad_c)
    right = tuple(fte.get_right_cost(np.ascontiguousarray(a)) for a in left)
    feats = np.empty((16, h, w, D), np.float32)
    sig = (cens_sigma, ncc_sigma, sad_sigma, sad_sigma)
    for base, vols in ((0, left), (8, right)):
        flat = [np.reshape(a, [h * w, D]) for a in vols]
        for k, v in enumerate(_normalise4(*flat)):
            feats[base + k] = np.reshape(v, [h, w, D])
        for k, (a, s) in enumerate(zip(flat, sig)):
            feats[base + 4 + k] = np.reshape(fte.extract_likelihood(a, s), [h, w, D])
    return np.ascontiguousarray(feats.transpose((0, 3, 1, 2)))


def ms_features(iml, imr, maxdisp=192, board_h=10, board_w_left=10, board_w_right=10,
                left_only=True, mtc=MTC, fte=FTE, **kw):
    """get_costs + extract_features_{left,lr} as generate_test_cbmv chains them
    (cbmv_generator.py:826-843) on an already bordered uint8 pair."""
    costs = get_costs(iml, imr, maxdisp, board_h=board_h, board_w_left=board_w_left,
                      board_w_right=board_w_right, mtc=mtc, fte=fte, **kw)
    f = extract_features_left if left_only else extract_features_lr
    return f(*costs, fte=fte)


# --------------------------------------------------------------- soft-argmin
def pad_test_pair(imgl, imgr, encoder_ds):
    """cbmv_generator.py:780-788 + :819-823: zero-pad top/right to a multiple of encoder_ds,
    then a 10-pixel zero border on all four sides.  Returns (L, R, h, w, crop_h, crop_w)."""
    h, w = imgl.shape[:2]
    crop_w = w + (encoder_ds - w % encoder_ds) % encoder_ds
    crop_h = h + (encoder_ds - h % encoder_ds) % encoder_ds
    out = []
    for im in (imgl, imgr):
        a = np.pad(im, ((crop_h - h, 0), (0, crop_w - w)), "constant").astype(np.uint8)
        out.append(np.ascontiguousarray(np.pad(a, ((10, 10), (10, 10)), "constant").astype(np.uint8)))
    return out[0], out[1], h, w, crop_h, crop_w


def rescale_antialiased(img_f32, scale):
    """skimage.transform.rescale(image, scale, anti_aliasing=True, preserve_range=True, mode='constant')
    for a 2-D float32 image, order 1 -- the call down_sampling_input makes (cbmv_generator.py:465-482).
    skimage is NOT installed in this image (PARITY UNPINNED against skimage itself); this restates what
    skimage >= 0.19 does (transform/_warps.py: rescale -> resize) on top of scipy.ndimage, which IS
    installed and is the engine skimage delegates to:
        output_shape = round(scale * shape); factors = shape / output_shape
        filtered = ndi.gaussian_filter(image, sigma=max(0,(factors-1)/2), mode='constant', cval=0)
        out = ndi.zoom(filtered, 1/factors, order=1, mode='grid-constant', cval=0, grid_mode=True)
        clip to [image.min(), image.max()]  (output pixels equal to cval stay cval)
    float32 in, float32 out (skimage >= 0.19 keeps float32)."""
    import scipy.ndimage as ndi
    image = np.ascontiguousarray(img_f32, np.float32)
    out_shape = tuple(int(v) for v in np.round(np.asarray(image.shape) * scale))
    factors = np.asarray(image.shape, np.float64) / np.asarray(out_shape, np.float64)
    sigma = np.maximum(0, (factors - 1) / 2)
    filtered = ndi.gaussian_filter(image, sigma, cval=0, mode="constant")
    zoom = [1 / f for f in factors]
    out = ndi.zoom(filtered, zoom, order=1, mode="grid-constant", cval=0, grid_mode=True)
    assert out.shape == out_shape and out.dtype == np.float32
    lo, hi = image.min(), image.max()
    preserve_cval = not (lo <= 0 <= hi)          # skimage _clip_warp_output, mode='constant', cval=0
    if preserve_cval:
        mask = out == 0
    np.clip(out, lo, hi, out=out)
    if preserve_cval:
        out[mask] = 0
    return out


def rescale_antialiased_replay(img_f32, scale):
    """The same, with scipy's arithmetic written out (ni_filters.c NI_Correlate1D symmetric branch,
    ni_interpolation.c NI_ZoomShift order 1): the form the CUDA kernel follows.  Checked against
    rescale_antialiased bit for bit in tests/test_oracle_golden.py."""
    image = np.ascontiguousarray(img_f32, np.float32)
    H, W = image.shape
    oh, ow = (int(v) for v in np.round(np.asarray(image.shape) * scale))
    cur = image
    for axis, (n_in, n_out) in enumerate(((H, oh), (W, ow))):
        sigma = max(0.0, (n_in / n_out - 1) / 2)
        if sigma <= 0:
            continue
        r = int(4.0 * sigma + 0.5)
        x = np.arange(-r, r + 1)
        w = np.exp(-0.5 / (sigma * sigma) * x ** 2)
        w = w / w.sum()
        a = np.moveaxis(cur, axis, 0).astype(np.float64)
        pad = np.zeros((r,) + a.shape[1:])
        e = np.concatenate([pad, a, pad], 0)
        n = a.shape[0]
        t = e[r:r + n] * w[r]
        for j in range(-r, 0):                          # farthest taps first, pairs added before the multiply
            t = t + (e[r + j:r + j + n] + e[r - j:r - j + n]) * w[r + j]
        cur = np.ascontiguousarray(np.moveaxis(t.astype(np.float32), 0, axis))
    zr, zc = H / oh, W / ow

    def taps(n_out, n_in, z):
        c = (np.arange(n_out, dtype=np.float64) + 0.5) * z - 0.5
        f = np.floor(c)
        return f.astype(np.int64), c - f
    fr, wr = taps(oh, H, zr)
    fc, wc = taps(ow, W, zc)
    g = np.pad(cur.astype(np.float64), 1)               # grid-constant: zeros outside
    out = np.zeros((oh, ow), np.float64)
    for i, wi in ((0, 1 - wr), (1, wr)):
        for j, wj in ((0, 1 - wc), (1, wc)):
            out += (g[np.ix_(fr + i + 1, fc + j + 1)] * wi[:, None]) * wj[None, :]
    out = out.astype(np.float32)
    lo, hi = image.min(), image.max()
    preserve_cval = not (lo <= 0 <= hi)
    if preserve_cval:
        mask = out == 0
    np.clip(out, lo, hi, out=out)
    if preserve_cval:
        out[mask] = 0
    return out


def down_sampling_input(ds_scale, imgl, imgr):
    """cbmv_generator.py:465-482: uint8 -> float32/255 -> rescale -> *255 -> uint8 (truncation)."""
    out = []
    for im in (imgl, imgr):
        f = im.astype(np.float32) / 255.0
        z = rescale_antialiased(f, ds_scale)
        out.append(np.ascontiguousarray((z * 255.0).astype(np.uint8)))
    return out[0], out[1]


def generate_test_cbmv(imgl, imgr, encoder_ds=64, maxdisp=192, args_dict=None, is_left_only=True, mtc=MTC,
                       fte=FTE):
    """cbmv_generator.py:727-861 on two uint8 gray images (the reference reads them with
    cv2.imread(name, 0)).  ds_scale > 1 goes through down_sampling_input (rescale_antialiased: pinned to
    scipy.ndimage, not to skimage itself -- see there).  `mtc`/`fte` as in get_costs.
    Returns (features float32 [C, D, crop_h, crop_w], h, w, crop_h, crop_w)."""
    ad = dict(censw=11, nccw=3, sadw=5, sobelw=5, cens_sigma=128.0, ncc_sigma=0.02, sad_sigma=20000.0,
              sobel_sigma=20000.0, ds_scale=1)
    if args_dict:
        ad.update(args_dict)
    ds = int(ad["ds_scale"])
    h, w = imgl.shape[:2]
    crop_w = w + (encoder_ds - w % encoder_ds) % encoder_ds
    crop_h = h + (encoder_ds - h % encoder_ds) % encoder_ds
    pl = np.pad(imgl, ((crop_h - h, 0), (0, crop_w - w)), "constant").astype(np.uint8)
    pr = np.pad(imgr, ((crop_h - h, 0), (0, crop_w - w)), "constant").astype(np.uint8)
    if ds > 1:
        pl, pr = down_sampling_input(1.0 / ds, pl, pr)                                  # :802-803
    L = np.ascontiguousarray(np.pad(pl, ((10, 10), (10, 10)), "constant").astype(np.uint8))
    R = np.ascontiguousarray(np.pad(pr, ((10, 10), (10, 10)), "constant").astype(np.uint8))
    costs = get_costs(L, R, maxdisp // ds, ad["censw"], ad["nccw"], ad["sadw"], ad["sobelw"],
                      10, 10, 10, mtc=mtc, fte=fte)
    fn = extract_features_left if is_left_only else extract_features_lr
    f = fn(*costs, cens_sigma=ad["cens_sigma"], ncc_sigma=ad["ncc_sigma"], sad_sigma=ad["sad_sigma"], fte=fte)
    return f, h, w, crop_h, crop_w


def soft_argmin(logits):
    """gcnet_3dcnn.py:127-141: softmax over dim 1 of [N,D,H,W], expectation of d."""
    x = _f32(logits)
    N, D, H, W = x.shape
    out = np.empty((N, H, W), np.float32)
    lib().orc_soft_argmin(_p(x, ctypes.c_float), N, D, H, W, _p(out, ctypes.c_float))
    return out


# ------------------------------------------- WTA / confidence (partly unpinned)
def wta(cost_hwd):
    """main_msnet.py:444-448: np.argmin over D, first minimal index wins; an
    all-fill pixel yields 0.  Also returns min and second-min (the 2nd smallest
    entry counting duplicates; no reference code -- definition lives here)."""
    c = np.asarray(cost_hwd, np.float32)
    idx = np.argmin(c, axis=-1).astype(np.int32)
    part = np.partition(c, 1, axis=-1)
    return idx, part[..., 0].copy(), part[..., 1].copy()


def pkrn_confidence(min1, min2, e):
    """Peak-ratio (naive) per pixel, same algebra as featextract.cpp:349 evaluated
    at the second minimum: (min1 + e) / (min2 + e); 0 where min1 is fill."""
    with np.errstate(all="ignore"):
        r = (min1 + np.float32(e)) / (min2 + np.float32(e))
    return np.where(min1 == FILL, np.float32(0), r).astype(np.float32)


def lr_consistency(cost_hwd, thresh=1):
    """Left-right check (no reference code; SURVEY.md 8a row 14):
    dL = argmin_d c[y,x,d]; dR = argmin_d get_right_cost(c)[y,x,d];
    mask[y,x] = 1 iff x-dL >= 0 and |dL[y,x] - dR[y,x-dL]| <= thresh."""
    c = np.ascontiguousarray(cost_hwd, np.float32)
    H, W, D = c.shape
    dl = np.argmin(c, axis=-1).astype(np.int32)
    dr = np.argmin(get_right_cost(c), axis=-1).astype(np.int32)
    xs = np.arange(W, dtype=np.int32)[None, :] - dl
    ok = xs >= 0
    drs = np.take_along_axis(dr, np.clip(xs, 0, W - 1), axis=1)
    mask = ok & (np.abs(dl - drs) <= thresh)
    return dl, dr, mask.astype(np.uint8)


# ---------------------------------------------- 4D volumes (unpinned, own def)
def concat_volume(fl, fr, ndisp):
    """GC-Net / PSMNet concat volume (shape the reference's dres0 expects,
    psmnet_3dcnn.py:96): vol[n,:C,d,y,x]=fl[n,:,y,x], vol[n,C:,d,y,x]=fr[n,:,y,x-d]
    for x >= d, zero elsewhere.  [N,C,H,W] x2 -> [N,2C,D,H,W]."""
    N, C, H, W = fl.shape
    vol = np.zeros((N, 2 * C, ndisp, H, W), fl.dtype)
    for d in range(min(ndisp, W)):
        vol[:, :C, d, :, d:] = fl[:, :, :, d:]
        vol[:, C:, d, :, d:] = fr[:, :, :, :W - d]
    return vol


def diff_volume(fl, fr, ndisp):
    """Difference volume: vol[n,c,d,y,x] = fl[n,c,y,x] - fr[n,c,y,x-d] for x >= d."""
    N, C, H, W = fl.shape
    vol = np.zeros((N, C, ndisp, H, W), fl.dtype)
    for d in range(min(ndisp, W)):
        vol[:, :, d, :, d:] = fl[:, :, :, d:] - fr[:, :, :, :W - d]
    return vol


# ----------------------------------------------------------- the real thing
def cpu_has_avx2():
    try:
        with open("/proc/cpuinfo") as f:
            return " avx2 " in f.read().replace("\n", " ")
    except OSError:
        return False


def load_ref(variant=None):
    """Imports the UNMODIFIED reference libmatchers / libfeatextract compiled by
    oracle/build_ref.py.  Returns (mtc, fte, variant) or None when absent."""
    order = [variant] if variant else (["avx2", "sse41"] if cpu_has_avx2() else ["sse41"])
    for v in order:
        d = os.path.join(_HERE, "_ref", v)
        paths = [os.path.join(d, m + ".so") for m in ("libmatchers", "libfeatextract")]
        if not all(os.path.isfile(p) for p in paths):
            continue
        mods = []
        for name, p in zip(("libmatchers", "libfeatextract"), paths):
            key = "_msnets_ref_%s_%s" % (v, name)
            if key in sys.modules:
                mods.append(sys.modules[key])
                continue
            spec = importlib.util.spec_from_file_location(name, p)
            m = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(m)
            sys.modules[key] = m
            mods.append(m)
        return mods[0], mods[1], v
    return None
