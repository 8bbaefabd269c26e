"""GPU: the pre-matching image ops and the two generator entry points at the reference's DEFAULT operating
point (ds_scale = 2): SURVEY.md 8f-1 / 8f-2.

  rescale_u8 / down_sampling_input   cbmv_generator.py:465-482   uint8 result identical to the oracle's
                                     (scipy.ndimage-backed restatement of skimage.transform.rescale;
                                     skimage itself is not installed: parity pinned to scipy, not skimage)
  generate_test_cbmv                 :727-861   against the UNMODIFIED reference function run over the
  generate_crop_train_cbmv           :549-725   unmodified reference C++ (oracle/_ref), its skimage call
                                                served by the oracle's rescale; same `random` seed -> same crop
"""
import os
import random
import tempfile

import numpy as np
import pytest

from tests._synth import assert_aml_close, synth_pair

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ms():
    import msnets_b200
    assert msnets_b200.device_count() >= 1
    return msnets_b200


@pytest.fixture(scope="module")
def refgen(oracle):
    """Unmodified cbmv_generator.py over the unmodified reference C++ (or the C oracle when _ref is absent);
    the oracle's restated glue when cbmv_generator.py is absent."""
    from oracle import ref_glue
    ref = oracle.load_ref()
    if ref is not None:
        mtc, fte = ref[0], ref[1]
    else:
        oracle.lib()
        mtc, fte = oracle.MTC, oracle.FTE
    g = ref_glue.load_generator(mtc, fte, rescale=oracle.rescale_antialiased)
    if g is None:
        g = ref_glue.restated_generator(mtc, fte)
    return g


@pytest.mark.parametrize("shape,scale", [((64, 96), 0.5), ((37, 53), 0.5), ((40, 60), 0.25), ((280, 704), 0.5),
                                         ((384, 1248), 0.5), ((31, 64), 0.5)])
def test_rescale_matches_oracle_bit_for_bit(ms, oracle, shape, scale):
    import torch
    rng = np.random.default_rng(shape[0] * 1000 + shape[1])
    a = rng.integers(0, 256, shape, dtype=np.uint8)
    b = np.maximum(rng.integers(0, 256, shape, dtype=np.uint8), 23).astype(np.uint8)   # minimum > 0: the clip lifts the border
    b[shape[0] // 2:, : shape[1] // 3] = 200                                           # flat block
    wa, wb = oracle.down_sampling_input(scale, a, b)
    ga, gb = ms.cbmv.down_sampling_input(scale, a, b)                                  # NumPy -> host C ABI
    assert ga.dtype == np.uint8 and np.array_equal(ga, wa) and np.array_equal(gb, wb)
    t = torch.from_numpy(np.stack([a, b])).cuda()                                      # batched device path
    gt = ms.cbmv.rescale_u8(t, scale).cpu().numpy()
    assert np.array_equal(gt[0], wa) and np.array_equal(gt[1], wb)


def _write_pfm(path, img):
    with open(path, "wb") as f:
        f.write(b"Pf\n%d %d\n-1.0\n" % (img.shape[1], img.shape[0]))
        np.flipud(img).astype("<f4").tofile(f)


@pytest.mark.parametrize("left_only", [True, False])
def test_generate_test_cbmv_reference_default_ds_scale_2(ms, refgen, left_only):
    import cv2
    L, R = synth_pair(150, 420, 5, 6)
    with tempfile.TemporaryDirectory() as td:
        fl, fr = os.path.join(td, "l.png"), os.path.join(td, "r.png")
        cv2.imwrite(fl, L)
        cv2.imwrite(fr, R)
        want, h, w, ch, cw = refgen.generate_test_cbmv(fl, fr, encoder_ds=16, maxdisp=48, is_left_only=left_only)
        got, h2, w2, ch2, cw2 = ms.cbmv.generate_test_cbmv(fl, fr, encoder_ds=16, maxdisp=48, is_left_only=left_only)
    assert (h, w, ch, cw) == (h2, w2, ch2, cw2) == (150, 420, 160, 432)
    want, got = want.numpy(), got.cpu().numpy()
    assert got.shape == want.shape == (8 if left_only else 16, 24, 80, 216)
    for lo in range(0, got.shape[0], 8):
        assert np.array_equal(got[lo:lo + 4], want[lo:lo + 4])
        assert_aml_close(got[lo + 4:lo + 8], want[lo + 4:lo + 8])


@pytest.mark.parametrize("ds,left_only,fixed", [(2, True, False), (2, False, False), (1, True, True), (2, True, True)])
def test_generate_crop_train_cbmv_matches_reference(ms, refgen, ds, left_only, fixed):
    import cv2
    if not hasattr(refgen, "generate_crop_train_cbmv"):
        pytest.skip("cbmv_generator.py not available; generate_crop_train_cbmv has no restatement in oracle/")
    L, R = synth_pair(200, 620, 9, 8)
    disp = (np.arange(200 * 620, dtype=np.float32).reshape(200, 620) % 97) / 2
    disp[5, 7] = np.inf
    ad = refgen.get_default_args_dict()
    ad["ds_scale"] = ds
    with tempfile.TemporaryDirectory() as td:
        fl, fr, fd = os.path.join(td, "l.png"), os.path.join(td, "r.png"), os.path.join(td, "d.pfm")
        cv2.imwrite(fl, L)
        cv2.imwrite(fr, R)
        _write_pfm(fd, disp)
        random.seed(4242)
        want = refgen.generate_crop_train_cbmv(fl, fr, fd, None, crop_height=96, crop_width=192, maxdisp=64,
                                               is_fixed_center_around_crop=fixed, args_dict=ad, is_left_only=left_only)
        random.seed(4242)
        got = ms.cbmv.generate_crop_train_cbmv(fl, fr, fd, None, crop_height=96, crop_width=192, maxdisp=64,
                                               is_fixed_center_around_crop=fixed, args_dict=ad, is_left_only=left_only)
    assert len(want) == len(got) == 5
    fw, fg = want[0].numpy(), got[0].cpu().numpy()
    assert fg.shape == fw.shape == ((8 if left_only else 16), 64 // ds, 96 // ds, 192 // ds)
    for lo in range(0, fg.shape[0], 8):
        assert np.array_equal(fg[lo:lo + 4], fw[lo:lo + 4])
        assert_aml_close(fg[lo + 4:lo + 8], fw[lo + 4:lo + 8])
    for k in range(1, 5):                                   # disparity crop, the two RGB crops, the label
        assert got[k].dtype == want[k].dtype and tuple(got[k].shape) == tuple(want[k].shape)
        assert np.array_equal(got[k].numpy(), want[k].numpy())
