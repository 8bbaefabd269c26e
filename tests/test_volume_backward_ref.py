"""CPU: the ordered fp32 backward of the concat / difference volumes (tests/_volume_ref.py), which the
GPU tests hold the kernels to bit for bit, against float64 torch autograd of PSMNet's slice-assignment
construction.  Per element the error is within the recursive-summation bound gamma_{k-1} * sum |terms|
(k = the element's term count), and G at masked voxels (x < d), NaN here, never reaches a gradient."""
import numpy as np
import pytest

from tests import _volume_ref as V
from tests.test_gpu_regression import VOLUME_CASES

CASES = dict(VOLUME_CASES, **{"D=W": (1, 2, 3, 8, 8)})


def _float64_grads(g, N, C, H, W, D, diff):
    import torch
    fl = torch.zeros((N, C, H, W), dtype=torch.float64, requires_grad=True)
    fr = torch.zeros((N, C, H, W), dtype=torch.float64, requires_grad=True)
    (V.torch_volume(fl, fr, D, diff) * torch.from_numpy(g.astype(np.float64))).sum().backward()
    return fl.grad.numpy(), fr.grad.numpy()


@pytest.mark.parametrize("diff", [False, True], ids=["concat", "diff"])
@pytest.mark.parametrize("case", list(CASES))
def test_ordered_backward_matches_float64_autograd(case, diff):
    N, C, H, W, D = CASES[case]
    rng = np.random.default_rng(sum(CASES[case]) + diff)
    g = rng.standard_normal((N, C if diff else 2 * C, D, H, W)).astype(np.float32)
    want_l, want_r = _float64_grads(g, N, C, H, W, D, diff)
    g_nan = g.copy()
    g_nan[V.masked(g.shape)] = np.nan
    got_l, got_r = V.volume_backward(g_nan, diff)
    assert got_l.dtype == np.float32 and got_r.dtype == np.float32
    assert not np.isnan(got_l).any() and not np.isnan(got_r).any()
    bl, br = V.summation_bounds(g, diff)
    assert (np.abs(got_l - want_l) <= bl).all()
    assert (np.abs(got_r - want_r) <= br).all()
    # the same bits from the NaN-free gradient: masked voxels are not read
    for a, b in zip(V.volume_backward(g, diff), (got_l, got_r)):
        assert np.array_equal(a, b)


def test_term_counts_are_the_slices_that_reach_each_column():
    """k(x) of the summation bound counts the disparities whose slice assignment covers the column."""
    import torch
    W, D = 7, 10
    fl = torch.zeros((1, 1, 1, W), dtype=torch.float64, requires_grad=True)
    fr = torch.zeros((1, 1, 1, W), dtype=torch.float64, requires_grad=True)
    V.torch_concat_volume(fl, fr, D).sum().backward()
    kl, kr = V.term_counts(W, D)
    assert np.array_equal(fl.grad.numpy()[0, 0, 0], kl) and np.array_equal(fr.grad.numpy()[0, 0, 0], kr)
