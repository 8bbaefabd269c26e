"""The backward of the concat / difference volumes (shift_volume_bwd_kernel, regress.cu) and the autograd
path of volume.concat_volume / diff_volume.

The kernels sum in fp32, d ascending from 0, one thread per output element, so their gradients equal the
ordered NumPy restatement (tests/_volume_ref.py) bit for bit, on the 128-bit path (W % 4 == 0, every base
16-byte aligned) and on the scalar path (W % 4 != 0, or a base 4 bytes past alignment).  Through autograd
they agree with float64 autograd of PSMNet's slice-assignment construction within the recursive-summation
bound.  G at masked voxels (x < d) never reaches a gradient, whatever it holds.
"""
import numpy as np
import pytest

from tests import _volume_ref as V
from tests.test_gpu_regression import VOLUME_CASES

pytestmark = pytest.mark.gpu

# (N, C, H, W, D): the forward's edge shapes, plus config P's per-sample shape (batch 16 in the benchmark)
CASES = dict(VOLUME_CASES, **{"P-shaped": (2, 32, 136, 240, 48)})
# which buffer sits 4 bytes past 16-byte alignment (forcing the scalar path); "aligned" is the 128-bit path
LAYOUTS = ["aligned", "grad+4", "out+4"]


@pytest.fixture(scope="module")
def ms():
    import msnets_b200
    assert msnets_b200.device_count() >= 1
    return msnets_b200


def _buffer(shape, fill, misaligned):
    import torch
    n = int(np.prod(shape))
    if not misaligned:
        return torch.full(shape, fill, dtype=torch.float32, device="cuda")
    t = torch.full((n + 1,), fill, dtype=torch.float32, device="cuda")[1:].view(shape)
    assert t.is_contiguous() and t.data_ptr() % 16 == 4
    return t


def _grad_volume(shape, seed, misaligned=False):
    """A seeded N(0,1) gradient volume on the device (optionally misaligned) and its host copy."""
    import torch
    gen = torch.Generator(device="cuda").manual_seed(seed)
    g = torch.randn(shape, generator=gen, device="cuda")
    if misaligned:
        gm = _buffer(shape, 0.0, True)
        gm.copy_(g)
        g = gm
    return g


def _raw_backward(g, N, C, H, W, D, diff, want=(True, True), out_misaligned=False):
    """One call of the backward entry point; outputs pre-filled with NaN so an unwritten element shows."""
    import torch
    from msnets_b200 import _lib
    gfl = _buffer((N, C, H, W), float("nan"), out_misaligned) if want[0] else None
    gfr = _buffer((N, C, H, W), float("nan"), out_misaligned) if want[1] else None
    L = _lib.lib()
    fn = L.msn_diff_volume_backward_dev if diff else L.msn_concat_volume_backward_dev
    _lib.check(fn(g.data_ptr(), N, C, H, W, D, gfl.data_ptr() if gfl is not None else None,
                  gfr.data_ptr() if gfr is not None else None, torch.cuda.current_stream().cuda_stream))
    return gfl, gfr


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("diff", [False, True], ids=["concat", "diff"])
@pytest.mark.parametrize("case", list(CASES))
def test_backward_bit_exact_against_ordered_sum(ms, case, diff, layout):
    N, C, H, W, D = CASES[case]
    g = _grad_volume((N, C if diff else 2 * C, D, H, W), seed=sum(CASES[case]) + diff,
                     misaligned=layout == "grad+4")
    want_l, want_r = V.volume_backward(g.cpu().numpy(), diff)
    gfl, gfr = _raw_backward(g, N, C, H, W, D, diff, out_misaligned=layout == "out+4")
    assert np.array_equal(gfl.cpu().numpy(), want_l)
    assert np.array_equal(gfr.cpu().numpy(), want_r)
    # either output alone: the same bits, and the other buffer is not needed
    assert np.array_equal(_raw_backward(g, N, C, H, W, D, diff, (True, False))[0].cpu().numpy(), want_l)
    assert np.array_equal(_raw_backward(g, N, C, H, W, D, diff, (False, True))[1].cpu().numpy(), want_r)


@pytest.mark.parametrize("layout", ["aligned", "grad+4"])
@pytest.mark.parametrize("diff", [False, True], ids=["concat", "diff"])
@pytest.mark.parametrize("case", ["D>=W", "W%4=1", "P-shaped"])
def test_masked_voxels_never_reach_the_gradient(ms, case, diff, layout):
    import torch
    N, C, H, W, D = CASES[case]
    shape = (N, C if diff else 2 * C, D, H, W)
    g = _grad_volume(shape, seed=7 + diff, misaligned=layout == "grad+4")
    ref = [t.cpu().numpy() for t in _raw_backward(g, N, C, H, W, D, diff)]
    m = torch.from_numpy(np.ascontiguousarray(V.masked(shape))).cuda()
    for junk in (float("nan"), 1e30, -1e30):
        g.masked_fill_(m, junk)
        got = [t.cpu().numpy() for t in _raw_backward(g, N, C, H, W, D, diff)]
        assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]), junk


@pytest.mark.parametrize("diff", [False, True], ids=["concat", "diff"])
@pytest.mark.parametrize("case", list(CASES))
def test_autograd_agrees_with_float64(ms, case, diff):
    """(vol * w).sum().backward() against float64 autograd of the slice-assignment construction, per element
    within gamma_{k-1} * sum |terms|."""
    import torch
    N, C, H, W, D = CASES[case]
    rng = np.random.default_rng(100 + sum(CASES[case]) + diff)
    fl = torch.from_numpy(rng.standard_normal((N, C, H, W)).astype(np.float32))
    fr = torch.from_numpy(rng.standard_normal((N, C, H, W)).astype(np.float32))
    w = rng.standard_normal((N, C if diff else 2 * C, D, H, W)).astype(np.float32)
    a, b = fl.cuda().requires_grad_(True), fr.cuda().requires_grad_(True)
    build = ms.volume.diff_volume if diff else ms.volume.concat_volume
    vol = build(a, b, D)
    assert vol.grad_fn is not None
    (vol * torch.from_numpy(w).cuda()).sum().backward()
    a64, b64 = fl.double().requires_grad_(True), fr.double().requires_grad_(True)
    (V.torch_volume(a64, b64, D, diff) * torch.from_numpy(w).double()).sum().backward()
    bl, br = V.summation_bounds(w, diff)
    for got, want, bound, name in ((a.grad, a64.grad, bl, "fl"), (b.grad, b64.grad, br, "fr")):
        err = np.abs(got.cpu().double().numpy() - want.numpy())
        assert (err <= bound).all(), "%s: %d elements over the bound" % (name, int((err > bound).sum()))


@pytest.mark.parametrize("diff", [False, True], ids=["concat", "diff"])
def test_one_input_requiring_grad(ms, diff, monkeypatch):
    """Only fl (or only fr) requires grad: the other's .grad stays None, the entry point gets NULL for it, and
    the gradient that is computed has the bits of the two-sided call."""
    import torch
    from msnets_b200 import _lib
    N, C, H, W, D = CASES["W%4=1"]
    rng = np.random.default_rng(5)
    fl = torch.from_numpy(rng.standard_normal((N, C, H, W)).astype(np.float32)).cuda()
    fr = torch.from_numpy(rng.standard_normal((N, C, H, W)).astype(np.float32)).cuda()
    w = torch.from_numpy(rng.standard_normal((N, C if diff else 2 * C, D, H, W)).astype(np.float32)).cuda()
    build = ms.volume.diff_volume if diff else ms.volume.concat_volume

    def grads(l_grad, r_grad):
        a, b = fl.clone().requires_grad_(l_grad), fr.clone().requires_grad_(r_grad)
        (build(a, b, D) * w).sum().backward()
        return a.grad, b.grad

    both = grads(True, True)
    real = _lib.lib()
    name = "msn_diff_volume_backward_dev" if diff else "msn_concat_volume_backward_dev"
    calls = []

    class Spy:
        def __getattr__(self, attr):
            fn = getattr(real, attr)
            if attr != name:
                return fn

            def spy(*args):
                calls.append(args)
                return fn(*args)
            return spy

    monkeypatch.setattr(_lib, "lib", lambda: Spy())
    only_l = grads(True, False)
    only_r = grads(False, True)
    assert len(calls) == 2
    assert calls[0][6] is not None and calls[0][7] is None
    assert calls[1][6] is None and calls[1][7] is not None
    assert only_l[1] is None and only_r[0] is None
    assert torch.equal(only_l[0], both[0]) and torch.equal(only_r[1], both[1])


def test_backward_is_deterministic(ms):
    import torch
    N, C, H, W, D = CASES["P-shaped"]
    for diff in (False, True):
        g = _grad_volume((N, C if diff else 2 * C, D, H, W), seed=11)
        r1 = _raw_backward(g, N, C, H, W, D, diff)
        r2 = _raw_backward(g, N, C, H, W, D, diff)
        torch.cuda.synchronize()
        for a, b in zip(r1, r2):
            assert np.array_equal(a.cpu().numpy().view(np.int32), b.cpu().numpy().view(np.int32))


@pytest.mark.parametrize("diff", [False, True], ids=["concat", "diff"])
def test_inference_path_unchanged(ms, oracle, diff):
    """Under torch.no_grad() inputs that require grad give a plain volume, bitwise the oracle's forward;
    out= with autograd raises; double backward raises."""
    import torch
    N, C, H, W, D = CASES["D%d_chunk!=0"]
    rng = np.random.default_rng(9)
    fl = rng.standard_normal((N, C, H, W)).astype(np.float32)
    fr = rng.standard_normal((N, C, H, W)).astype(np.float32)
    a, b = torch.from_numpy(fl).cuda().requires_grad_(True), torch.from_numpy(fr).cuda().requires_grad_(True)
    build = ms.volume.diff_volume if diff else ms.volume.concat_volume
    want = (oracle.diff_volume if diff else oracle.concat_volume)(fl, fr, D)
    with torch.no_grad():
        vol = build(a, b, D)
    assert vol.grad_fn is None and not vol.requires_grad
    assert np.array_equal(vol.cpu().numpy(), want)
    assert np.array_equal(build(a.detach(), b.detach(), D).cpu().numpy(), want)
    with torch.no_grad():
        out = torch.empty_like(vol)
        assert build(a, b, D, out=out) is out
    with pytest.raises(ValueError, match="out="):
        build(a, b, D, out=torch.empty_like(vol))
    vol = build(a, b, D)
    assert np.array_equal(vol.detach().cpu().numpy(), want)
    ga, = torch.autograd.grad((vol * vol).sum(), a, create_graph=True)
    with pytest.raises(RuntimeError, match="once_differentiable"):
        ga.sum().backward()


def test_psmnet_shaped_training_step(ms):
    """Conv2d features -> concat_volume -> Conv3d -> squeeze -> soft_argmin -> smooth-L1 -> backward: the
    Conv2d weight gradient matches the same step built with the slice-assignment loop."""
    import torch
    import torch.nn.functional as F
    torch.manual_seed(0)
    N, H, W, D = 2, 32, 64, 48
    D4 = D // 4
    feat = torch.nn.Conv2d(3, 8, 3, stride=4, padding=1).cuda()
    agg = torch.nn.Conv3d(16, 1, 3, padding=1).cuda()
    left, right = torch.randn((N, 3, H, W), device="cuda"), torch.randn((N, 3, H, W), device="cuda")
    target = torch.rand((N, H // 4, W // 4), device="cuda") * (D4 - 1)

    def step(make_volume):
        feat.zero_grad()
        agg.zero_grad()
        vol = make_volume(feat(left), feat(right), D4)
        disp = ms.regression.soft_argmin(agg(vol).squeeze(1))
        F.smooth_l1_loss(disp, target).backward()
        return feat.weight.grad.clone(), agg.weight.grad.clone()

    saved = torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic
    torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic = False, True
    try:
        got = step(ms.volume.concat_volume)
        want = step(V.torch_concat_volume)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cudnn.deterministic = saved
    for g, w in zip(got, want):
        assert float(w.abs().max()) > 0
        assert float((g - w).abs().max()) <= 1e-5 * max(1.0, float(w.abs().max()))
