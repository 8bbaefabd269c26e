"""The regression kernels of regress.cu against a float64 reference of the same operation.

soft-argmin (modes 0 / 1 / 2 of soft_argmin_kernel), its backward and the slab merge replace
F.softmax + disparityregression in training, so their results and gradients are held to
float64 torch on the CPU, computed from the very fp32 tensor the kernel read:

    p = softmax(x.double(), 1);  disp = sum_d d * p_d;  gradients by float64 autograd.

Bars: forward, expectation and merge within SOFTARGMIN_ATOL px, NaN exactly where the
reference is NaN; backward within 1e-5 * max(1, max |grad|) (test_gpu_parity.py's
test_soft_argmin_autograd), and exactly 0 at masked (-inf) logits.  The 128-bit and the scalar
load paths do the same per-pixel operations in the same order, so they agree bit for bit, and so
does the host entry with the device entry.

Contract: -inf masks a disparity, as with torch's softmax.  A column that is -inf at every
disparity has no distribution: its disparity (and gradient) is NaN, as torch gives.

Each call packs many logit families into one tensor, one family per image row, so a failure
names every family that missed and by how much.  They target the kernel's edges: D around its
chunk of 8 disparities, logits far from 0 (the exponent must be formed as (x - max) * log2(e):
with fma(x, log2(e), -fl(max * log2(e))) the rounding of the product grows with |max| and differs
between chunks, up to 2e-2 px at an offset of 1e4 and D = 192 in an fp32 emulation), -inf runs
that fill whole chunks and slabs, one-hot peaks and exact ties.

The volume builders (concat / diff) are held bit for bit to the oracle at their edges.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SOFTARGMIN_ATOL = 1e-3      # px, the project's soft-argmin bar (README, DESIGN.md section 5)
GRAD_RTOL = 1e-5            # of max(1, max |grad|)

DS = [1, 2, 7, 8, 9, 16, 47, 48, 192, 193, 640]

# name -> (N, W, misaligned).  H is the number of logit families.  "vec": HW % 4 == 0 and a 16-byte aligned
# base, the float4 path; "scalar": HW odd; "offset": HW % 4 == 0 but the base 4 bytes past alignment,
# which also takes the scalar path.
LAYOUTS = {"vec-n1": (1, 8, False), "vec-n3": (3, 8, False), "scalar-n1": (1, 7, False),
           "scalar-n3": (3, 7, False), "offset-n1": (1, 8, True), "offset-n3": (3, 8, True)}


@pytest.fixture(scope="module")
def ms():
    import msnets_b200
    assert msnets_b200.device_count() >= 1
    return msnets_b200


def _families(D, N, W, seed):
    """[(name, float64 logits [N, D, W])]: the logit families, each a column set of its own."""
    rng = np.random.default_rng(seed)

    def randn(sigma=4.0):
        return rng.standard_normal((N, D, W)) * sigma

    n_idx, w_idx = np.meshgrid(np.arange(N), np.arange(W), indexing="ij")
    fam = []
    for sigma in (0.01, 1.0, 4.0, 30.0):
        fam.append(("randn*%g" % sigma, randn(sigma)))
        for c in (-1e4, -1e3, 1e3, 1e4):
            fam.append(("randn*%g%+g" % (sigma, c), randn(sigma) + c))
    for d in sorted({0, 7, 8, D - 1}):
        if d < D:
            x = np.zeros((N, D, W))
            x[:, d] = 60.0                                   # every other weight is e^-60
            fam.append(("one-hot d=%d" % d, x))
    if D >= 2:
        a, b = rng.choice(D, 2, replace=False)
        x = randn(1.0)
        x[:, a] = x[:, b] = 25.0
        fam.append(("tie d=%d,%d" % (a, b), x))
    for k in (1, 7, 8, 9, 16):
        if k < D:
            x = randn()
            x[:, :k] = -np.inf
            fam.append(("leading -inf x%d" % k, x))
            x = randn()
            x[:, D - k:] = -np.inf
            fam.append(("trailing -inf x%d" % k, x))
    if D > 9:
        x = randn() + 1e3
        x[:, :9] = -np.inf
        fam.append(("leading -inf x9 +1000", x))
    if D >= 2:
        x = randn()
        mask = rng.random((N, D, W)) < 0.6
        mask[n_idx, rng.integers(0, D, (N, W)), w_idx] = False   # one finite logit per column at least
        x[mask] = -np.inf
        fam.append(("scattered -inf", x))
    x = np.full((N, D, W), -np.inf)
    x[n_idx, rng.integers(0, D, (N, W)), w_idx] = rng.standard_normal((N, W)) * 4
    fam.append(("one finite logit", x))
    fam.append(("all -inf", np.full((N, D, W), -np.inf)))
    return fam


def _pack(fam, W):
    """-> (names, float32 CPU tensor [N, D, F, W]); F is made odd when W is odd, so that HW is odd."""
    import torch
    if W % 2 and len(fam) % 2 == 0:
        fam = fam + [("randn*4 (row padding)", np.random.default_rng(1).standard_normal(fam[0][1].shape) * 4)]
    names = [n for n, _ in fam]
    x = np.stack([f for _, f in fam], axis=2).astype(np.float32)
    return names, torch.from_numpy(x)


def _logits(D, layout, seed):
    N, W, misaligned = LAYOUTS[layout]
    names, x = _pack(_families(D, N, W, seed), W)
    return names, x, misaligned


def _to_device(x, misaligned):
    """A contiguous CUDA copy of x; misaligned: its base pointer 4 bytes past 16-byte alignment."""
    import torch
    if not misaligned:
        return x.cuda()
    y = torch.empty(x.numel() + 1, dtype=torch.float32, device="cuda")[1:].view(x.shape)
    y.copy_(x)
    assert y.is_contiguous() and y.data_ptr() % 16 == 4
    return y


def _ref_disp(x):
    """float64 softmax over dim 1 of a CPU tensor [N, D, H, W], then the expectation of d."""
    import torch
    p = torch.softmax(x.double(), 1)
    return _ref_expect(p)


def _ref_expect(p):
    import torch
    d = torch.arange(p.shape[1], dtype=torch.float64).view(1, -1, 1, 1)
    return (p.double() * d).sum(1)


def _bits(t):
    return t.detach().cpu().numpy().view(np.int32) if hasattr(t, "detach") else t.view(np.int32)


def _check_disp(got, want, names, atol=SOFTARGMIN_ATOL):
    """got / want [N, F, W]: per family, NaN exactly where the reference is NaN and |got - want| <= atol."""
    got = got.detach().cpu().double().numpy() if hasattr(got, "detach") else np.asarray(got, np.float64)
    want = want.numpy()
    bad = []
    for f, name in enumerate(names):
        g, w = got[:, f], want[:, f]
        if not np.array_equal(np.isnan(g), np.isnan(w)):
            bad.append("%s: %d NaN, reference %d NaN of %d" % (name, np.isnan(g).sum(), np.isnan(w).sum(), g.size))
            continue
        ok = ~np.isnan(w)
        err = float(np.abs(g[ok] - w[ok]).max()) if ok.any() else 0.0
        if not err <= atol:
            bad.append("%s: max error %.3g px" % (name, err))
    assert not bad, "%d of %d families fail: %s" % (len(bad), len(names), "; ".join(bad))


def _assert_all_masked_is_nan(want, names):
    assert np.isnan(want[:, names.index("all -inf")].numpy()).all()


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("D", DS)
def test_soft_argmin_matches_float64(ms, D, layout):
    """regression.soft_argmin (mode 0), device and host entries, both load paths."""
    names, x, misaligned = _logits(D, layout, seed=D)
    want = _ref_disp(x)
    _assert_all_masked_is_nan(want, names)
    got = ms.regression.soft_argmin(_to_device(x, misaligned))
    _check_disp(got, want, names)
    if misaligned:      # the same data through the float4 path when HW % 4 == 0: the same bits
        assert np.array_equal(_bits(got), _bits(ms.regression.soft_argmin(x.cuda())))
    assert np.array_equal(_bits(ms.regression.soft_argmin(x.numpy())), _bits(got))


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("D", DS)
def test_expected_disparity_matches_float64(ms, D, layout):
    """regression.expected_disparity and the disparityregression module (mode 2) on float64-softmax
    probabilities rounded to fp32."""
    import torch
    names, x, misaligned = _logits(D, layout, seed=1000 + D)
    p = torch.softmax(x.double(), 1).float()
    want = _ref_expect(p)
    _assert_all_masked_is_nan(want, names)
    pd = _to_device(p, misaligned)
    got = ms.regression.expected_disparity(pd)
    _check_disp(got, want, names)
    assert np.array_equal(_bits(ms.regression.disparityregression(D)(pd)), _bits(got))
    if misaligned:
        assert np.array_equal(_bits(ms.regression.expected_disparity(p.cuda())), _bits(got))


def _slab_families(D, N, W, P, seed):
    from msnets_b200 import sharding
    fam = _families(D, N, W, seed)
    rng = np.random.default_rng(seed + 1)
    if P > 1:
        for r in range(P):
            b, c = sharding.shard_range(D, r, P)
            x = rng.standard_normal((N, D, W)) * 4
            x[:, b:b + c] -= 200.0                  # this slab's scale underflows to 0 in the merge
            fam.append(("slab %d 200 below" % r, x))
            x = rng.standard_normal((N, D, W)) * 4
            x[:, b:b + c] = -np.inf
            fam.append(("slab %d all -inf" % r, x))
    return fam


@pytest.mark.parametrize("layout", ["vec-n3", "scalar-n1"])
@pytest.mark.parametrize("D,P", [(D, P) for D in DS for P in (1, 2, 3, 8) if P <= D])
def test_slab_partials_and_merge_match_float64(ms, D, P, layout):
    """msn_soft_argmin_partial_dev (mode 1) on the uneven disparity cuts of sharding.shard_range, then
    msn_soft_argmin_merge_dev; slabs one disparity wide when P is close to D."""
    import torch
    from msnets_b200 import _lib, sharding
    N, W, _ = LAYOUTS[layout]
    names, x = _pack(_slab_families(D, N, W, P, seed=2000 + D), W)
    want = _ref_disp(x)
    _assert_all_masked_is_nan(want, names)
    xd = x.cuda()
    H = x.shape[2]
    L = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    parts = torch.empty((P, N, 3, H, W), dtype=torch.float32, device="cuda")
    for r in range(P):
        b, c = sharding.shard_range(D, r, P)
        slab = xd[:, b:b + c].contiguous()
        _lib.check(L.msn_soft_argmin_partial_dev(slab.data_ptr(), N, c, H, W, b, parts[r].data_ptr(), st))
    disp = torch.empty((N, H, W), dtype=torch.float32, device="cuda")
    _lib.check(L.msn_soft_argmin_merge_dev(parts.data_ptr(), P, N, H, W, disp.data_ptr(), st))
    _check_disp(disp, want, names)


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("D", DS)
def test_soft_argmin_backward_matches_float64(ms, D, layout):
    """The autograd backward (msn_soft_argmin_backward_dev) against float64 autograd of softmax + expectation."""
    import torch
    names, x, misaligned = _logits(D, layout, seed=3000 + D)
    w = torch.from_numpy(np.random.default_rng(D).standard_normal((x.shape[0],) + tuple(x.shape[2:]))
                         .astype(np.float32))
    xd = _to_device(x, misaligned).requires_grad_(True)
    disp = ms.regression.soft_argmin(xd)
    assert disp.grad_fn is not None
    (disp * w.cuda()).sum().backward()
    got = xd.grad.cpu().double().numpy()
    xr = x.double().requires_grad_(True)
    (_ref_disp(xr) * w.double()).sum().backward()
    want = xr.grad.numpy()
    all_masked = np.isneginf(x.numpy()).all(axis=1, keepdims=True) & np.ones_like(want, bool)
    assert np.isnan(want[all_masked]).all() and not np.isnan(want[~all_masked]).any()
    tol = GRAD_RTOL * max(1.0, float(np.abs(want[~all_masked]).max()))
    masked = np.isneginf(x.numpy()) & ~all_masked
    bad = []
    for f, name in enumerate(names):
        g, r, m, a = got[:, :, f], want[:, :, f], masked[:, :, f], all_masked[:, :, f]
        if not np.array_equal(np.isnan(g), a):
            bad.append("%s: %d NaN gradients, reference %d" % (name, np.isnan(g).sum(), a.sum()))
            continue
        if not (g[m] == 0).all():
            bad.append("%s: %d nonzero gradients at -inf logits" % (name, int((g[m] != 0).sum())))
        err = float(np.abs(g[~a] - r[~a]).max()) if (~a).any() else 0.0
        if not err <= tol:
            bad.append("%s: max error %.3g (bar %.3g)" % (name, err, tol))
    assert not bad, "%d of %d families fail: %s" % (len(bad), len(names), "; ".join(bad))


def test_out_is_checked(ms):
    """out= must be a contiguous float32 [N,H,W] tensor on the logits' device; anything else would be
    written through as raw memory."""
    import torch
    x = torch.randn((2, 5, 3, 4), device="cuda")
    want = ms.regression.soft_argmin(x)
    for fn in (ms.regression.soft_argmin, ms.regression.expected_disparity):
        for bad in (torch.empty((2, 3, 5), device="cuda"),
                    torch.empty((2, 3), device="cuda"),
                    torch.empty((2, 3, 4), dtype=torch.float64, device="cuda"),
                    torch.empty((2, 4, 3), device="cuda").transpose(1, 2),
                    torch.empty((2, 3, 4))):
            with pytest.raises(ValueError):
                fn(x, out=bad)
        out = torch.empty((2, 3, 4), device="cuda")
        assert fn(x, out=out) is out
    assert torch.equal(ms.regression.soft_argmin(x, out=torch.empty((2, 3, 4), device="cuda")), want)


def _d_chunk(N, C, H, W, D):
    """launch_shift_volume's split of D over blockIdx.y (regress.cu)."""
    gx = -(-H * ((W + 3) // 4) // 256)
    chunks = 1
    while chunks < D and gx * N * C * chunks < 4 * 148 * 8:
        chunks *= 2
    return -(-D // chunks)


# (N, C, H, W, D)
VOLUME_CASES = {"D>=W": (2, 3, 5, 6, 9), "D=1": (1, 4, 7, 16, 1), "W%4=1": (2, 3, 6, 13, 8),
                "D%d_chunk!=0": (2, 4, 300, 61, 45)}


@pytest.mark.parametrize("misaligned_out", [False, True])
@pytest.mark.parametrize("case", list(VOLUME_CASES))
def test_volume_builders_edges_bit_exact(ms, oracle, case, misaligned_out):
    """concat_volume / diff_volume bit for bit against the oracle: every column masked at high d, one
    disparity, ragged rows, a D split unevenly across blockIdx.y, and an out= tensor 4 bytes past 16-byte
    alignment (the scalar-store path).  out= is pre-filled with NaN, so a voxel left unwritten shows."""
    import torch
    N, C, H, W, D = VOLUME_CASES[case]
    if case == "D%d_chunk!=0":
        assert D % _d_chunk(N, C, H, W, D) != 0
    rng = np.random.default_rng(sum(VOLUME_CASES[case]))
    fl = rng.standard_normal((N, C, H, W)).astype(np.float32)
    fr = rng.standard_normal((N, C, H, W)).astype(np.float32)
    tl, tr = torch.from_numpy(fl).cuda(), torch.from_numpy(fr).cuda()
    for fn, ofn, c_out in ((ms.volume.concat_volume, oracle.concat_volume, 2 * C),
                           (ms.volume.diff_volume, oracle.diff_volume, C)):
        out = _to_device(torch.full((N, c_out, D, H, W), float("nan")), misaligned_out)
        assert fn(tl, tr, D, out=out) is out
        assert np.array_equal(out.cpu().numpy(), ofn(fl, fr, D))
