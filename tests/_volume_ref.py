"""References for the backward of the concat / difference volumes (volume.concat_volume, diff_volume).

With G the gradient of the volume (oracle/ms_oracle.py:concat_volume / diff_volume for the forward):

    concat: gfl[n,c,y,x]  = sum_{d=0..min(x, D-1)}      G[n,  c, d, y, x]
            gfr[n,c,y,x'] = sum_{d=0..min(W-1-x', D-1)} G[n, C+c, d, y, x'+d]
    diff:   gfl as concat, gfr = -sum_{d=0..min(W-1-x', D-1)} G[n, c, d, y, x'+d]

`concat_volume_backward` / `diff_volume_backward` restate these as the kernel orders them: a float32
accumulator starting at 0, one rounding per add, d ascending; masked voxels (x < d) are never read.
`torch_concat_volume` / `torch_diff_volume` are PSMNet's slice-assignment construction, the stock-PyTorch
path whose autograd is the float64 reference.
"""
import numpy as np


def _sum_left(g):
    """g [N,C,D,H,W] -> [N,C,H,W]: acc[..., x] += g[:, :, d, :, x] for x >= d, d ascending."""
    N, C, D, H, W = g.shape
    acc = np.zeros((N, C, H, W), g.dtype)
    for d in range(min(D, W)):
        acc[..., d:] += g[:, :, d, :, d:]
    return acc


def _sum_right(g):
    """g [N,C,D,H,W] -> [N,C,H,W]: acc[..., x'] += g[:, :, d, :, x'+d] for x'+d < W, d ascending."""
    N, C, D, H, W = g.shape
    acc = np.zeros((N, C, H, W), g.dtype)
    for d in range(min(D, W)):
        acc[..., :W - d] += g[:, :, d, :, d:]
    return acc


def concat_volume_backward(g):
    """g float32 [N,2C,D,H,W] -> (gfl, gfr) float32 [N,C,H,W]."""
    C = g.shape[1] // 2
    return _sum_left(g[:, :C]), _sum_right(g[:, C:])


def diff_volume_backward(g):
    """g float32 [N,C,D,H,W] -> (gfl, gfr) float32 [N,C,H,W]; gfr is the negated sum."""
    return _sum_left(g), -_sum_right(g)


def volume_backward(g, diff):
    return diff_volume_backward(g) if diff else concat_volume_backward(g)


def masked(shape):
    """Boolean mask of the voxels x < d of a volume shape [N,C',D,H,W] (the forward writes 0 there)."""
    D, W = shape[2], shape[4]
    m = np.arange(W)[None, :] < np.arange(D)[:, None]            # [D, W]
    return np.broadcast_to(m[None, None, :, None, :], shape)


def term_counts(W, D):
    """Number of terms of each column's sum: gfl k(x) = min(x, D-1)+1, gfr k(x') = min(W-1-x', D-1)+1."""
    x = np.arange(W)
    return np.minimum(x, D - 1) + 1, np.minimum(W - 1 - x, D - 1) + 1


def summation_bounds(g, diff):
    """Per-element bound on |fp32 ordered sum - exact sum| for (gfl, gfr): gamma_{k-1} * sum |terms| with
    gamma_m = m u / (1 - m u), u = 2^-24 (recursive summation), computed in float64."""
    a = np.abs(g.astype(np.float64))
    al, ar = (_sum_left(a), _sum_right(a)) if diff else (_sum_left(a[:, :g.shape[1] // 2]),
                                                         _sum_right(a[:, g.shape[1] // 2:]))
    kl, kr = term_counts(g.shape[4], g.shape[2])
    u = 2.0 ** -24

    def gamma(k):
        m = (k - 1) * u
        return m / (1 - m)
    return gamma(kl) * al, gamma(kr) * ar


def torch_concat_volume(fl, fr, D):
    """PSMNet's construction (a zero volume and one slice assignment per disparity and half)."""
    N, C, H, W = fl.shape
    vol = fl.new_zeros((N, 2 * C, D, H, W))
    for d in range(min(D, W)):
        vol[:, :C, d, :, d:] = fl[:, :, :, d:]
        vol[:, C:, d, :, d:] = fr[:, :, :, :W - d]
    return vol


def torch_diff_volume(fl, fr, D):
    N, C, H, W = fl.shape
    vol = fl.new_zeros((N, C, D, H, W))
    for d in range(min(D, W)):
        vol[:, :, d, :, d:] = fl[:, :, :, d:] - fr[:, :, :, :W - d]
    return vol


def torch_volume(fl, fr, D, diff):
    return torch_diff_volume(fl, fr, D) if diff else torch_concat_volume(fl, fr, D)
