"""4D cost-volume builders for learned unary features (GC-Net / PSMNet style).

The reference has no such builder (SURVEY.md 0.3): its PSMNet head expects the
classic 2x32-channel concat volume (`dres0`, psmnet_3dcnn.py:96) but nothing
produces it.  Definitions (oracle/ms_oracle.py:concat_volume / diff_volume):

    concat[n, :C, d, y, x] = fl[n, :, y, x]      for x >= d, else 0
    concat[n, C:, d, y, x] = fr[n, :, y, x - d]  for x >= d, else 0
    diff  [n, c, d, y, x]  = fl[n,c,y,x] - fr[n,c,y,x-d]  for x >= d, else 0

Both are differentiable: when grad mode is on and `fl` or `fr` requires grad, the
volume carries a grad_fn whose backward is one kernel launch
(msn_concat_volume_backward_dev / msn_diff_volume_backward_dev).  With G the
gradient of the volume:

    concat: gfl[n,c,y,x]  = sum_{d=0..min(x, D-1)}      G[n,  c, d, y, x]
            gfr[n,c,y,x'] = sum_{d=0..min(W-1-x', D-1)} G[n, C+c, d, y, x'+d]
    diff:   gfl as concat, gfr = -sum_{d=0..min(W-1-x', D-1)} G[n, c, d, y, x'+d]

Each sum is in fp32, d ascending from 0, so the gradients are deterministic.  G at
masked voxels (x < d) never reaches them.  Double backward is not supported
and raises.  `out=` is for inference only.
"""
from . import _lib


def _build(fl, fr, ndisp, diff, out):
    import torch
    if not (fl.is_cuda and fr.is_cuda):
        raise _lib.MsnetsError("volume builders need CUDA tensors (no CPU fallback)")
    if fl.dtype != torch.float32 or fr.dtype != torch.float32 or fl.shape != fr.shape or fl.dim() != 4:
        raise ValueError("expected two float32 [N,C,H,W] tensors of equal shape")
    a, b = fl.contiguous(), fr.contiguous()
    N, C, H, W = a.shape
    shape = (N, C if diff else 2 * C, int(ndisp), H, W)
    if out is None:
        out = torch.empty(shape, dtype=torch.float32, device=a.device)
    elif tuple(out.shape) != shape or not out.is_contiguous():
        raise ValueError("out must be contiguous with shape %s" % (shape,))
    fn = _lib.lib().msn_diff_volume_dev if diff else _lib.lib().msn_concat_volume_dev
    with torch.cuda.device(a.device):
        _lib.check(fn(a.data_ptr(), b.data_ptr(), N, C, H, W, int(ndisp), out.data_ptr(),
                      torch.cuda.current_stream().cuda_stream))
    return out


_functions = {}


def _autograd_function():
    """The torch.autograd.Function, built on first use (torch is imported lazily).  The volume is linear in
    (fl, fr), so nothing is saved but the shape."""
    if _functions:
        return _functions["shift_volume"]
    import torch
    from torch.autograd.function import once_differentiable

    class ShiftVolume(torch.autograd.Function):
        @staticmethod
        def forward(ctx, fl, fr, ndisp, diff):
            vol = _build(fl, fr, ndisp, diff, None)
            ctx.diff = diff
            ctx.shape = tuple(fl.shape) + (int(ndisp),)
            return vol

        @staticmethod
        @once_differentiable
        def backward(ctx, grad):
            g = grad.contiguous().to(torch.float32)
            N, C, H, W, D = ctx.shape
            want_l, want_r = ctx.needs_input_grad[:2]     # at least one, or autograd would not call this
            gfl = torch.empty((N, C, H, W), dtype=torch.float32, device=g.device) if want_l else None
            gfr = torch.empty((N, C, H, W), dtype=torch.float32, device=g.device) if want_r else None
            L = _lib.lib()
            fn = L.msn_diff_volume_backward_dev if ctx.diff else L.msn_concat_volume_backward_dev
            with torch.cuda.device(g.device):
                _lib.check(fn(g.data_ptr(), N, C, H, W, D, gfl.data_ptr() if want_l else None,
                              gfr.data_ptr() if want_r else None, torch.cuda.current_stream().cuda_stream))
            return gfl, gfr, None, None

    _functions["shift_volume"] = ShiftVolume
    return ShiftVolume


def _volume(fl, fr, ndisp, diff, out):
    import torch
    if torch.is_grad_enabled() and (fl.requires_grad or fr.requires_grad):
        if out is not None:
            raise ValueError("%s_volume: out= cannot be combined with autograd" % ("diff" if diff else "concat"))
        return _autograd_function().apply(fl, fr, int(ndisp), diff)
    return _build(fl, fr, ndisp, diff, out)


def concat_volume(fl, fr, ndisp, out=None):
    """fl, fr: float32 CUDA [N,C,H,W] -> [N,2C,ndisp,H,W].  Differentiable in fl and fr."""
    return _volume(fl, fr, ndisp, False, out)


def diff_volume(fl, fr, ndisp, out=None):
    """fl, fr: float32 CUDA [N,C,H,W] -> [N,C,ndisp,H,W].  Differentiable in fl and fr."""
    return _volume(fl, fr, ndisp, True, out)
