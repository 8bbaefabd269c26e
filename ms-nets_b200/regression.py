"""Soft-argmin disparity regression: drop-in for `F.softmax(out, 1)` followed by
`disparityregression` (src/models/gcnet_3dcnn.py:127-141; duplicate modules at
gcnet_3dcnn.py:46-54, psmnet_3dcnn.py:28-37, basic_convs.py:279-287).

The reference splits the op in two (softmax, then sum(prob * arange)); both halves
are kept so either call site can be swapped:

    soft_argmin(logits)                  fused softmax + expectation, one pass
    disparityregression(maxdisp)(prob)   module with the reference's signature; fed
                                         probabilities it returns sum_d d * prob_d
    patch_gcnet(model)                   swaps model.disparityregression and makes
                                         the final softmax+regression one kernel
"""
import numpy as np

from . import _lib


def _torch():
    import torch
    return torch


def _output(x, out, who):
    """out= for a [N,D,H,W] input: a new tensor, or the caller's after checking it.  The kernels write
    N*H*W floats through its raw pointer, so anything but a contiguous float32 [N,H,W] tensor on x's
    device would be overrun or misread."""
    torch = _torch()
    N, D, H, W = x.shape
    if out is None:
        return torch.empty((N, H, W), dtype=torch.float32, device=x.device)
    if (not isinstance(out, torch.Tensor) or tuple(out.shape) != (N, H, W) or out.dtype != torch.float32
            or not out.is_contiguous() or out.device != x.device):
        raise ValueError("%s: out must be a contiguous float32 [%d,%d,%d] tensor on %s" % (who, N, H, W, x.device))
    return out


def _raw_soft_argmin(x, out=None):
    torch = _torch()
    N, D, H, W = x.shape
    out = _output(x, out, "soft_argmin")
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().msn_soft_argmin_dev(x.data_ptr(), N, D, H, W, out.data_ptr(),
                                                  torch.cuda.current_stream().cuda_stream))
    return out


def _raw_expected_disparity(x, out=None):
    torch = _torch()
    N, D, H, W = x.shape
    out = _output(x, out, "disparityregression")
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().msn_expect_disp_dev(x.data_ptr(), N, D, H, W, out.data_ptr(),
                                                  torch.cuda.current_stream().cuda_stream))
    return out


_functions = {}


def _autograd_functions():
    """torch.autograd.Function wrappers, built on first use (torch is imported lazily).  The
    reference trains THROUGH softmax + disparityregression (gcnet_3dcnn.py:127-141,
    psmnet_3dcnn.py:149-176), so the kernels must carry gradients when they stand in for them."""
    if _functions:
        return _functions
    torch = _torch()

    class SoftArgmin(torch.autograd.Function):
        @staticmethod
        def forward(ctx, logits):
            x = logits.contiguous()
            disp = _raw_soft_argmin(x)
            ctx.save_for_backward(x, disp)
            return disp

        @staticmethod
        def backward(ctx, grad_out):
            x, disp = ctx.saved_tensors
            g = grad_out.contiguous().to(torch.float32)
            N, D, H, W = x.shape
            grad_in = torch.empty_like(x)
            with torch.cuda.device(x.device):
                _lib.check(_lib.lib().msn_soft_argmin_backward_dev(
                    x.data_ptr(), disp.data_ptr(), g.data_ptr(), N, D, H, W, grad_in.data_ptr(),
                    torch.cuda.current_stream().cuda_stream))
            return grad_in

    class ExpectedDisparity(torch.autograd.Function):
        @staticmethod
        def forward(ctx, prob):
            x = prob.contiguous()
            ctx.D = x.shape[1]
            return _raw_expected_disparity(x)

        @staticmethod
        def backward(ctx, grad_out):
            # d/dp_d sum_d d * p_d = d : one broadcast product, no saved tensors
            d = torch.arange(ctx.D, dtype=grad_out.dtype, device=grad_out.device).view(1, ctx.D, 1, 1)
            return grad_out.unsqueeze(1) * d

    _functions["soft_argmin"] = SoftArgmin
    _functions["expected_disparity"] = ExpectedDisparity
    return _functions


def soft_argmin(logits, out=None):
    """logits: float32 [N,D,H,W] (CUDA tensor or NumPy array) -> disp float32 [N,H,W].
    A -inf logit masks its disparity; a pixel masked at every disparity gives NaN, as torch's softmax does.
    Differentiable: when `logits` requires grad the result carries a grad_fn (backward =
    grad * softmax * (d - disp), msn_soft_argmin_backward_dev); `out=` is inference only."""
    if isinstance(logits, np.ndarray):
        x = np.ascontiguousarray(logits, dtype=np.float32)
        if x.ndim != 4:
            raise ValueError("soft_argmin: expected [N,D,H,W]")
        N, D, H, W = x.shape
        res = np.empty((N, H, W), np.float32)
        _lib.check(_lib.lib().msn_soft_argmin_host(x.ctypes.data, N, D, H, W, res.ctypes.data))
        return res
    torch = _torch()
    if logits.dim() != 4 or logits.dtype != torch.float32:
        raise ValueError("soft_argmin: expected a float32 [N,D,H,W] tensor")
    if not logits.is_cuda:
        raise _lib.MsnetsError("soft_argmin: tensor must live on a CUDA device (no CPU fallback)")
    if torch.is_grad_enabled() and logits.requires_grad:
        if out is not None:
            raise ValueError("soft_argmin: out= cannot be combined with autograd")
        return _autograd_functions()["soft_argmin"].apply(logits)
    return _raw_soft_argmin(logits.contiguous(), out)


def expected_disparity(prob, out=None):
    """sum_d d * prob_d for probabilities [N,D,H,W]: the body of the reference's
    disparityregression (gcnet_3dcnn.py:136-139) without materialising
    arange(D).repeat(N,1,H,W) or the product tensor.  Differentiable like soft_argmin."""
    torch = _torch()
    if prob.dim() != 4 or prob.dtype != torch.float32:
        raise ValueError("disparityregression: expected a float32 [N,D,H,W] tensor")
    if not prob.is_cuda:
        raise _lib.MsnetsError("disparityregression: tensor must live on a CUDA device (no CPU fallback)")
    if torch.is_grad_enabled() and prob.requires_grad:
        if out is not None:
            raise ValueError("disparityregression: out= cannot be combined with autograd")
        return _autograd_functions()["expected_disparity"].apply(prob)
    return _raw_expected_disparity(prob.contiguous(), out)


def _module_base():
    import torch.nn as nn
    return nn.Module


class disparityregression(_module_base()):
    """Same constructor/forward signature as the reference module (gcnet_3dcnn.py:46-54)."""

    def __init__(self, maxdisp, sumKeepDim=False):
        super(disparityregression, self).__init__()
        self.maxdisp = int(maxdisp)
        self.sumKeepDim = sumKeepDim

    def forward(self, x):
        if x.size(1) != self.maxdisp:
            raise AssertionError("%d != %d" % (x.size(1), self.maxdisp))  # gcnet_3dcnn.py:135
        out = expected_disparity(x)
        return out.unsqueeze(1) if self.sumKeepDim else out


def patch_gcnet(model):
    """Swaps the `disparityregression` method of a reference GCNet_CostVolumeAggre
    (gcnet_3dcnn.py:132-141) for the expectation kernel.  The model's forward keeps
    its own `F.softmax(out,1)` (:127); to fuse both halves replace lines :127-128 with
    `disp = msnets_b200.regression.soft_argmin(out)` (see INTEGRATION.md).
    Works in training too: both kernels are wrapped in torch.autograd.Functions."""
    import types

    def _regress(self, x):
        N, D, H, W = x.size()[:]
        assert D == self.maxdisp, "%d != %d" % (D, self.maxdisp)  # gcnet_3dcnn.py:135
        return expected_disparity(x)

    model.disparityregression = types.MethodType(_regress, model)
    return model
