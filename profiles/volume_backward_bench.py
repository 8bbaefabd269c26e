#!/usr/bin/env python
"""Config P (PSMNet-shaped: unary features [16,32,136,240], D/4 = 48): the concat / difference volumes
forward and backward, CUDA events over warmed-up repetitions, beside PSMNet's stock-PyTorch construction
(a zero volume plus 2*D/4 slice assignments) forward + backward through autograd, the path a trainer used
before the volume builders were differentiable.

Algorithmic bytes (compulsory traffic, computed below from the shapes): a backward reads each half of the
gradient volume it needs once and writes each requested [N,C,h,w] gradient once.  Every working set
(>= 3.3 GB) is far larger than the 126 MB L2, so each timed pass streams from HBM.  Fraction of peak is
against the measured HBM copy rate (MEASURED_PEAKS.json when present, else 6551.7 GB/s).

Results are checked in the same run: the kernel gradients equal a GPU fp32 run of the ordered formula
(tests/_volume_ref.py: d ascending from 0, one rounding per add) bit for bit, and agree with the gradients
of the stock construction within twice the recursive-summation bound.

Usage: python profiles/volume_backward_bench.py [--out FILE.json]   (prints one JSON object)
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import __graft_entry__  # noqa: E402

__graft_entry__.build()
from msnets_b200 import _lib, volume  # noqa: E402
from tests import _volume_ref  # noqa: E402

N, C, h, w, D4 = 16, 32, 136, 240, 48
PEAK = 6551.7
try:
    PEAK = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
except Exception:
    pass


def timed(fn, reps, windows=3):
    """Median over `windows` CUDA-event windows of `reps` calls each, after 3 warm-up calls; ms per call."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    res = []
    for _ in range(windows):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        res.append(e0.elapsed_time(e1) / reps)
    return sorted(res)[len(res) // 2]


def raw_backward(diff, g, gfl, gfr):
    L = _lib.lib()
    fn = L.msn_diff_volume_backward_dev if diff else L.msn_concat_volume_backward_dev
    _lib.check(fn(g.data_ptr(), N, C, h, w, D4, gfl.data_ptr() if gfl is not None else None,
                  gfr.data_ptr() if gfr is not None else None, torch.cuda.current_stream().cuda_stream))


def ordered_sums(g):
    """The ordered fp32 restatement on the GPU: g [N,C,D,h,w] -> (left sums, right sums) [N,C,h,w]."""
    acc_l = torch.zeros((g.shape[0], g.shape[1], h, w), device=g.device, dtype=g.dtype)
    acc_r = torch.zeros_like(acc_l)
    for d in range(min(D4, w)):
        acc_l[..., d:] += g[:, :, d, :, d:]
        acc_r[..., :w - d] += g[:, :, d, :, d:]
    return acc_l, acc_r


def hardware():
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = q.stdout.strip()
    except Exception as e:  # the numbers are still reported, marked without the card's settings
        info["nvidia_smi"] = "unavailable: %s" % e
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="also write the JSON object to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this script measures on a CUDA device"
    torch.cuda.set_device(0)
    gen = torch.Generator(device="cuda").manual_seed(1234)
    fl = torch.randn((N, C, h, w), generator=gen, device="cuda")
    fr = torch.randn((N, C, h, w), generator=gen, device="cuda")
    feat = 4 * N * C * h * w                      # bytes of one [N,C,h,w] fp32 tensor
    vol_c, vol_d = 2 * feat * D4, feat * D4       # bytes of the concat / difference volume
    res = {"config": "P: features [16,32,136,240], D/4 = 48; concat volume [16,64,48,136,240]",
           "hardware": hardware(), "peak_GBps": PEAK, "kernels": {}, "paths": {}, "checks": {}}

    def kernel(name, ms, nbytes):
        gbs = nbytes / ms / 1e6
        res["kernels"][name] = {"ms": round(ms, 4), "algorithmic_GB": round(nbytes / 1e9, 3), "GBps": round(gbs, 1),
                                "frac_of_measured_peak": round(gbs / PEAK, 3)}

    for diff, vbytes in ((False, vol_c), (True, vol_d)):
        tag = "diff" if diff else "concat"
        Cg = C if diff else 2 * C
        out = torch.empty((N, Cg, D4, h, w), device="cuda")
        build = volume.diff_volume if diff else volume.concat_volume
        kernel(tag + "_forward", timed(lambda: build(fl, fr, D4, out=out), 50), 2 * feat + vbytes)
        del out
        g = torch.randn((N, Cg, D4, h, w), generator=gen, device="cuda")
        gfl, gfr = torch.empty_like(fl), torch.empty_like(fr)
        half = vbytes if diff else vbytes // 2           # the gradient bytes one output needs
        kernel(tag + "_backward_both", timed(lambda: raw_backward(diff, g, gfl, gfr), 50), vbytes + 2 * feat)
        kernel(tag + "_backward_gfl_only", timed(lambda: raw_backward(diff, g, gfl, None), 50), half + feat)

        # checks: bit-exact against the ordered formula, and within 2 gamma_{k-1} sum |terms| of the stock path
        raw_backward(diff, g, gfl, gfr)
        if diff:
            want_l, want_r = ordered_sums(g)
            want_r = -want_r
            abs_l, abs_r = ordered_sums(g.abs())
        else:
            want_l, _ = ordered_sums(g[:, :C])
            _, want_r = ordered_sums(g[:, C:])
            abs_l, _ = ordered_sums(g[:, :C].abs())
            _, abs_r = ordered_sums(g[:, C:].abs())
        bit_exact = bool(torch.equal(gfl, want_l) and torch.equal(gfr, want_r))
        a, b = fl.clone().requires_grad_(True), fr.clone().requires_grad_(True)
        _volume_ref.torch_volume(a, b, D4, diff).backward(g)
        kl, kr = (torch.from_numpy(k).to(device="cuda", dtype=torch.float64) for k in _volume_ref.term_counts(w, D4))
        u = 2.0 ** -24
        bound_l = 2 * ((kl - 1) * u / (1 - (kl - 1) * u)) * abs_l.double()
        bound_r = 2 * ((kr - 1) * u / (1 - (kr - 1) * u)) * abs_r.double()
        err_l = (gfl.double() - a.grad.double()).abs()
        err_r = (gfr.double() - b.grad.double()).abs()
        res["checks"][tag] = {"bit_exact_vs_ordered_fp32": bit_exact,
                              "within_bound_vs_torch_construction": bool((err_l <= bound_l).all() and
                                                                         (err_r <= bound_r).all()),
                              "max_abs_diff_vs_torch_construction": float(max(err_l.max(), err_r.max()))}
        del a, b, want_l, want_r, abs_l, abs_r, bound_l, bound_r, err_l, err_r

        # forward + backward through autograd: this library vs the stock construction
        a, b = fl.clone().requires_grad_(True), fr.clone().requires_grad_(True)

        def ours():
            a.grad = b.grad = None
            build(a, b, D4).backward(g)

        def stock():
            a.grad = b.grad = None
            _volume_ref.torch_volume(a, b, D4, diff).backward(g)
        t_ours, t_stock = timed(ours, 20), timed(stock, 5)
        res["paths"][tag + "_forward_backward_autograd"] = {"ms": round(t_ours, 3)}
        res["paths"][tag + "_forward_backward_torch_slice_loop"] = {"ms": round(t_stock, 3),
                                                                    "slowdown_vs_autograd": round(t_stock / t_ours, 2)}
        del g, gfl, gfr, a, b
        torch.cuda.empty_cache()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    assert all(c["bit_exact_vs_ordered_fp32"] and c["within_bound_vs_torch_construction"]
               for c in res["checks"].values()), "result check failed"


if __name__ == "__main__":
    main()
