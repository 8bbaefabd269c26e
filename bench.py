#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

metric : stereo pairs/sec for "MS features + cost volume + soft-argmin" at 540x960,
         D=192 (BASELINE.json configs[1]: SceneFlow-shaped batch of 8 pairs per GPU).
         In MS-GCNet the cost volume IS the 8-channel MS feature tensor
         [N,8,D,h,w] (SURVEY.md 0.3), so one step = that tensor for 8 pairs + the
         soft-argmin over a [8,192,540,960] logit volume.
step   : ours      -> prep + sadsob scan + fused volume kernel + soft-argmin kernel on
                      cuda:<local rank>, inputs resident in HBM (value), and the same
                      through the public API with pinned host buffers, H2D of the pairs
                      and D2H of the disparities inside the timed region (e2e).
         reference -> the reference's own CPU implementation: its UNMODIFIED NumPy glue
                      (cbmv_generator.py get_costs + extract_features_left) over oracle/_ref =
                      the unmodified matchers.cpp / featextract.cpp compiled in the build
                      container with THREADS_NUM_USED = the host's core count; one full
                      540x960 pair per step (a row band only if the run would not fit).
Multi-GPU: one process per GPU (torchrun), pairs are independent -> weak scaling, no
data-path collective; time = max over ranks.
Prints ONE JSON line on rank 0.
"""
import argparse
import ctypes
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "stereo pairs/sec (MS features+cost volume+soft-argmin, 540x960 D=192)"
H_IMG, W_IMG, D_MAX, BORDER, BATCH = 540, 960, 192, 10, 8


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
        except Exception:
            pass
    return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


def algorithmic_bytes():
    """SURVEY.md 8d: compulsory traffic per pair."""
    Hp, Wp = H_IMG + 2 * BORDER, W_IMG + 2 * BORDER
    b_ms = 2 * Hp * Wp + 8 * D_MAX * H_IMG * W_IMG * 4
    b_sa = 4 * D_MAX * H_IMG * W_IMG + 4 * H_IMG * W_IMG
    return b_ms, b_sa


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons during the timed region (pynvml)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None

    def run(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
            names = {0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
                     0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
                     0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}
            while not self.stop_flag:
                self.samples.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                try:
                    r = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, n in names.items():
                    if r & bit:
                        self.reasons.add(n)
                time.sleep(0.05)
        except Exception as e:  # never let the sampler kill the bench
            self.reasons.add("sampler_error:%s" % type(e).__name__)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


def physical_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# --------------------------------------------------------------------- ours --
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from tests._synth import bordered_pair

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    import __graft_entry__
    if rank == 0:
        __graft_entry__.build()
    if world > 1:
        dist.barrier()
    import msnets_b200
    from msnets_b200 import _lib, cbmv, regression

    dev = torch.device("cuda", local_rank)
    Hb, Wb = H_IMG + 2 * BORDER, W_IMG + 2 * BORDER
    # synthetic SceneFlow-shaped batch (SURVEY.md 8d): seeded uniform pairs, 7 px shift,
    # 10 px zero border; every rank gets its own pairs
    NSETS = 2
    host_l = torch.empty((NSETS, BATCH, Hb, Wb), dtype=torch.uint8).pin_memory()
    host_r = torch.empty((NSETS, BATCH, Hb, Wb), dtype=torch.uint8).pin_memory()
    for s in range(NSETS):
        for i in range(BATCH):
            L, R = bordered_pair(H_IMG, W_IMG, 1234 + 1000 * rank + 10 * s + i, border=BORDER)
            host_l[s, i] = torch.from_numpy(L)
            host_r[s, i] = torch.from_numpy(R)
    dev_l, dev_r = host_l.to(dev), host_r.to(dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)
    logits = torch.randn((BATCH, D_MAX, H_IMG, W_IMG), generator=gen, device=dev, dtype=torch.float32)
    ex = cbmv.MSFeatureExtractor(BATCH, Hb, Wb, maxdisp=D_MAX, board_h=BORDER, board_w_left=BORDER,
                                 board_w_right=BORDER, device=dev)
    feats = ex.empty_output()
    disp = torch.empty((BATCH, H_IMG, W_IMG), dtype=torch.float32, device=dev)

    def step_resident(i):
        s = i % NSETS
        ex(dev_l[s], dev_r[s], out=feats)
        regression.soft_argmin(logits, out=disp)

    # End-to-end pipeline through the public API, as a consumer would run it: every step's pairs are
    # copied from pinned host memory and every step's disparities are copied back; copies use their
    # own streams and two sets of buffers, so the H2D of step i+1 and the D2H of step i-1 overlap
    # the kernels of step i.  The host blocks on a step's result before its buffers are reused.
    h2d_stream, d2h_stream = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    stage_l = [torch.empty_like(dev_l[0]) for _ in range(2)]
    stage_r = [torch.empty_like(dev_r[0]) for _ in range(2)]
    disp2 = [torch.empty_like(disp) for _ in range(2)]
    host_disp2 = [torch.empty((BATCH, H_IMG, W_IMG), dtype=torch.float32).pin_memory() for _ in range(2)]
    ev_h2d = [torch.cuda.Event() for _ in range(2)]
    ev_comp = [torch.cuda.Event() for _ in range(2)]
    ev_d2h = [torch.cuda.Event() for _ in range(2)]
    used = [False, False]

    def step_e2e(i):
        s, b = i % NSETS, i & 1
        cur = torch.cuda.current_stream()
        if used[b]:
            ev_d2h[b].synchronize()          # the caller consumes the disparities of step i-2
            h2d_stream.wait_event(ev_comp[b])  # ... whose kernels were the last readers of stage[b]
        with torch.cuda.stream(h2d_stream):
            stage_l[b].copy_(host_l[s], non_blocking=True)
            stage_r[b].copy_(host_r[s], non_blocking=True)
            ev_h2d[b].record(h2d_stream)
        cur.wait_event(ev_h2d[b])
        ex(stage_l[b], stage_r[b], out=feats)
        regression.soft_argmin(logits, out=disp2[b])
        ev_comp[b].record(cur)
        with torch.cuda.stream(d2h_stream):
            d2h_stream.wait_event(ev_comp[b])
            host_disp2[b].copy_(disp2[b], non_blocking=True)
            ev_d2h[b].record(d2h_stream)
        used[b] = True

    def drain_e2e():
        cur = torch.cuda.current_stream()
        for b in range(2):
            if used[b]:
                cur.wait_event(ev_d2h[b])     # the timed region ends when the last result is on the host

    def timed(fn, steps, warmup, profile=False, drain=None):
        for i in range(warmup):
            fn(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if profile:
            _lib.check(_lib.lib().msn_profile_enable(1))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        if drain is not None:
            drain()
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        prof = None
        if profile:
            a, b, c, n = ctypes.c_double(), ctypes.c_double(), ctypes.c_double(), ctypes.c_int()
            _lib.check(_lib.lib().msn_profile_read(ctypes.byref(a), ctypes.byref(b), ctypes.byref(c), ctypes.byref(n)))
            _lib.check(_lib.lib().msn_profile_enable(0))
            prof = {"prep_ms": a.value, "sadsob_ms": b.value, "fused_ms": c.value, "calls": n.value}
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, prof

    sampler = ClockSampler(physical_index(local_rank))
    sampler.start()
    ms_res, prof = timed(step_resident, args.steps, args.warmup, profile=True)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, feats, disp)
    ms_e2e, _ = timed(step_e2e, args.steps, min(args.warmup, 3), drain=drain_e2e)

    # soft-argmin kernel alone (for the per-kernel breakdown)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        regression.soft_argmin(logits, out=disp)
    e1.record()
    torch.cuda.synchronize()
    sa_ms = e0.elapsed_time(e1) / args.steps

    slab = None
    if world > 1:
        # BASELINE configs[4] on the same launch: one Middlebury-shaped frame, disparity-slab sharded over the
        # ranks -- the one mode of the path with a data-plane exchange between the GPUs
        del feats, logits, disp, stage_l, stage_r, disp2, dev_l, dev_r, ex
        torch.cuda.empty_cache()
        slab = slab_config_m(dev, rank, world)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pairs = BATCH * world * args.steps
    value = pairs / (ms_res / 1e3)
    e2e_value = pairs / (ms_e2e / 1e3)
    b_ms, b_sa = algorithmic_bytes()
    peak, peak_src = peaks()
    fused_ms = prof["fused_ms"] / max(prof["calls"], 1)
    achieved = BATCH * b_ms / (fused_ms / 1e3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.isfile(tp):
        try:
            traffic = int(json.load(open(tp)).get("ms_fused_kernel_dram_bytes_per_pair") * BATCH)
        except Exception:
            traffic = None
    step_ms = ms_res / args.steps
    roofline = {
        "bound": "hbm", "kernel": "ms_fused_kernel", "achieved": round(achieved, 1), "peak": peak,
        "unit": "GB/s", "frac": round(achieved / peak, 4), "traffic": traffic,
        "peak_source": peak_src,
        "algorithmic_bytes_per_launch": BATCH * b_ms,
        "kernel_ms_per_launch": round(fused_ms, 4),
        "step_frac": round(BATCH * (b_ms + b_sa) / (step_ms / 1e3) / 1e9 / peak, 4),
        "breakdown_ms_per_step": {"prep": round(prof["prep_ms"] / prof["calls"], 4),
                                  "sadsob_scan": round(prof["sadsob_ms"] / prof["calls"], 4),
                                  "ms_fused": round(fused_ms, 4), "soft_argmin": round(sa_ms, 4)},
    }
    cpu, dropin = None, None
    if world == 1:
        cpu = cpu_baseline_sample(budget_s=30.0)
        # drop-in NumPy API, one pair, full 3.2 GB volume copied back to the host
        t0 = time.time()
        vol = cbmv.ms_features(host_l[0, 0].numpy(), host_r[0, 0].numpy(), D_MAX, board_h=BORDER,
                               board_w_left=BORDER, board_w_right=BORDER)
        dropin_s = time.time() - t0
        dropin = {"pairs_per_s": round(1.0 / dropin_s, 3), "d2h_bytes": int(vol.nbytes),
                  "note": "msn_ms_features_host, 1 pair, whole volume returned to pageable host memory"}
        del vol
    line = {
        "metric": METRIC, "value": round(value, 2), "unit": "pairs/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(step_ms, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: SceneFlow-shaped 540x960 D=192, batch 8 pairs per GPU: MS features "
                               "[8,8,192,540,960] + soft-argmin over [8,192,540,960]",
                   "pairs_per_step_per_gpu": BATCH, "border_px": BORDER, "windows": [11, 3, 5, 5],
                   "parallelism": "batch-sharded x%d (no collective)" % world,
                   "l2": "per-step working set 28.7 GB (25.5 GB written + 3.2 GB read) >> 126 MB L2; "
                         "two input sets alternate; no flush needed"},
        "clocks": sampler.summary(),
        "e2e": {"value": round(e2e_value, 2), "unit": "pairs/s", "h2d_bytes_per_step": 2 * BATCH * Hb * Wb,
                "d2h_bytes_per_step": BATCH * H_IMG * W_IMG * 4, "ms_per_step": round(ms_e2e / args.steps, 4),
                "api": "MSFeatureExtractor(pinned uint8 pairs) -> soft_argmin -> pinned disparities; "
                       "double-buffered: copies on their own streams overlap the previous / next step"},
        "gpu_launches": 5 * args.steps,
        "roofline": roofline,
        "cpu_baseline": cpu,
        "numpy_dropin": dropin,
    }
    if slab is not None:
        line["slab_config_m"] = slab
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


DUMP_FEATURE_SAMPLES = 1 << 22


def dump_outputs(out_dir, feats, disp):
    """Writes what the last timed step returned, for comparing two builds output for output:
    disparity.npy, the whole [8,540,960] soft-argmin result, and ms_features_sample.npy, the MS feature
    volume [8,8,192,540,960] (25.5 GB) at DUMP_FEATURE_SAMPLES voxels drawn with a fixed seed, in
    ascending flat-index order.  Both float32, 33 MB in all."""
    import numpy as np
    import torch
    n = feats.numel()
    idx = np.sort(np.random.default_rng(0).integers(0, n, DUMP_FEATURE_SAMPLES))
    sample = feats.reshape(-1).index_select(0, torch.from_numpy(idx).to(feats.device))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "disparity.npy"), disp.float().cpu().numpy())
    np.save(os.path.join(out_dir, "ms_features_sample.npy"), sample.float().cpu().numpy())


def slab_config_m(dev, rank, world, steps=3, warmup=2):
    """BASELINE configs[4]: one Middlebury-shaped 1984x2880, D=640 frame, every rank owning D/world
    disparities.  Per frame: the slab volume through ExchangeSlabMSFeatures (minima / denominators traded
    inside the kernel over peer-mapped memory; falls back to the three-phase NCCL path when the slab does not
    cut into equal sub-slabs), WTA over the sharded census channel (int64 key all-reduce) and soft-argmin over
    a sharded logit volume (all-gather of partials).  Timed with CUDA events, max over ranks."""
    import torch
    import torch.distributed as dist
    from msnets_b200 import sharding
    from tests._synth import bordered_pair
    H, W, D, B = 1984, 2880, 640, BORDER
    L, R = bordered_pair(H, W, 99, border=B, shift=13)
    l, r = torch.from_numpy(L[None]).to(dev), torch.from_numpy(R[None]).to(dev)
    mode = "exchange"
    bands, grp = 1, None
    try:
        bands = sharding.ExchangeSlabMSFeatures.default_row_bands(D, world)
        ex = sharding.ExchangeSlabMSFeatures(1, H + 2 * B, W + 2 * B, maxdisp=D, row_bands=bands, board_h=B,
                                             board_w_left=B, board_w_right=B)
        grp = ex.slab_group
    except ValueError:
        mode, bands = "phases", 1
        ex = sharding.SlabShardedMSFeatures(1, H + 2 * B, W + 2 * B, maxdisp=D, board_h=B, board_w_left=B,
                                            board_w_right=B)
    out = torch.empty(ex.shape, dtype=torch.float32, device=dev)
    gen = torch.Generator(device=dev)
    gen.manual_seed(77 + rank)
    rows = ex.shape[3]
    logits = torch.randn((1, ex.d_count, rows, W), generator=gen, device=dev, dtype=torch.float32)

    parts = ex.empty_wta_parts() if mode == "exchange" else None

    def step():
        if mode == "exchange":     # WTA / second-min triples are a by-product of the slab kernel: merge them
            ex(l, r, out=out, wta=parts)
            am, m1, m2 = sharding.slab_wta_merge(*parts, group=grp)
        else:
            ex(l, r, out=out)
            am, m1 = sharding.slab_wta(out[0, 0], ex.d_begin, layout="dhw")
        return am, sharding.slab_soft_argmin(logits, ex.d_begin, group=grp)

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        am, disp = step()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1) / steps], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    col = out[0, 4:8].sum(1)                      # AML columns over ALL slabs' disparities sum to 1
    if getattr(ex, "slabs", world) > 1:
        dist.all_reduce(col, op=dist.ReduceOp.SUM, group=grp)
    err = float((col[col > 0.5] - 1).abs().max())
    peak, _ = peaks()
    vox = D * H * W
    tiles = rows * ((W + 31) // 32)
    subs = getattr(ex, "subs", 1) or 1
    slabs = getattr(ex, "slabs", world)
    res = {
        "workload": "configs[4]: Middlebury-shaped 1984x2880 D=640, one frame over %d GPUs: %d disparity slab(s) x %d row "
                    "band(s) (MS volume [1,8,%d,%d,2880] per GPU + WTA + soft-argmin merges)"
                    % (world, slabs, bands, ex.d_count, rows),
        "mode": mode, "slabs": slabs, "row_bands": bands, "ms_per_frame": round(ms, 3), "frames_per_s": round(1e3 / ms, 2), "steps": steps,
        "algorithmic_GB_per_gpu": round((32.0 + 4.0) * vox / world / 1e9, 2),
        "GBps_per_gpu": round((32.0 + 4.0) * vox / world / ms / 1e6, 1),
        "frac_of_hbm_peak_per_gpu": round((32.0 + 4.0) * vox / world / ms / 1e6 / peak, 4),
        "collectives_per_frame": {
            "aml_min_and_den": ("in-kernel: %d sub-slab(s) per rank push 2 x 640 B per tile to the %d other rank(s) of the row band "
                                "over NVLink = %.1f MB out per rank" % (subs, slabs - 1, tiles * subs * 2 * 640 * (slabs - 1) / 1e6))
            if mode == "exchange" else "2 x NCCL all_reduce over [4,1984,2880] f32 = 91.4 MB each",
            "wta": ("NCCL all_gather of the kernel's (argmin, min1, min2) by-product, 4 channels: 3 x [1,4,%d,2880] "
                    "x 4 B = %.1f MB per rank (sub-slabs merged locally first), merged by msn_wta_merge_dev"
                    % (rows, 3 * 4 * rows * W * 4 / 1e6))
            if mode == "exchange" else "NCCL all_reduce(min) over [1984,2880] int64 keys = 45.7 MB",
            "soft_argmin": "NCCL all_gather of [3,%d,2880] f32 partials = %.1f MB per rank" % (rows, 3 * rows * W * 4 / 1e6)},
        "aml_column_sum_max_err": err,
    }
    del out, logits
    if hasattr(ex, "close"):
        ex.close()
    return res


# ---------------------------------------------------------------- reference --
class _Timed(object):
    """Proxy of a native module that accumulates the wall time spent inside its functions (the
    native-only subtotal BASELINE.md section 3 asks for: get_costs' matchers + 4x extract_likelihood,
    as opposed to the NumPy glue around them)."""

    def __init__(self, mod, acc):
        self._mod, self._acc = mod, acc

    def __getattr__(self, name):
        fn = getattr(self._mod, name)
        if not callable(fn):
            return fn

        def timed(*a, **k):
            t0 = time.perf_counter()
            try:
                return fn(*a, **k)
            finally:
                self._acc[0] += time.perf_counter() - t0
        return timed


def _reference_arm(variant=None):
    """-> dict(gen, kind, what, cores, native_s): the reference's own CPU path.  `gen` is the UNMODIFIED
    src/dataloader/cbmv_generator.py (get_costs :27, extract_features_left :258) bound to oracle/_ref = the
    unmodified matchers.cpp / featextract.cpp compiled in the build container; when neither travels, the
    restated oracle (kind "port")."""
    from oracle import ms_oracle as O
    from oracle import ref_glue
    ref = None
    for v in ([variant] if variant else ["avx2_nproc", "avx2", "sse41"]):
        if v in ("avx2", "avx2_nproc") and not O.cpu_has_avx2():
            continue
        ref = O.load_ref(v)
        if ref is not None:
            break
    native = [0.0]
    if ref is not None:
        mtc, fte = _Timed(ref[0], native), _Timed(ref[1], native)
        gen = ref_glue.load_generator(mtc, fte)
        cores = int(ref[0].initthreads())
        if gen is not None:
            return {"gen": gen, "kind": "reference", "cores": cores, "native_s": native,
                    "what": "unmodified cbmv_generator.py (get_costs + extract_features_left) over oracle/_ref/%s "
                            "(unmodified matchers.cpp/featextract.cpp, %d OpenMP threads)" % (ref[2], cores)}

        class G(object):   # the glue file did not travel: restated glue over the reference C++
            get_costs = staticmethod(lambda *a: O.get_costs(*a, mtc=mtc, fte=fte))
            extract_features_left = staticmethod(lambda *c: O.extract_features_left(*c, fte=fte))
        return {"gen": G, "kind": "reference", "cores": cores, "native_s": native,
                "what": "oracle/_ref/%s driven by the restated NumPy glue" % ref[2]}
    O.lib()

    class P(object):
        get_costs = staticmethod(lambda *a: O.get_costs(*a))
        extract_features_left = staticmethod(lambda *c: O.extract_features_left(*c))
    return {"gen": P, "kind": "port", "cores": 1, "native_s": native, "what": "oracle/libms_oracle.so (C restatement)"}


def _cpu_step(arm, L, R, logits):
    """One reference step on the host: MS features of one pair + softmax/regression of one logit volume."""
    import torch
    import torch.nn.functional as F
    gen = arm["gen"]
    costs = gen.get_costs(L, R, D_MAX, 11, 3, 5, 5, BORDER, BORDER, BORDER)      # cbmv_generator.py:826-834
    f = gen.extract_features_left(*costs)                                         # :838
    del costs
    x = torch.from_numpy(logits)
    prob = F.softmax(x, 1)                                    # gcnet_3dcnn.py:127
    d = torch.arange(D_MAX, dtype=torch.float32).view(1, D_MAX, 1, 1)
    disp = torch.sum(prob * d, 1)                             # gcnet_3dcnn.py:136-139
    return f, disp


def _sample_inputs(rows):
    import numpy as np

    from tests._synth import bordered_pair
    L, R = bordered_pair(rows, W_IMG, 1234, border=BORDER)
    logits = np.random.default_rng(1234).standard_normal((1, D_MAX, rows, W_IMG)).astype(np.float32)
    return L, R, logits


def _rows_for_budget(arm, steps, budget_s):
    """Full 540-row frames when `steps` of them fit the budget (calibrated on a 32-row band), else the
    largest band that does."""
    L, R, lg = _sample_inputs(32)
    _cpu_step(arm, L, R, lg)
    t0 = time.time()
    _cpu_step(arm, L, R, lg)
    t32 = max(time.time() - t0, 1e-3)
    per_row = t32 / 32.0
    if steps * per_row * H_IMG * 1.15 <= budget_s:
        return H_IMG
    return int(max(32, min(H_IMG, budget_s / max(steps, 1) / per_row)))


def _cpu_sample_one(variant, budget_s):
    """One full-frame (or largest fitting band) step of the reference's CPU path with one build of oracle/_ref."""
    arm = _reference_arm(variant)
    rows = _rows_for_budget(arm, 1, budget_s)
    L, R, lg = _sample_inputs(rows)
    arm["native_s"][0] = 0.0
    t0 = time.time()
    _cpu_step(arm, L, R, lg)
    dt = time.time() - t0
    frac = rows / float(H_IMG)
    return {"value": round(frac / dt, 4), "unit": "pairs/s", "cores": arm["cores"], "kind": arm["kind"],
            "sample": "%d of 540 rows (x960, D=192) of one pair, one step: %s + softmax/regression; %d host cpus"
                      % (rows, arm["what"], os.cpu_count() or 0),
            "seconds": round(dt, 2), "native_only_seconds": round(arm["native_s"][0], 2),
            "native_only_pairs_per_s": round(frac / max(arm["native_s"][0], 1e-9), 4)}


def cpu_baseline_sample(budget_s=30.0):
    """The reference's CPU path timed beside the GPU run (rank 0, N = 1): one full 540x960 frame per
    build when it fits the budget -- the host-core-count build (value) and the shipped 8-thread build.  The
    second build runs in a child process: two builds of one extension module (same PyInit name) cannot be
    loaded side by side."""
    import subprocess
    out = _cpu_sample_one(None if not os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "avx2_nproc")) else "avx2_nproc",
                          budget_s / 2)
    if out["kind"] == "reference":
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-sample", "avx2", "--budget",
                                str(budget_s / 2)], capture_output=True, text=True, timeout=300)
            out["threads_as_shipped"] = json.loads(r.stdout.strip().splitlines()[-1])
        except Exception as e:
            out["threads_as_shipped"] = {"unavailable": "%s: %s" % (type(e).__name__, e)}
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = _reference_arm()
    total = args.steps + args.warmup
    rows = _rows_for_budget(arm, total, 420.0)
    L, R, lg = _sample_inputs(rows)
    for _ in range(args.warmup):
        _cpu_step(arm, L, R, lg)
    arm["native_s"][0] = 0.0
    t0 = time.time()
    for _ in range(args.steps):
        _cpu_step(arm, L, R, lg)
    dt = time.time() - t0
    frac = rows / float(H_IMG)
    value = args.steps * frac / dt
    sample = ("each step = %d of 540 rows (x960, D=192) of one pair through %s + softmax/regression; %d host cpus"
              % (rows, arm["what"], os.cpu_count() or 0))
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 4), "unit": "pairs/s",
        "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(1e3 * dt / args.steps, 2), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "configs[1]: SceneFlow-shaped 540x960 D=192 MS features + soft-argmin, CPU reference, "
                               "one pair per step (%s)" % ("full frames" if rows == H_IMG else "%d-row band" % rows),
                   "sample_rows": rows, "pairs_per_step": 1},
        "cpu_baseline": {"value": round(value, 4), "unit": "pairs/s", "cores": arm["cores"], "kind": arm["kind"],
                         "sample": sample,
                         "native_only_pairs_per_s": round(args.steps * frac / max(arm["native_s"][0], 1e-9), 4)},
        "e2e": {"value": round(value, 4), "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cpu-sample", default=None, help="internal: time one reference step with this oracle/_ref build")
    ap.add_argument("--budget", type=float, default=15.0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's outputs to DIR/<name>.npy (--impl ours)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.cpu_sample:
        print(json.dumps(_cpu_sample_one(args.cpu_sample, args.budget)))
        return
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
