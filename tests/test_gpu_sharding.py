"""GPU: the slab-sharded path (three kernel phases + merges) against the single-pass
path, first with two virtual ranks on one GPU, then -- when the box has >= 2 GPUs -- as
two real ranks over NCCL."""
import ctypes
import os
import socket

import numpy as np
import pytest

from tests._synth import bordered_pair

pytestmark = pytest.mark.gpu
AML_ATOL = 2e-6


def _two_virtual_ranks(ms, L, R, D, border):
    import torch
    from msnets_b200 import _lib, cbmv, sharding
    lib = _lib.lib()
    N, (H, W) = 1, L.shape
    l, r = torch.from_numpy(L[None]).cuda(), torch.from_numpy(R[None]).cuda()
    st = torch.cuda.current_stream().cuda_stream
    slabs = []
    for rank in range(2):
        d0, dn = sharding.shard_range(D, rank, 2)
        p = cbmv.make_params(D, board_h=border, board_w_left=border, board_w_right=border, d_begin=d0, d_count=dn)
        shape = cbmv.output_shape(N, H, W, p)
        ws = torch.empty(lib.msn_ms_slab_workspace_bytes(N, H, W, ctypes.byref(p)), dtype=torch.uint8, device="cuda")
        out = torch.empty(shape, dtype=torch.float32, device="cuda")
        mins = torch.empty((N, 4, shape[3], shape[4]), dtype=torch.float32, device="cuda")
        _lib.check(lib.msn_ms_slab_phase_a_dev(l.data_ptr(), r.data_ptr(), N, H, W, ctypes.byref(p), None,
                                               out.data_ptr(), mins.data_ptr(), ws.data_ptr(), ws.numel(), st))
        slabs.append((p, out, mins, shape))
    gmin = torch.minimum(slabs[0][2], slabs[1][2])           # what all-reduce(min) yields
    dens = []
    for p, out, _, shape in slabs:
        den = torch.empty_like(gmin)
        _lib.check(lib.msn_ms_slab_phase_b_dev(out.data_ptr(), gmin.data_ptr(), N, shape[3], shape[4],
                                               ctypes.byref(p), den.data_ptr(), st))
        dens.append(den)
    gden = dens[0] + dens[1]                                  # what all-reduce(sum) yields
    for p, out, _, shape in slabs:
        _lib.check(lib.msn_ms_slab_phase_c_dev(out.data_ptr(), gmin.data_ptr(), gden.data_ptr(), N, shape[3],
                                               shape[4], ctypes.byref(p), st))
    torch.cuda.synchronize()
    return torch.cat([slabs[0][1], slabs[1][1]], dim=2)[0].cpu().numpy()


def test_slab_phases_match_single_pass(oracle):
    import msnets_b200 as ms
    L, R = bordered_pair(36, 70, 11, border=10, patches=True)
    D = 40
    got = _two_virtual_ranks(ms, L, R, D, 10)
    want = oracle.ms_features(L, R, D)
    assert np.array_equal(got[:4], want[:4])
    assert np.abs(got[4:] - want[4:]).max() <= AML_ATOL
    fused = ms.cbmv.ms_features(L, R, D, board_h=10, board_w_left=10, board_w_right=10)
    assert np.array_equal(got[:4], fused[:4]) and np.abs(got[4:] - fused[4:]).max() <= AML_ATOL


def _virtual_exchange_ranks(L, R, D, border, world):
    """`world` virtual ranks of the FUSED slab exchange inside one process on one GPU: one launch per
    rank, each on its own stream, all resident at once (the tiles wait for each other's minima), tables
    wired by plain device pointers."""
    import torch
    from msnets_b200 import sharding
    N, (H, W) = 1, L.shape
    l, r = torch.from_numpy(L[None]).cuda(), torch.from_numpy(R[None]).cuda()
    ranks = [sharding.ExchangeSlabMSFeatures(N, H, W, maxdisp=D, rank=k, world=world, connect=False, board_h=border,
                                             board_w_left=border, board_w_right=border) for k in range(world)]
    ptrs = [x.table_ptr for x in ranks]
    for x in ranks:
        x.wire(ptrs)
    outs = []
    for frame in range(3):     # three frames: both halves of the double-buffered tables and an epoch wrap of the half
        streams = [torch.cuda.Stream() for _ in ranks]
        torch.cuda.synchronize()
        outs = []
        for x, st in zip(ranks, streams):
            with torch.cuda.stream(st):
                outs.append(x(l, r))
        torch.cuda.synchronize()
    vol = torch.cat(outs, dim=2)[0].cpu().numpy()
    for x in ranks:
        x.close()
    return vol


@pytest.mark.parametrize("world,H,W,D", [(1, 36, 70, 40), (2, 36, 70, 40), (2, 50, 116, 64), (4, 30, 84, 96),
                                          (1, 34, 70, 384), (2, 30, 52, 640),   # two sub-slabs per rank (192 / 160 wide)
                                          (1, 36, 70, 191), (2, 36, 70, 262)])
def test_fused_slab_exchange_virtual_ranks(oracle, world, H, W, D):
    """msn_ms_slab_fused_dev: the slab kernel with the min / denominator exchange inside the tile."""
    import msnets_b200 as ms
    L, R = bordered_pair(H, W, 11 + world, border=10, patches=True)
    got = _virtual_exchange_ranks(L, R, D, 10, world)
    want = oracle.ms_features(L, R, D)
    assert got.shape == want.shape
    assert np.array_equal(got[:4], want[:4])
    assert np.abs(got[4:] - want[4:]).max() <= AML_ATOL
    if world == 1 and D <= 192:   # one rank, one sub-slab: the same sums in the same order as the single-pass kernel
        fused = ms.cbmv.ms_features(L, R, D, board_h=10, board_w_left=10, board_w_right=10)
        assert np.array_equal(got, fused)


@pytest.mark.parametrize("world,D", [(2, 64), (4, 96), (1, 384)])
def test_fused_slab_wta_parts_merge(oracle, world, D):
    """The slab kernels' WTA by-product per virtual rank / sub-slab, merged by msn_wta_merge_dev, equals
    (argmin, min, second min) over ALL disparities of channels 0-3."""
    import torch
    from msnets_b200 import sharding
    L, R = bordered_pair(30, 84, 21, border=10, patches=True)
    H, W = L.shape
    l, r = torch.from_numpy(L[None]).cuda(), torch.from_numpy(R[None]).cuda()
    ranks = [sharding.ExchangeSlabMSFeatures(1, H, W, maxdisp=D, rank=k, world=world, connect=False, board_h=10,
                                             board_w_left=10, board_w_right=10) for k in range(world)]
    ptrs = [x.table_ptr for x in ranks]
    for x in ranks:
        x.wire(ptrs)
    streams = [torch.cuda.Stream() for _ in ranks]
    parts = [x.empty_wta_parts() for x in ranks]
    torch.cuda.synchronize()
    outs = []
    for x, st, wp in zip(ranks, streams, parts):
        with torch.cuda.stream(st):
            outs.append(x(l, r, wta=wp))
    torch.cuda.synchronize()
    cat = [torch.cat([p[i] for p in parts], dim=0) for i in range(3)]       # what the all-gather yields
    idx, m1, m2 = sharding.slab_wta_merge(*cat)
    torch.cuda.synchronize()
    want = oracle.ms_features(L, R, D)
    for c in range(4):
        wi, w1, w2 = oracle.wta(np.ascontiguousarray(want[c].transpose(1, 2, 0)))
        assert np.array_equal(idx[0, c].cpu().numpy(), wi)
        assert np.array_equal(m1[0, c].cpu().numpy(), w1) and np.array_equal(m2[0, c].cpu().numpy(), w2)
    for x in ranks:
        x.close()


def test_fused_slab_exchange_narrow_sub_slabs(oracle, monkeypatch):
    """The exchange kernel with slabs cut into sub-slabs at most 96 wide instead of 192: four of 96 disparities
    at D = 384 on one rank, four of 80 per rank at D = 640 on two, beside slabs narrow enough to stay whole."""
    from msnets_b200 import sharding
    monkeypatch.setattr(sharding.ExchangeSlabMSFeatures, "TILE_D_CHOICES", (96,))
    for world, H, W, D in ((2, 36, 70, 40), (1, 34, 70, 384), (2, 30, 52, 640), (2, 34, 100, 128)):
        L, R = bordered_pair(H, W, 31 + world, border=10, patches=True)
        got = _virtual_exchange_ranks(L, R, D, 10, world)
        want = oracle.ms_features(L, R, D)
        assert np.array_equal(got[:4], want[:4])
        assert np.abs(got[4:] - want[4:]).max() <= AML_ATOL


def test_slab_wta_and_soft_argmin_single_rank(oracle):
    import torch
    import msnets_b200 as ms
    from msnets_b200 import sharding
    rng = np.random.default_rng(3)
    x = (rng.standard_normal((2, 48, 10, 16)) * 3).astype(np.float32)
    t = torch.from_numpy(x).cuda()
    parts = []
    for d0, dn in (sharding.shard_range(48, r, 3) for r in range(3)):
        part = torch.empty((2, 3, 10, 16), dtype=torch.float32, device="cuda")
        ms._lib.check(ms._lib.lib().msn_soft_argmin_partial_dev(t[:, d0:d0 + dn].contiguous().data_ptr(), 2, dn, 10,
                                                                16, d0, part.data_ptr(), None))
        parts.append(part)
    parts = torch.stack(parts).contiguous()
    disp = torch.empty((2, 10, 16), dtype=torch.float32, device="cuda")
    ms._lib.check(ms._lib.lib().msn_soft_argmin_merge_dev(parts.data_ptr(), 3, 2, 10, 16, disp.data_ptr(), None))
    torch.cuda.synchronize()
    assert np.abs(disp.cpu().numpy() - oracle.soft_argmin(x)).max() <= 1e-3
    cost = torch.from_numpy(x[0]).cuda()                     # [D,h,w] plane layout, negative values included
    keys = []
    for d0, dn in (sharding.shard_range(48, r, 2) for r in range(2)):
        k = torch.empty((10, 16), dtype=torch.int64, device="cuda")
        ms._lib.check(ms._lib.lib().msn_wta_keys_dev(cost[d0:d0 + dn].contiguous().data_ptr(), 160, dn, 1, d0,
                                                     k.data_ptr(), None))
        keys.append(k)
    merged = torch.minimum(keys[0], keys[1])
    am, m1 = sharding.wta_key_unpack(merged.cpu())
    assert np.array_equal(am.numpy(), x[0].argmin(0).astype(np.int32)) and np.array_equal(m1.numpy(), x[0].min(0))


def _nccl_worker(rank, world, port, ret):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method="tcp://127.0.0.1:%d" % port, rank=rank, world_size=world)
    try:
        import msnets_b200
        from msnets_b200 import cbmv, sharding
        L, R = bordered_pair(48, 96, 77, border=10, patches=True)
        D = 64
        l, r = torch.from_numpy(L[None]).cuda(), torch.from_numpy(R[None]).cuda()
        slab = sharding.SlabShardedMSFeatures(1, L.shape[0], L.shape[1], maxdisp=D, board_h=10, board_w_left=10,
                                              board_w_right=10)
        out = slab(l, r)
        full = cbmv.MSFeatureExtractor(1, L.shape[0], L.shape[1], maxdisp=D, board_h=10, board_w_left=10,
                                       board_w_right=10)(l, r)
        mine = full[:, :, slab.d_begin:slab.d_begin + slab.d_count]
        exact = bool(torch.equal(out[:, :4], mine[:, :4]))
        err = float((out[:, 4:] - mine[:, 4:]).abs().max())
        # the same slab with the exchange fused into the kernel: tables wired through CUDA IPC handles
        xs = sharding.ExchangeSlabMSFeatures(1, L.shape[0], L.shape[1], maxdisp=D, board_h=10, board_w_left=10,
                                             board_w_right=10)
        for _ in range(3):
            out2 = xs(l, r)
        torch.cuda.synchronize()
        exact = exact and bool(torch.equal(out2[:, :4], mine[:, :4]))
        err = max(err, float((out2[:, 4:] - mine[:, 4:]).abs().max()))
        dist.barrier()
        xs.close()
        am, m1 = sharding.slab_wta(out[0, 1].contiguous(), slab.d_begin)       # NCC channel, D-sharded
        wta_ok = bool(torch.equal(am.long(), full[0, 1].argmin(0)))
        logits = torch.randn((1, D, 28, 76), generator=torch.Generator("cuda").manual_seed(1), device="cuda")
        disp = sharding.slab_soft_argmin(logits[:, slab.d_begin:slab.d_begin + slab.d_count].contiguous(), slab.d_begin)
        from msnets_b200 import regression
        sa_err = float((disp - regression.soft_argmin(logits)).abs().max())
        ret[rank] = (exact, err, wta_ok, sa_err)
    finally:
        dist.destroy_process_group()


def test_slab_sharding_two_gpus_nccl():
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (run under gpurun --gpus 2)")
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mgr = mp.get_context("spawn").Manager()
    ret = mgr.dict()
    mp.spawn(_nccl_worker, args=(2, port, ret), nprocs=2, join=True)
    for rank in range(2):
        exact, err, wta_ok, sa_err = ret[rank]
        assert exact and err <= AML_ATOL and wta_ok and sa_err <= 1e-3, (rank, ret[rank])


def test_row_band_of_the_fused_volume(oracle):
    """msn_ms_params.row_begin / row_count: a band of rows through the fused kernel equals those rows of the full
    volume bit for bit -- the SAD-of-Sobel table of a row is built from row 0 even when only the band is scanned."""
    import torch
    import msnets_b200 as ms
    L, R = bordered_pair(120, 84, 5, border=10, patches=True)
    H, W = L.shape
    l, r = torch.from_numpy(L[None]).cuda(), torch.from_numpy(R[None]).cuda()
    kw = dict(maxdisp=48, board_h=10, board_w_left=10, board_w_right=10)
    full = ms.cbmv.MSFeatureExtractor(1, H, W, **kw)(l, r)
    for y0, yn in ((0, 17), (31, 60), (95, 25), (119, 1)):
        band = ms.cbmv.MSFeatureExtractor(1, H, W, row_begin=y0, row_count=yn, **kw)(l, r)
        assert tuple(band.shape) == (1, 8, 48, yn, 84)
        assert torch.equal(band, full[:, :, :, y0:y0 + yn])
    want = oracle.ms_features(L, R, 48)
    assert np.array_equal(full[0, :4].cpu().numpy(), want[:4])


@pytest.mark.parametrize("world,bands,H,W,D", [(4, 2, 44, 84, 64), (4, 4, 40, 52, 40), (2, 2, 36, 70, 40)])
def test_fused_slab_exchange_with_row_bands(oracle, world, bands, H, W, D):
    """2-D sharding of one frame: row bands x disparity slabs, virtual ranks on one GPU; only the ranks of a band
    trade minima / denominators.  The assembled volume equals the reference."""
    import torch
    from msnets_b200 import sharding
    L, R = bordered_pair(H, W, 41 + world, border=10, patches=True)
    Hb, Wb = L.shape
    l, r = torch.from_numpy(L[None]).cuda(), torch.from_numpy(R[None]).cuda()
    ranks = [sharding.ExchangeSlabMSFeatures(1, Hb, Wb, maxdisp=D, rank=k, world=world, connect=False, row_bands=bands,
                                             board_h=10, board_w_left=10, board_w_right=10) for k in range(world)]
    ptrs = [x.table_ptr for x in ranks]
    for x in ranks:
        x.wire(ptrs)
    streams = [torch.cuda.Stream() for _ in ranks]
    torch.cuda.synchronize()
    outs = []
    for x, st in zip(ranks, streams):
        with torch.cuda.stream(st):
            outs.append(x(l, r))
    torch.cuda.synchronize()
    slabs = world // bands
    rows = [torch.cat(outs[b * slabs:(b + 1) * slabs], dim=2) for b in range(bands)]     # slabs along D
    got = torch.cat(rows, dim=3)[0].cpu().numpy()                                        # bands along rows
    want = oracle.ms_features(L, R, D)
    assert got.shape == want.shape
    assert np.array_equal(got[:4], want[:4])
    assert np.abs(got[4:] - want[4:]).max() <= AML_ATOL
    for x in ranks:
        x.close()
    assert sharding.ExchangeSlabMSFeatures.default_row_bands(640, 8) == 4
    assert sharding.ExchangeSlabMSFeatures.default_row_bands(640, 4) == 2
    assert sharding.ExchangeSlabMSFeatures.default_row_bands(640, 2) == 1
    assert sharding.ExchangeSlabMSFeatures.default_row_bands(192, 8) == 8
