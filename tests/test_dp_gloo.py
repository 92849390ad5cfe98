"""CPU tests (world_size 2, gloo): the data-parallel host logic - view sharding and the flat gradient bucket whose
single all-reduce replaces the per-parameter reductions DDP would do."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn as nn


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from ngp_b200.parallel import FlatGradBucket, shard_views
        torch.manual_seed(0)                       # identical replicas
        net = nn.Sequential(nn.Linear(6, 5), nn.ReLU(), nn.Linear(5, 3))
        table = nn.Parameter(torch.randn(40, 2))
        params = [table] + list(net.parameters())
        bucket = FlatGradBucket(params, torch.device("cpu"), extra=1)
        assert bucket.numel == sum(p.numel() for p in params) and bucket.flat.numel() == bucket.numel + 1
        # every rank owns a contiguous share of 8 "views"
        g = torch.Generator().manual_seed(1)
        views = torch.randn(8, 16, 6, generator=g)
        idx = torch.randint(0, 40, (8, 16), generator=g)
        first, count = shard_views(8, rank, world)
        bucket.zero()
        bucket.attach()
        x, ii = views[first:first + count].reshape(-1, 6), idx[first:first + count].reshape(-1)
        loss = (net(x) * table[ii].sum(-1, keepdim=True)).sum()
        loss.backward()
        assert all(p.grad.data_ptr() >= bucket.flat.data_ptr() for p in params)   # autograd wrote into the bucket
        bucket.extra[0] = float(count)                      # piggy-backed scalar (e.g. a sample count)
        bucket.all_reduce(average=False)
        # single-process ground truth over all 8 views
        torch.manual_seed(0)
        net2 = nn.Sequential(nn.Linear(6, 5), nn.ReLU(), nn.Linear(5, 3))
        table2 = nn.Parameter(table.detach().clone())
        (net2(views.reshape(-1, 6)) * table2[idx.reshape(-1)].sum(-1, keepdim=True)).sum().backward()
        want = torch.cat([table2.grad.reshape(-1)] + [p.grad.reshape(-1) for p in net2.parameters()])
        ok = torch.allclose(bucket.flat[:bucket.numel], want, rtol=1e-5, atol=1e-6) and bucket.extra[0].item() == 8.0
        out[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


def test_shard_views_partitions_evenly():
    from ngp_b200.parallel import shard_views
    for n, w in [(8, 1), (8, 2), (8, 4), (8, 8), (7, 2), (3, 4)]:
        spans = [shard_views(n, r, w) for r in range(w)]
        assert sum(c for _, c in spans) == n
        assert spans[0][0] == 0 and all(spans[i][0] + spans[i][1] == spans[i + 1][0] for i in range(w - 1))
        assert max(c for _, c in spans) - min(c for _, c in spans) <= 1


def test_flat_bucket_allreduce_equals_single_process_gradient():
    world = 2
    port = _free_port()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, port, out), nprocs=world, join=True)
    assert dict(out) == {0: True, 1: True}


def test_shard_pixels_partitions_every_view_evenly():
    from ngp_b200.parallel import shard_pixels, shard_rows
    for world in (1, 2, 4, 8):
        parts = [shard_pixels(64, 64, r, world) for r in range(world)]
        assert sorted(p for part in parts for p in part) == list(range(64 * 64))
        assert all(len(part) == 64 * 64 // world for part in parts)
        # every rank owns one 8x8 block per block-row: the same mix of image centre and border
        for part in parts:
            rows = sorted({p // 64 for p in part})
            assert rows == list(range(64))
    # tiling that does not divide: interleaved rows
    assert shard_pixels(6, 4, 1, 3) == [r * 4 + c for r in shard_rows(6, 1, 3) for c in range(4)]


def test_owner_slice_partitions_the_flat_buffer():
    from ngp_b200.parallel import owner_slice
    for numel in (8, 1816256, 4 * 1001, 4 * 7):
        for world in (1, 2, 3, 4, 8):
            spans = [owner_slice(numel, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == numel
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            assert all(lo % 4 == 0 and hi % 4 == 0 and lo <= hi for lo, hi in spans)


def _sharded_adam_worker(rank, world, port, out):
    """Host-side model of csrc/adam.cu on CPU tensors: reduce-scatter by reading every rank's bucket, Adam on the owned
    slice with sharded moments, parameters broadcast from their owner - against single-process Adam on the summed grads."""
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from ngp_b200.parallel import gather_owner_slices, owner_slice
        numel, lr, b1, b2, eps = 4 * 53, 1e-2, 0.9, 0.99, 1e-15
        torch.manual_seed(0)
        p = torch.randn(numel)
        p_ref = p.clone()
        m, v = torch.zeros(numel), torch.zeros(numel)           # only [lo, hi) is maintained on this rank
        m_ref, v_ref = torch.zeros(numel), torch.zeros(numel)
        lo, hi = owner_slice(numel, rank, world)
        for t in range(1, 4):
            g_all = [torch.randn(numel, generator=torch.Generator().manual_seed(100 * t + r)) for r in range(world)]
            # P1: rank r sums slice r of every bucket, in rank order
            s = g_all[0][lo:hi].clone()
            for q in range(1, world):
                s += g_all[q][lo:hi]
            gr = s / world
            # P2: Adam on the slice
            m[lo:hi] = m[lo:hi] + (1 - b1) * (gr - m[lo:hi])
            v[lo:hi] = b2 * v[lo:hi] + (1 - b2) * gr * gr
            step = lr / (1 - b1 ** t)
            new = p[lo:hi] - step * m[lo:hi] / (v[lo:hi].sqrt() / (1 - b2 ** t) ** 0.5 + eps)
            # ... written to every replica: here an all_gather of the (padded) slices
            stale = torch.full((numel,), float("nan"))
            stale[lo:hi] = new
            p = gather_owner_slices(stale)
            # single-process reference on the summed gradients
            g = sum(g_all) / world
            m_ref = m_ref + (1 - b1) * (g - m_ref)
            v_ref = b2 * v_ref + (1 - b2) * g * g
            p_ref = p_ref - (lr / (1 - b1 ** t)) * m_ref / (v_ref.sqrt() / (1 - b2 ** t) ** 0.5 + eps)
        ok = torch.isfinite(p).all() and torch.allclose(p, p_ref, rtol=1e-5, atol=1e-6)
        # checkpointing: the sharded moments reassemble to the full ones
        ok = ok and torch.allclose(gather_owner_slices(m), m_ref, rtol=1e-5, atol=1e-7)
        ok = ok and torch.allclose(gather_owner_slices(v), v_ref, rtol=1e-5, atol=1e-9)
        out[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_adam_with_owner_broadcast_equals_single_process_adam(world):
    port = _free_port()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_sharded_adam_worker, args=(world, port, out), nprocs=world, join=True)
    assert dict(out) == {r: True for r in range(world)}
