"""world_size-2 gloo tests (CPU) of the multi-rank host logic: gradient all-reduce, weight broadcast,
sharding of the Monte Carlo batch and the (sum, sum of squares, n) combination used by integrate()."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from nf_b200.normalizing_flows.manager import BasicManager, PWQuadManager, shard_bounds


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.manual_seed(100 + rank)                      # ranks start from DIFFERENT weights
        NF = PWQuadManager(n_flow=3)
        NF.create_model(3, 4, [8, 8])
        before = torch.cat([p.detach().reshape(-1) for p in NF._model.parameters()]).clone()
        NF._sync_model()
        after = torch.cat([p.detach().reshape(-1) for p in NF._model.parameters()])
        gathered = [torch.zeros_like(after) for _ in range(world)]
        dist.all_gather(gathered, after)
        same = all(torch.equal(g, gathered[0]) for g in gathered)
        changed = (rank == 0) == torch.equal(before, after)
        # gradient all-reduce: rank r contributes r+1 everywhere -> sum = world(world+1)/2
        params = list(NF._model.parameters())
        for i, p in enumerate(params):
            p.grad = None if (i == 1 and rank == 1) else torch.full_like(p, float(rank + 1))
        BasicManager._allreduce_grads(params)
        expect = [world * (world + 1) / 2] * len(params)
        expect[1] = 1.0                                    # rank 1 had no gradient there
        grads_ok = all(torch.allclose(p.grad, torch.full_like(p, e)) for p, e in zip(params, expect))
        # fast path: the gradients are views of ONE flat buffer (what nis_flow_backward + autograd leave behind):
        # a single in-place collective, the views stay views; the buffer lives where the parameters do (create_model
        # places them on cuda:0 when a GPU is present)
        dev = params[0].device
        flat = torch.arange(sum(p.numel() for p in params), dtype=torch.float32, device=dev) * (rank + 1)
        off = 0
        for p in params:
            p.grad = flat[off:off + p.numel()].view(p.shape)
            off += p.numel()
        ptrs = [p.grad.data_ptr() for p in params]
        BasicManager._allreduce_grads(params)
        want = torch.arange(flat.numel(), dtype=torch.float32, device=dev) * (world * (world + 1) / 2)
        grads_ok = grads_ok and torch.equal(flat, want) and ptrs == [p.grad.data_ptr() for p in params] and \
            torch.equal(torch.cat([p.grad.reshape(-1) for p in params]), want)
        # latent-point streams: identical user seed on every rank -> different points per rank, same on re-run
        torch.manual_seed(5)
        g1 = BasicManager._rank_generator(torch.device("cpu"), rank, world)
        pts = torch.rand(64, 3, generator=g1)
        torch.manual_seed(5)
        g2 = BasicManager._rank_generator(torch.device("cpu"), rank, world)
        again = torch.rand(64, 3, generator=g2)
        allpts = [torch.zeros_like(pts) for _ in range(world)]
        dist.all_gather(allpts, pts)
        grads_ok = grads_ok and torch.equal(pts, again) and not torch.equal(allpts[0], allpts[1])
        # sharded moments == single-process moments
        g = torch.Generator().manual_seed(7)
        v = torch.rand(1003, generator=g, dtype=torch.float64)
        first, count = shard_bounds(1003, rank, world)
        mine = v[first:first + count]
        m = torch.stack((mine.sum(), (mine ** 2).sum(), torch.tensor(float(count), dtype=torch.float64)))
        dist.all_reduce(m)
        full = torch.stack((v.sum(), (v ** 2).sum(), torch.tensor(1003.0, dtype=torch.float64)))
        moments_ok = torch.allclose(m, full, rtol=1e-13)
        out.put((rank, same, changed, grads_ok, moments_ok))
    finally:
        dist.destroy_process_group()


def test_two_rank_gloo_host_logic():
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    res = [out.get(timeout=180) for _ in procs]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    for rank, same, changed, grads_ok, moments_ok in res:
        assert same, "weights differ across ranks after broadcast"
        assert changed, "rank 0 must keep its weights, the others must take rank 0's"
        assert grads_ok and moments_ok


@pytest.mark.parametrize("n,world", [(10, 1), (10, 3), (7, 8), (1 << 26, 8), (0, 2)])
def test_shards_partition_the_batch(n, world):
    nxt = 0
    for r in range(world):
        first, count = shard_bounds(n, r, world)
        assert first == nxt and count >= 0
        nxt += count
    assert nxt == n
    counts = [shard_bounds(n, r, world)[1] for r in range(world)]
    assert max(counts) - min(counts) <= 1
