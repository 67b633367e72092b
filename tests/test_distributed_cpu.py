"""Host-side distributed logic on CPU: world_size-2 gloo process groups
(127.0.0.1) exercising init_distributed_mode, shard_range, the packed gradient
all-reduce and the global-batch Frobenius loss (SURVEY.md §8e)."""
import os
import socket
import types

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import videoad_b200 as V


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank),
                      MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    args = types.SimpleNamespace(dist_url="env://")
    V.init_distributed_mode(args)                       # gloo on a CPU-only host, nccl with CUDA
    assert (args.rank, args.world_size, args.gpu) == (rank, world, rank)
    assert dist.get_backend() == "gloo"
    out = {}
    # contiguous clip sharding covers every item exactly once
    a, b = V.shard_range(7)
    out["shard"] = (a, b)
    # packed all-reduce: three tensors, one collective, summed in place
    g = torch.Generator().manual_seed(100 + rank)
    ts = [torch.randn(4, 3, generator=g), torch.randn(5, generator=g), torch.randn(1, generator=g)]
    ref = [t.clone() for t in ts]
    V.allreduce_sum_packed(ts).finish()
    out["packed"] = [t.numpy().copy() for t in ts]
    out["local"] = [t.numpy().copy() for t in ref]
    h = V.allreduce_sum_packed([ref[0].clone()], average=True, async_op=True)
    h.finish()
    # global Frobenius loss: value = sqrt(sum over ranks), gradient flows to the local sum of squares
    v = torch.tensor([float(rank + 1)]).requires_grad_(True)
    s = (v * v).sum().reshape(1)
    L = V.global_frobenius(s)
    L.backward()
    out["loss"] = float(L)
    out["grad"] = float(v.grad)
    Lc = V.global_frobenius((v.detach() ** 2).sum().reshape(1), ddp_compat=True)
    out["loss_compat"] = float(Lc)
    # the reductions of the global-batch memory (SURVEY 8e): column maxima (MAX), column sums and update sums (SUM)
    from videoad_b200.memory import _dist_reduce
    out["colmax"] = _dist_reduce(torch.tensor([1.0 + rank, 5.0 - 3 * rank, -2.0]), "max").numpy().copy()
    out["colsum"] = _dist_reduce(torch.tensor([1.0 + rank, 10.0]), "sum").numpy().copy()
    # scoring under data parallelism (SURVEY 8e): every rank scored its own videos (contiguous shard_range), the merged
    # list comes back in video order on every rank
    lo, hi = V.shard_range(5)
    local = [(i, np.full(3, float(i)), np.arange(3) % 2) for i in range(lo, hi)]
    merged = V.gather_video_scores(local)
    out["gathered"] = [(i, s_.tolist(), l_.tolist()) for i, s_, l_ in merged]
    # print is muted on non-master ranks (utils/distritributed_model.py:23-35)
    import builtins
    out["print_wrapped"] = getattr(builtins.print, "_vadc_wrapped", False)
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_gloo(monkeypatch):
    # the workers see no GPU, so they take the gloo path on any host (with CUDA, init_distributed_mode picks nccl and
    # binds rank r to cuda:r, which a one-GPU machine does not have)
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    try:
        for p in procs:
            p.start()
        res = dict(q.get(timeout=120) for _ in range(world))
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
    finally:
        for p in procs:                                  # a worker left waiting for a dead peer must not outlive the test
            if p.is_alive():
                p.kill()
                p.join()
    assert res[0]["shard"] == (0, 4) and res[1]["shard"] == (4, 7)
    for i in range(3):
        want = res[0]["local"][i] + res[1]["local"][i]
        np.testing.assert_allclose(res[0]["packed"][i], want, rtol=1e-6)
        np.testing.assert_allclose(res[1]["packed"][i], want, rtol=1e-6)
    for r in (0, 1):
        np.testing.assert_allclose(res[r]["colmax"], [2.0, 5.0, -2.0])
        np.testing.assert_allclose(res[r]["colsum"], [3.0, 20.0])
    for r in (0, 1):
        assert res[r]["gathered"] == [(i, [float(i)] * 3, [0, 1, 0]) for i in range(5)]
    Lg = (1.0 + 4.0) ** 0.5
    for r in (0, 1):
        assert abs(res[r]["loss"] - Lg) < 1e-6
        assert abs(res[r]["grad"] - (r + 1) / Lg) < 1e-6        # d sqrt(S)/dv_r = v_r / sqrt(S)
        assert abs(res[r]["loss_compat"] - (r + 1)) < 1e-6       # per-rank norm (reference DDP behaviour)
        assert res[r]["print_wrapped"]


def test_single_process_helpers():
    assert V.shard_range(10, 0, 3) == (0, 4) and V.shard_range(10, 1, 3) == (4, 7) and V.shard_range(10, 2, 3) == (7, 10)
    assert V.shard_range(2, 3, 4) == (2, 2)                    # more ranks than items: empty shard
    t = torch.ones(3)
    V.allreduce_sum_packed([t]).finish()                       # no process group: a no-op
    assert torch.equal(t, torch.ones(3))
    assert abs(float(V.global_frobenius(torch.tensor([9.0]))) - 3.0) < 1e-7
    V.fix_random_seeds(31)
    a = torch.rand(2)
    V.fix_random_seeds(31)
    assert torch.equal(a, torch.rand(2))
    assert V.get_sha().startswith("sha:")


def test_numa_helpers_cpu():
    """cpulist parsing and the no-GPU behaviour of the NUMA-local allocation helper"""
    import os
    import videoad_b200 as V
    from videoad_b200.distributed import _parse_cpulist
    assert _parse_cpulist("0-3,8,10-11\n") == {0, 1, 2, 3, 8, 10, 11}
    assert _parse_cpulist("") == set()
    before = os.sched_getaffinity(0)
    with V.numa_local(0) as ctx:          # no CUDA device here: topology unreadable -> no-op
        assert ctx.cpus == set() or ctx.cpus <= before
    assert os.sched_getaffinity(0) == before
