"""World-size-2 gloo test of the sharded multi-GPU schedule (SURVEY.md §8e) on CPU, with the oracle as the model.
The expected result is composed from single-process decoder calls only: shard-local updates against the replicated
memory, new tokens appended in rank order, then sharded renders."""
import os
import sys

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
V, H, W = 3, 32, 48


def _models():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from helpers import tiny_oracle
    return tiny_oracle(7)


def _views(rank, n=V):
    from must3r_b200 import synthetic as syn
    imgs, ts = syn.synthetic_views(V, H, W, seed=300 + rank)
    return imgs[:n].contiguous(), ts[:n].contiguous()


def _worker(rank, world, port, q, counts=None):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    sys.path.insert(0, ROOT)
    torch.set_num_threads(1)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from must3r_b200.engine import sharded
    enc, dec = _models()
    imgs, ts = _views(rank, counts[rank] if counts else V)
    mem, outs = sharded.inference_sharded(enc, dec, imgs, ts, device="cpu", return_mem=True, view_counts=counts)
    q.put((rank, torch.stack(outs).clone(), [m.clone() for m in mem[0]], mem[1].clone()))
    dist.barrier()
    dist.destroy_process_group()


def _composed_expected(world, counts=None):
    enc, dec = _models()
    counts = counts or [V] * world
    feats = []
    for r in range(world):
        imgs, ts = _views(r, counts[r])
        x, pos = enc(imgs, ts)
        feats.append((x, pos, ts))
    x0, p0, t0 = feats[0]
    mem, _ = dec(x0[None, :2], p0[None, :2], t0[None, :2], None)
    mem = list(mem)
    for s in range(max(counts)):
        new_parts = []
        for r in range(world):
            if (r == 0 and s < 2) or s >= counts[r]:
                continue
            x, pos, ts = feats[r]
            m2, _ = dec(x[None, s:s + 1], pos[None, s:s + 1], ts[None, s:s + 1], tuple(mem))
            Nm = mem[0][0].shape[1]
            new_parts.append([v[:, Nm:] for v in m2[0]])
        if not new_parts:
            continue
        n_old = mem[2]
        N = new_parts[0][0].shape[1]
        mem[0] = [torch.cat([mem[0][l]] + [p[l] for p in new_parts], 1) for l in range(len(mem[0]))]
        lab = torch.arange(n_old, n_old + len(new_parts)).repeat_interleave(N)[None]
        mem[1] = torch.cat([mem[1], lab], 1)
        mem[2] = mem[3] = n_old + len(new_parts)
        mem[4] = mem[1].shape[1]
    renders = []
    for r in range(world):
        x, pos, ts = feats[r]
        _, pm = dec(x[None], pos[None], ts[None], tuple(mem), render=True)
        renders.append(pm[0])
    return mem, renders


def test_world1_equals_reference_chain():
    """No process group: the schedule must be the plain chain (init 2 views, 1 view per step, render)."""
    sys.path.insert(0, ROOT)
    from must3r_b200.engine import sharded
    enc, dec = _models()
    imgs, ts = _views(0)
    mem, outs = sharded.inference_sharded(enc, dec, imgs, ts, device="cpu", return_mem=True)
    x, pos = enc(imgs, ts)
    m, _ = dec(x[None, :2], pos[None, :2], ts[None, :2], None)
    m, _ = dec(x[None, 2:3], pos[None, 2:3], ts[None, 2:3], m)
    _, pm = dec(x[None], pos[None], ts[None], m, render=True)
    assert torch.allclose(torch.stack(outs), pm[0], atol=1e-6)
    assert torch.equal(mem[1], m[1]) and torch.allclose(mem[0][2], m[0][2], atol=1e-6)


@pytest.mark.timeout(300)
@pytest.mark.parametrize("world,counts", [(2, None), (3, [3, 2, 1])])
def test_gloo_matches_composed_oracle(world, counts):
    """world 2 with equal shards; world 3 with a ragged split (a fixed scene ceil-split over the ranks: some ranks sit
    rounds out but still take part in the collective)."""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    import socket
    with socket.socket() as so:           # a port the kernel says is free right now (fixed numbers collide now and then)
        so.bind(("127.0.0.1", 0))
        port = so.getsockname()[1]
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, counts)) for r in range(world)]
    for p in procs:
        p.start()
    got = {}
    for _ in range(world):
        r, outs, mem_vals, labels = q.get(timeout=240)
        got[r] = (outs, mem_vals, labels)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    threads = torch.get_num_threads()
    torch.set_num_threads(1)              # as in the workers: how a CPU GEMM splits its sums depends on the thread count
    try:
        mem, renders = _composed_expected(world, counts)
    finally:
        torch.set_num_threads(threads)
    for r in range(world):
        outs, mem_vals, labels = got[r]
        assert torch.equal(labels, mem[1])                                   # identical memory on every rank
        for l in range(len(mem_vals)):
            assert torch.allclose(mem_vals[l], mem[0][l], atol=1e-6)
        assert torch.allclose(outs, renders[r], atol=1e-5)
    assert torch.equal(got[0][1][0], got[1][1][0])                           # bitwise-equal replicas
