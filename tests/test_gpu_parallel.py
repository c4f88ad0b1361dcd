"""NCCL tests of the batch-sharded QP layer on >= 2 GPUs (SURVEY 8e, BASELINE config 5): the real QPFunction on every
rank, inputs scattered from rank 0 over NCCL, z* gathered, shared-parameter gradients all-reduced with the `.mean(0)`
rule. Skipped on a machine with one GPU; run on two or more with `python -m pytest tests/test_gpu_parallel.py -m gpu`."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _worker(rank, world, port, results):
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from qpth_b200 import QPFunction, parallel, qp as qpmod
        from qpth_b200.problems import random_qp_batch
        # one kernel family everywhere: "auto" would pick by batch size (a 64-QP shard vs the 512-QP reference solve on rank
        # 0), and the families differ in the summation order of the W passes (1e-13), which a bit-for-bit check would see
        qpmod.MODE = "latency"
        f = QPFunction(verbose=-1, check_Q_spd=False)
        e = torch.Tensor().to(dev).double()
        # (1) ragged scatter / gather through sharded_qp, equality-constrained problems
        nb = 37
        pr = random_qp_batch(nb, 30, 20, 5, seed=11)
        T = {k: (torch.tensor(pr[k], dtype=torch.float64, device=dev) if rank == 0 else None) for k in ("Q", "p", "G", "h", "A", "b")}
        z = parallel.sharded_qp(f, T["Q"], T["p"], T["G"], T["h"], T["A"], T["b"], nb, device=dev)
        if rank == 0:
            z1 = f(T["Q"], T["p"], T["G"], T["h"], T["A"], T["b"])
            results["ragged_equal"] = bool(torch.equal(z, z1))
        # (2) the config-5 job (equal shards, dist.scatter / dist.gather), C2-sized QPs
        nb5 = 64 * world
        pr5 = random_qp_batch(nb5, 100, 100, 0, seed=12)
        glob = {k: torch.tensor(pr5[k], dtype=torch.float64, device=dev) for k in ("Q", "p", "G", "h")} if rank == 0 else None
        out = parallel.sharded_qp_timed(f, glob, nb5, 100, 100, dev, include_comm=True)
        if rank == 0:
            z1 = f(glob["Q"], glob["p"], glob["G"], glob["h"], e, e)
            results["c5_equal"] = bool(torch.equal(out["z"], z1))
            results["c5_ms"] = out["ms"]
        # (3) shared G: per-shard mean gradients -> global batch mean (qp.py:159-177) through an all-reduce
        nbs = 16 * world + 3
        prs = random_qp_batch(nbs, 20, 15, 0, seed=13)
        Gs = torch.tensor(prs["G"][0], dtype=torch.float64, device=dev)
        lo, hi = parallel.shard_bounds(nbs, world, rank)
        t = {k: torch.tensor(prs[k][lo:hi], dtype=torch.float64, device=dev, requires_grad=True) for k in ("Q", "p", "h")}
        Gl = Gs.clone().requires_grad_(True)
        zl = f(t["Q"], t["p"], Gl, t["h"], e, e)
        dl = torch.tensor(prs["dl"][lo:hi], dtype=torch.float64, device=dev)
        zl.backward(dl)
        gG = parallel.allreduce_shared_grad(Gl.grad, hi - lo, nbs)
        if rank == 0:
            tf = {k: torch.tensor(prs[k], dtype=torch.float64, device=dev, requires_grad=True) for k in ("Q", "p", "h")}
            Gf = Gs.clone().requires_grad_(True)
            zf = f(tf["Q"], tf["p"], Gf, tf["h"], e, e)
            zf.backward(torch.tensor(prs["dl"], dtype=torch.float64, device=dev))
            results["shared_grad_err"] = float((gG - Gf.grad).abs().max() / Gf.grad.abs().max())
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_sharded_qp_over_nccl():
    world = min(torch.cuda.device_count(), 8)
    mgr = mp.Manager()
    results = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), results), nprocs=world, join=True)
    assert results["ragged_equal"] and results["c5_equal"], dict(results)
    assert results["shared_grad_err"] < 1e-9, dict(results)
