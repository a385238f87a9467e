"""N = 2 on real GPUs over NCCL (needs two devices: `python -m pytest tests/test_gpu_multi.py -m gpu` on a machine with
two GPUs; skipped with one).  Batch-sharded replicas: the reduced parameter grads of the two ranks must equal the sum
of the two single-GPU grads, and HostStep(reduce_fn=...) must equal autograd + allreduce_grads."""
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _make(dev, D, L, seed=5):
    import hyena_dna_b200 as H
    torch.manual_seed(seed)
    return H.HyenaOperator(D, L, emb_dim=5, w=10.0, lr_pos_emb=0.0).to(dev)


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    torch.backends.cuda.matmul.allow_tf32 = False
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        import hyena_dna_b200 as H
        B, L, D = 1, 8192, 32
        op = _make(dev, D, L)
        params = [p for p in op.parameters() if p.requires_grad]
        us = [torch.randn(B, L, D, generator=torch.Generator().manual_seed(10 + r)) for r in range(world)]
        dys = [torch.randn(B, L, D, generator=torch.Generator().manual_seed(20 + r)) for r in range(world)]
        # single-GPU grads of every rank's shard, computed locally (same weights everywhere)
        single = []
        for r in range(world):
            for p in params:
                p.grad = None
            op(us[r].to(dev)).backward(dys[r].to(dev))
            single.append([p.grad.clone() for p in params])
        expect = [sum(g[i] for g in single) for i in range(len(params))]
        # data-parallel step: own shard + flat all-reduce
        for p in params:
            p.grad = None
        op(us[rank].to(dev)).backward(dys[rank].to(dev))
        H.distributed.allreduce_grads(params)
        torch.cuda.synchronize()
        for p, e in zip(params, expect):
            tol = 1e-5 * max(1.0, float(e.abs().max())) + 1e-4 * e.abs()
            assert bool(((p.grad - e).abs() <= tol).all()), "reduced grads != sum of per-rank grads"
        # HostStep with reduce_fn == autograd + allreduce_grads
        if H.ops.gemm_mode() == "bf16x9" or hasattr(H.ops, "proj_mode"):
            hs = H.HostStep(op, B, L, chunks=2)
            uh, dyh = us[rank].pin_memory(), dys[rank].pin_memory()
            yh, duh = torch.empty(B, L, D).pin_memory(), torch.empty(B, L, D).pin_memory()
            gh = [torch.empty(p.shape).pin_memory() for p in params]
            hs.step(uh, dyh, yh, duh, gh, H.distributed.allreduce_tensors)
            torch.cuda.synchronize()
            for g, p in zip(gh, params):
                tol = 1e-5 * max(1.0, float(p.grad.abs().max())) + 2e-3 * p.grad.abs().cpu()
                assert bool(((g - p.grad.cpu()).abs() <= tol).all()), "HostStep(reduce_fn) != autograd + allreduce"
        out.put((rank, "ok"))
    except Exception as e:   # pragma: no cover
        import traceback
        out.put((rank, traceback.format_exc()[-1500:]))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
def test_two_rank_nccl_reduced_grads_equal_sum_of_single_gpu_grads():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    res = [out.get(timeout=500) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, "ok"), (1, "ok")], res
