"""Host-side data-parallel logic on CPU: world_size 2, gloo backend, 127.0.0.1 rendezvous."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


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
        from importlib import import_module
        D = import_module("hyena_dna_b200.distributed")
        # batch sharding: ranks own disjoint contiguous slices that cover the batch
        x = torch.arange(5 * 3, dtype=torch.float32).reshape(5, 3)
        mine = D.shard_batch(x)
        lo, hi = D.shard_bounds(5, world, rank)
        assert torch.equal(mine, x[lo:hi])
        # one flat all-reduce of "parameter grads": every rank ends with the sum over ranks
        torch.manual_seed(0)
        params = [torch.nn.Parameter(torch.zeros(4, 3)), torch.nn.Parameter(torch.zeros(7)),
                  torch.nn.Parameter(torch.zeros(2))]
        params[0].grad = torch.full((4, 3), float(rank + 1))
        params[1].grad = torch.arange(7, dtype=torch.float32) * (rank + 1)
        # params[2] has no grad: must be skipped consistently
        n = D.allreduce_grads(params)
        assert n == 12 + 7
        tot = sum(r + 1 for r in range(world))
        assert torch.equal(params[0].grad, torch.full((4, 3), float(tot)))
        assert torch.equal(params[1].grad, torch.arange(7, dtype=torch.float32) * tot)
        D.allreduce_grads(params, average=True)
        assert torch.allclose(params[0].grad, torch.full((4, 3), float(tot)))
        # gather of batch shards restores the global batch order
        y = D.gather_outputs(x[rank * 2: rank * 2 + 2])
        assert torch.equal(y, x[:4])
        # hook-driven two-bucket reducer: same sums as the flat all-reduce, both buckets, reusable across steps
        lin1, lin2 = torch.nn.Linear(3, 4), torch.nn.Linear(4, 2)
        with torch.no_grad():
            for q in list(lin1.parameters()) + list(lin2.parameters()):
                q.copy_(torch.arange(q.numel(), dtype=torch.float32).reshape(q.shape) * 0.01)
        named = [("a.weight", lin1.weight), ("a.bias", lin1.bias), ("implicit_filter.w", lin2.weight),
                 ("implicit_filter.b", lin2.bias)]
        red = D.OverlappedGradReducer([q for _, q in named], named=named)
        for step in range(2):
            for _, q in named:
                q.grad = None
            xin = torch.full((2, 3), float(rank + 1 + step))
            lin2(lin1(xin)).sum().backward()
            local = [q.grad.clone() for _, q in named]
            red.finish()
            outs = [torch.zeros_like(g) for g in local]
            for g, o in zip(local, outs):
                gl = [torch.zeros_like(g) for _ in range(world)]
                dist.all_gather(gl, g)
                o.copy_(sum(gl))
            for (_, q), o in zip(named, outs):
                assert torch.allclose(q.grad, o, rtol=1e-6, atol=1e-6), "OverlappedGradReducer sum mismatch"
        red.remove()
        out.put((rank, "ok"))
    except Exception as e:   # pragma: no cover
        out.put((rank, repr(e)))
    finally:
        dist.destroy_process_group()


def test_shard_bounds_cover_batch():
    from importlib import import_module
    D = import_module("hyena_dna_b200.distributed")
    for gb in (1, 5, 8, 13):
        for w in (1, 2, 4, 8):
            spans = [D.shard_bounds(gb, w, r) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == gb
            for (a, b), (c, d) in zip(spans, spans[1:]):
                assert b == c and a <= b and c <= d


@pytest.mark.timeout(120)
def test_two_rank_gloo_allreduce_and_gather():
    ctx = mp.get_context("spawn")
    out = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, out)) for r in range(2)]
    for p in procs:
        p.start()
    res = [out.get(timeout=100) for _ in procs]
    for p in procs:
        p.join(timeout=30)
    assert sorted(res) == [(0, "ok"), (1, "ok")], res


def test_c_abi_v2_exports_every_declared_symbol():
    """The library loads on a CPU-only box, reports ABI version 2 (no hyena_b200_filter_bwd) and exports exactly what
    include/hyena_b200.h declares."""
    import re
    from importlib import import_module
    _lib = import_module("hyena_dna_b200._lib")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "hyena_b200.h")).read()
    declared = set(re.findall(r"HY_API[^;(]*?\b(hyena_b200_\w+)\s*\(", hdr))
    assert declared, "no declarations parsed"
    L = _lib.lib()
    for name in declared:
        assert hasattr(L, name), f"{name} declared in include/hyena_b200.h but not exported"
    assert declared == set(_lib.SIGNATURES), (declared ^ set(_lib.SIGNATURES))
    assert L.hyena_b200_abi_version() == 2
    assert not hasattr(L, "hyena_b200_filter_bwd"), "version 2 no longer exports the CUDA-core filter backward"
    assert L.hyena_b200_max_seqlen() == 1 << 20
    assert L.hyena_b200_spectrum_elems(1000) == 1024 and L.hyena_b200_spectrum_elems(160000) == 262144


def test_product_path_fails_loudly_without_gpu():
    import hyena_dna_b200 as H
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    op = H.HyenaOperator(8, 64, emb_dim=3)
    with pytest.raises(H.HyenaB200Error):
        op(torch.randn(1, 64, 8))
    with pytest.raises(H.HyenaB200Error):
        H.fftconv_func(torch.randn(1, 2, 64), torch.randn(2, 64), torch.randn(2), gelu=False)
    with pytest.raises(H.HyenaB200Error):
        H.HyenaOperator(8, 64, num_heads=2)
