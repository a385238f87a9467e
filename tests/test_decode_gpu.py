"""Incremental decoding on the GPU: prefill + per-token steps against the full-sequence forward and the fp64 oracle
(tests/decode_oracle.py:hyena_operator_decode).  Tolerance policy: tests/parity_util.py."""
from functools import partial

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import hyena_oracle as O
from tests import decode_oracle as DO
from tests import parity_util as PU

pytestmark = pytest.mark.gpu


def _dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    torch.backends.cuda.matmul.allow_tf32 = False
    return torch.device("cuda:0")


def _operator(D, l_max, seed, **kw):
    """HyenaOperator with seeded unit-scale parameters, and the oracle's parameter dict for it."""
    import hyena_dna_b200 as H
    P = O.init_params(D, l_max, emb_dim=5, w=10.0, generator=torch.Generator().manual_seed(seed))
    sd = dict(P)
    for extra in ("filter_fn.implicit_filter.3.freq", "filter_fn.implicit_filter.5.freq"):
        sd[extra] = sd["filter_fn.implicit_filter.1.freq"]
    op = H.HyenaOperator(D, l_max, emb_dim=5, w=10.0, lr_pos_emb=0.0, **kw)
    op.load_state_dict(sd)
    if not op.filter_fn.use_bias:
        P["filter_fn.bias"] = torch.zeros_like(P["filter_fn.bias"])
    return op.to(_dev()), P


def _decode(op, u, prompt_len):
    """Prefill u[:, :prompt_len] (skipped for 0), then step through the rest one token at a time: (prefill out, steps)."""
    B, L, _ = u.shape
    cache = op.allocate_inference_cache(B, L)
    y0 = op.prefill(u[:, :prompt_len], cache) if prompt_len else None
    steps = [op.step(u[:, t:t + 1], cache) for t in range(prompt_len, L)]
    assert cache.seqlen_offset == L
    return y0, torch.cat(steps, dim=1)


def _inputs(B, L, D, seed):
    return torch.randn(B, L, D, generator=torch.Generator().manual_seed(seed))


@pytest.mark.parametrize("prompt_len", [0, 1, 2, 777])
@pytest.mark.parametrize("B", [1, 3])
@pytest.mark.parametrize("D", [16, 256])
def test_teacher_forced_decode_equals_full_sequence(D, B, prompt_len):
    dev = _dev()
    L = prompt_len + 128
    op, P = _operator(D, 1024, seed=D + B)
    u = _inputs(B, L, D, seed=prompt_len)
    with torch.no_grad():
        y_full = op(u.to(dev))
        y_prompt = op(u[:, :prompt_len].to(dev)) if prompt_len else None
    y0, ys = _decode(op, u.to(dev), prompt_len)
    if prompt_len:
        assert torch.equal(y0, y_prompt)
    y64 = DO.hyena_operator_decode(u.to(dev).double(), O.to_dtype({k: v.to(dev) for k, v in P.items()}, torch.float64),
                                   prompt_len, prompt_outputs=False)
    what = f"decode D={D} B={B} Lp={prompt_len}"
    PU.check(ys, y_full[:, prompt_len:], what + " vs forward", ref64=y64)
    PU.check(ys, y64, what + " vs fp64 oracle")


@pytest.mark.parametrize("B", [3, 11])
def test_decode_over_many_history_chunks(B):
    """t > 8192: the step's history is split over several CTAs per channel; B = 11 also takes two batch groups."""
    dev = _dev()
    D, prompt_len, L = 16, 20000, 20016
    op, P = _operator(D, L, seed=7)
    u = _inputs(B, L, D, seed=B)
    with torch.no_grad():
        y_full = op(u.to(dev))
    _, ys = _decode(op, u.to(dev), prompt_len)
    y64 = DO.hyena_operator_decode(u.to(dev).double(), O.to_dtype({k: v.to(dev) for k, v in P.items()}, torch.float64),
                                   prompt_len, prompt_outputs=False)
    PU.check(ys, y_full[:, prompt_len:], f"decode chunks B={B} vs forward", ref64=y64)
    PU.check(ys, y64, f"decode chunks B={B} vs fp64 oracle")


def test_prefill_is_forward_and_cached_filter_is_a_prefix():
    dev = _dev()
    D, B, Lp, max_len = 256, 2, 777, 2048
    op, _ = _operator(D, 4096, seed=3)
    u = _inputs(B, Lp, D, seed=11).to(dev)
    cache = op.allocate_inference_cache(B, max_len)
    y = op.prefill(u, cache)
    assert torch.equal(y, op(u))                       # with autograd recording
    with torch.no_grad():
        assert torch.equal(y, op(u))
        assert torch.equal(op.filter_fn.filter_channel_major(Lp), cache.k[:, :Lp])
    assert cache.seqlen_offset == Lp and cache.k.shape == (D, max_len)


def test_long_context_decode():
    """B = 1, D = 256: a 2^20 - 8 token prompt, then the last 8 positions one at a time."""
    dev = _dev()
    D, L, n = 256, 1 << 20, 8
    op, P = _operator(D, L, seed=5)
    u = O.nucleotide_activations(1, L, D, seed=9)[0].to(dev)
    with torch.no_grad():
        y_full = op(u)[:, L - n:].clone()
    _, ys = _decode(op, u, L - n)
    del op
    torch.cuda.empty_cache()
    y64 = DO.hyena_operator_decode(u.double(), O.to_dtype({k: v.to(dev) for k, v in P.items()}, torch.float64), L - n,
                                   prompt_outputs=False)
    rec = PU.check(ys, y_full, "decode 2^20 vs forward", ref64=y64)
    # |y| reaches ~1.6e3 here: judged against the fp64 oracle, the step is as close as the FFT forward or closer
    assert rec["e_ours64"] <= 2.0 * rec["e_ref64"], rec


class _Mlp(nn.Module):
    def __init__(self, dim, hidden_features):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden_features)
        self.fc2 = nn.Linear(hidden_features, dim)

    def forward(self, x):
        return self.fc2(F.gelu(self.fc1(x), approximate="tanh"))


def test_backbone_decode_equals_forward():
    import hyena_dna_b200 as H
    dev = _dev()
    D, B, Lp, L = 32, 2, 100, 164
    torch.manual_seed(0)
    mixer = partial(H.HyenaOperator, l_max=256, emb_dim=5, w=10.0, lr_pos_emb=0.0)
    m = H.Backbone(D, 2, mixer, mlp_cls=partial(_Mlp, hidden_features=2 * D), residual_in_fp32=True).to(dev)
    x = _inputs(B, L, D, seed=1).to(dev)
    with torch.no_grad():
        y_full = m(x)
        caches = m.allocate_inference_cache(B, L)
        y0 = m.prefill(x[:, :Lp], caches)
        ys = torch.cat([m.step(x[:, t:t + 1], caches) for t in range(Lp, L)], dim=1)
    PU.check(y0, y_full[:, :Lp], "backbone prefill")
    PU.check(ys, y_full[:, Lp:], "backbone decode")


def test_decode_is_deterministic():
    dev = _dev()
    D, B, Lp, L = 256, 3, 9000, 9040
    op, _ = _operator(D, L, seed=13)
    u = _inputs(B, L, D, seed=2).to(dev)
    a = _decode(op, u, Lp)
    b = _decode(op, u, Lp)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.parametrize("kw", [dict(normalized=True), dict(bias=False)], ids=["normalized", "no_filter_bias"])
def test_decode_filter_options(kw):
    dev = _dev()
    D, B, Lp, L = 16, 2, 300, 364
    op, P = _operator(D, 512, seed=21, **kw)
    u = _inputs(B, L, D, seed=4).to(dev)
    with torch.no_grad():
        y_full = op(u)
    _, ys = _decode(op, u, Lp)
    y64 = DO.hyena_operator_decode(u.double(), O.to_dtype({k: v.to(dev) for k, v in P.items()}, torch.float64), Lp,
                                   normalized=kw.get("normalized", False), prompt_outputs=False)
    PU.check(ys, y_full[:, Lp:], f"decode {kw} vs forward", ref64=y64)
    PU.check(ys, y64, f"decode {kw} vs fp64 oracle")


def test_step_keeps_dtype_and_stops_when_full():
    import hyena_dna_b200 as H
    dev = _dev()
    op, _ = _operator(16, 64, seed=1)
    cache = op.allocate_inference_cache(2, 4)
    u = _inputs(2, 4, 16, seed=0).to(dev)
    y = op.step(u[:, :1].double(), cache)
    assert y.dtype == torch.float64 and y.shape == (2, 1, 16)
    for t in range(1, 4):
        op.step(u[:, t:t + 1], cache)
    with pytest.raises(H.HyenaB200Error, match="full"):
        op.step(u[:, :1], cache)
    with pytest.raises(H.HyenaB200Error, match="batch"):
        op.step(u[:1, :1], op.allocate_inference_cache(2, 4))
