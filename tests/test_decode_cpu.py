"""Incremental decoding without a GPU: the decode oracle against the reference's own outputs, and the argument checks of
the C ABI and of HyenaOperator.allocate_inference_cache."""
import ctypes
from functools import partial
from importlib import import_module

import pytest
import torch

from oracle import hyena_oracle as O
from tests import decode_oracle as DO
from tests.golden_util import load

_lib = import_module("hyena_dna_b200._lib")


@pytest.mark.parametrize("prompt_len", [0, 1, 2, 100])
@pytest.mark.parametrize("case", ["ref_L256_D16", "ref_L250_lmax300_D8"])
def test_oracle_decode_matches_reference(case, prompt_len):
    """Token-by-token direct sums reproduce the reference's FFT forward at every position.  fp32: the tolerance
    test_oracle_golden.py uses for du, because direct sums and FFTs round differently (both land ~2.4e-6 from the fp64
    truth on ref_L250_lmax300_D8)."""
    G = load(case)
    P = O.canonical(G["sd"])
    y = DO.hyena_operator_decode(G["u"], P, prompt_len)
    assert y.shape == (G["B"], G["L"], G["D"])
    torch.testing.assert_close(y, G["y"], rtol=1e-5, atol=1e-6)
    y64 = DO.hyena_operator_decode(G["u"].double(), O.to_dtype(P, torch.float64), prompt_len)
    torch.testing.assert_close(y64, G["y64"], rtol=1e-10, atol=1e-12)
    tail = DO.hyena_operator_decode(G["u"].double(), O.to_dtype(P, torch.float64), prompt_len, prompt_outputs=False)
    assert torch.equal(tail, y64[:, prompt_len:])


def _err():
    return _lib.lib().hyena_b200_last_error().decode()


def _step(L, ptrs, B=2, D=8, t=5, max_len=64, ws_bytes=1 << 20):
    return L.hyena_b200_decode_step(*ptrs, B, D, t, max_len, ptrs[0], ws_bytes, None)


def test_decode_abi_rejects_bad_arguments():
    L = _lib.lib()
    one = ctypes.c_void_p(256)        # never dereferenced: every call below fails its checks first
    ok = [one] * 12
    assert _step(L, [None] * 12) != 0 and "null pointer" in _err()
    for i in (0, 1, 3, 4, 5, 6, 7, 9, 10, 11):            # every required pointer (in_bias and out_bias may be NULL)
        ptrs = list(ok)
        ptrs[i] = None
        assert _step(L, ptrs) != 0 and "null pointer" in _err(), i
    assert _step(L, ok, t=64, max_len=64) != 0 and "position t = 64" in _err()
    assert _step(L, ok, t=-1) != 0 and "position t = -1" in _err()
    assert _step(L, ok, max_len=(1 << 20) + 1, t=0) != 0 and "exceeds the supported maximum" in _err()
    assert _step(L, ok, B=65) != 0 and "decode batch" in _err()
    assert _step(L, ok, ws_bytes=16) != 0 and "workspace too small" in _err()
    assert L.hyena_b200_decode_prefill(*([None] * 6), 2, 8, 10, 64, None) != 0 and "null pointer" in _err()
    assert L.hyena_b200_decode_prefill(*([one] * 6), 2, 8, 65, 64, None) != 0 and "prompt length" in _err()
    assert L.hyena_b200_decode_prefill(*([one] * 6), 2, 8, 4, (1 << 20) + 4, None) != 0 and "exceeds" in _err()
    # the partial sums of every history chunk plus x0 and y_pre, (B, D) each
    assert L.hyena_b200_decode_workspace_bytes(1, 256, 1 << 20) == (128 + 2) * 256 * 4
    assert L.hyena_b200_decode_workspace_bytes(3, 16, 1) == 3 * 3 * 16 * 4


def test_allocate_inference_cache_rejects_unsupported_operators():
    import hyena_dna_b200 as H
    with pytest.raises(H.HyenaB200Error, match="order"):
        H.HyenaOperator(8, 64, order=3, emb_dim=3).allocate_inference_cache(1, 32)
    with pytest.raises(H.HyenaB200Error, match="bidirectional"):
        H.HyenaOperator(8, 64, emb_dim=3, bidirectional=True).allocate_inference_cache(1, 32)
    op = H.HyenaOperator(8, 64, emb_dim=3)
    with pytest.raises(H.HyenaB200Error, match="max_seqlen 65"):
        op.allocate_inference_cache(1, 65)
    with pytest.raises(H.HyenaB200Error, match="max_seqlen 0"):
        op.allocate_inference_cache(1, 0)
    with pytest.raises(H.HyenaB200Error, match="CUDA"):          # a CPU module: no fallback
        op.allocate_inference_cache(1, 64)


def test_block_step_needs_a_mixer_with_step():
    import hyena_dna_b200 as H

    class Plain(torch.nn.Module):
        def __init__(self, dim):
            super().__init__()

        def forward(self, x):
            return x

    blk = H.Block(8, mixer_cls=Plain)
    with pytest.raises(H.HyenaB200Error, match="no incremental decoding"):
        blk.step(torch.zeros(1, 1, 8), None, None)
    with pytest.raises(H.HyenaB200Error, match="no incremental decoding"):
        blk.prefill(torch.zeros(1, 4, 8), None, None)
    m = H.Backbone(8, 2, partial(H.HyenaOperator, l_max=64, emb_dim=3))
    with pytest.raises(H.HyenaB200Error, match="CUDA"):
        m.allocate_inference_cache(1, 64)
