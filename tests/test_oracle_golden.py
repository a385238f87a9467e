"""Pin the oracle (oracle/hyena_oracle.py) against outputs of the reference code itself."""
import pytest
import torch

from oracle import hyena_oracle as O
from tests.golden_util import CASES, CASES_OPTIONS, CASES_ORDER3, load, stored


@pytest.mark.parametrize("case", CASES + CASES_ORDER3)
def test_oracle_forward_backward_matches_reference(case):
    G = load(case)
    P = O.canonical(G["sd"])
    y, du, grads = O.operator_fwd_bwd(G["u"], P, G["dy"])
    assert y.shape == (G["B"], G["L"], G["D"])
    torch.testing.assert_close(stored(G, y), G["y"], rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(stored(G, du), G["du"], rtol=1e-5, atol=1e-6)
    for k, g in G["grad"].items():
        kk = "filter_fn.implicit_filter.1.freq" if k.endswith(".freq") else k
        scale = float(g.abs().max()) + 1e-30
        assert float((grads[kk] - g).abs().max()) <= 2e-5 * scale + 1e-7, k


@pytest.mark.parametrize("case", ["ref_L64_D8", "ref_L256_D16", "ref_L250_lmax300_D8"] + CASES_ORDER3)
def test_oracle_fp64_matches_reference_fp64(case):
    G = load(case)
    P = O.to_dtype(O.canonical(G["sd"]), torch.float64)
    y, du, _ = O.operator_fwd_bwd(G["u"].double(), P, G["dy"].double())
    torch.testing.assert_close(y, G["y64"], rtol=1e-10, atol=1e-12)
    torch.testing.assert_close(du, G["du64"], rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("case", CASES_OPTIONS)
def test_oracle_filter_options_match_reference(case):
    """normalized=True, modulation_lr != 0 (deltas gradient), shift != 0: fixture from the unmodified src module."""
    G = load(case)
    P = O.canonical(G["sd"])
    names = [k for k in P if k not in ("filter_fn.pos_emb.z", "filter_fn.pos_emb.t")]
    y, du, grads = O.operator_fwd_bwd(G["u"], P, G["dy"], shift=G["extra"]["shift"], grads_for=names,
                                      normalized=G["extra"]["normalized"])
    torch.testing.assert_close(y, G["y"], rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(du, G["du"], rtol=1e-5, atol=1e-6)
    assert "filter_fn.modulation.deltas" in G["grad"]
    for k, g in G["grad"].items():
        kk = "filter_fn.implicit_filter.1.freq" if k.endswith(".freq") else k
        scale = float(g.abs().max()) + 1e-30
        assert float((grads[kk] - g).abs().max()) <= 2e-5 * scale + 1e-7, k


def test_positional_embedding_and_deltas_match_reference_buffers():
    G = load("ref_L256_D16")
    z, t = O.positional_embedding(G["E"], G["l_max"])
    assert torch.equal(z, G["sd"]["filter_fn.pos_emb.z"])
    assert torch.equal(t, G["sd"]["filter_fn.pos_emb.t"])
    assert torch.equal(O.modulation_deltas(G["D"]), G["sd"]["filter_fn.modulation.deltas"])


def test_state_dict_keys_are_the_reference_keys():
    G = load("ref_L64_D8")
    P = O.init_params(G["D"], G["l_max"], emb_dim=G["E"])
    ref_keys = set(O.canonical(G["sd"]).keys())
    assert set(P.keys()) == ref_keys
    for k in ref_keys:
        assert tuple(P[k].shape) == tuple(G["sd"][k].shape), k


def test_fftconv_equals_direct_causal_convolution():
    g = torch.Generator().manual_seed(5)
    u = torch.randn(2, 3, 40, generator=g, dtype=torch.float64)
    k = torch.randn(3, 40, generator=g, dtype=torch.float64)
    D = torch.randn(3, generator=g, dtype=torch.float64)
    torch.testing.assert_close(O.fftconv_ref(u, k, D), O.fftconv_direct(u, k, D), rtol=1e-10, atol=1e-10)


def test_causality():
    G = load("ref_L64_D8")
    P = O.canonical(G["sd"])
    u = G["u"].clone()
    y0 = O.hyena_operator(u, P)
    u2 = u.clone(); u2[:, 40:] += 1.0
    y1 = O.hyena_operator(u2, P)
    torch.testing.assert_close(y0[:, :40], y1[:, :40], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("case", ["block_L128_D32_mlp", "block_L96_D16_nomlp"])
def test_oracle_prenorm_backbone_matches_reference_block(case):
    """Block glue (S8 f1): the oracle's restatement against fixtures from the unmodified flash_attn Block + HyenaOperator + Mlp
    (tests/golden/make_golden_block.py), forward, input gradient and every parameter gradient, fp32 and fp64."""
    import os
    import numpy as np
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", case + ".npz"))
    for dt, tag, tol in ((torch.float32, "", 3e-5), (torch.float64, "64", 1e-9)):
        sd = {k[3:]: torch.from_numpy(z[k]).to(dt) for k in z.files if k.startswith("sd/")}
        want = [k[5:] for k in z.files if k.startswith("grad/")]
        for k in want:
            sd[k].requires_grad_(True)
        x = torch.from_numpy(z["x"]).to(dt).requires_grad_(True)
        y = O.prenorm_backbone(x, sd, 2)
        y.backward(torch.from_numpy(z["dy"]).to(dt))
        assert float((y.detach() - torch.from_numpy(z["y" + tag])).abs().max()) <= tol * max(1.0, float(np.abs(z["y" + tag]).max()))
        assert float((x.grad - torch.from_numpy(z["dx" + tag])).abs().max()) <= tol * max(1.0, float(np.abs(z["dx" + tag]).max()))
        for k in want:                          # named_parameters() of the reference lists the shared freq tensor once (.1.freq)
            ref = torch.from_numpy(z[("grad64/" if tag else "grad/") + k])
            assert sd[k].grad is not None, k
            assert float((sd[k].grad - ref).abs().max()) <= 10 * tol * max(1.0, float(ref.abs().max())), k
