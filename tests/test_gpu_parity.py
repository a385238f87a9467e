"""GPU parity tests: the sm_100a path (through the C ABI) against the CPU oracle and the committed
reference-generated golden vectors.  Tolerance from BASELINE.json north_star: 1e-3 rel / 1e-5 abs
in fp32 (applied elementwise, with the abs term scaled by the tensor's magnitude where outputs are
far from unit scale -- see SURVEY.md S8(c) for why)."""
import math

import pytest
import torch

from oracle import hyena_oracle as O
from tests import parity_util as PU
from tests.golden_util import CASES, CASES_OPTIONS, load, stored

pytestmark = pytest.mark.gpu

RTOL, ATOL = 1e-3, 1e-5


def _dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return torch.device("cuda:0")


def _close(got, ref, what, scale_abs=True, ref64=None):
    """All comparisons go through tests/parity_util.check (north_star tolerance 1e-3 rel / 1e-5 abs, S8(c) hatch, book-keeping
    printed at the end of the run).  Parameter gradients ("grad" in `what`): absolute term 1e-5 * max(1, max|ref|) (sums over up to
    2^20 positions).  scale_abs (activations compared against a reference whose fp32 twin was not run at this size): the same
    scaling of the absolute term, stated in the record's name."""
    if any(tag in what for tag in ("grad", " dW", " dD", " db")):
        return PU.check(got, ref, what, ref64=ref64, param_grad=True)
    if scale_abs:
        s = max(1.0, float(ref.detach().abs().max()))
        return PU.check(got, ref, what + (f" [abs term x{s:.3g}]" if s > 1.0 else ""), ref64=ref64, atol=ATOL * s)
    return PU.check(got, ref, what, ref64=ref64)


def _module_from_sd(sd, D, l_max, E, w, dev, **kw):
    import hyena_dna_b200 as H
    op = H.HyenaOperator(D, l_max, order=2, filter_order=64, emb_dim=E, w=w, lr_pos_emb=kw.pop("lr_pos_emb", 0.0),
                         layer_idx=0, device=None, dtype=None, **kw)
    missing, unexpected = op.load_state_dict(sd, strict=True)
    return op.to(dev)


# ------------------------------------------------------------------------------------------ library
def test_library_loads_and_counts_launches():
    import hyena_dna_b200 as H
    dev = _dev()
    n0 = H.launch_count()
    k = torch.randn(4, 256, device=dev)
    H.ops.filter_spectrum(k)
    torch.cuda.synchronize()
    assert H.launch_count() > n0


# ------------------------------------------------------------------------------------------ plain fftconv
@pytest.mark.parametrize("L", [16, 250, 1001, 1024, 2048, 3000, 4096, 8192, 16384, 32768, 65536, 100000, 160000,
                               262144, 524288, 1048576])
def test_fftconv_func_forward_backward(L):
    import hyena_dna_b200 as H
    dev = _dev()
    B, Hc = (2, 3) if L <= 262144 else (1, 2)
    g = torch.Generator().manual_seed(L)
    u = torch.randn(B, Hc, L, generator=g)
    # decaying filter with unit-ish gain so outputs stay near unit scale (like a trained Hyena filter)
    k = torch.randn(Hc, L, generator=g) * torch.exp(-torch.arange(L) / (0.05 * L + 1))[None] / math.sqrt(0.05 * L + 1)
    Dv = torch.randn(Hc, generator=g)
    dout = torch.randn(B, Hc, L, generator=g)
    ur, kr, Dr = (x.double().clone().requires_grad_(True) for x in (u, k, Dv))
    ref = O.fftconv_ref(ur, kr, Dr)
    ref.backward(dout.double())
    ug, kg, Dg = (x.to(dev).requires_grad_(True) for x in (u, k, Dv))
    out = H.fftconv_func(ug, kg, Dg, gelu=False)
    out.backward(dout.to(dev))
    _close(out, ref, f"fftconv out L={L}")
    _close(ug.grad, ur.grad, f"fftconv du L={L}")
    _close(kg.grad, kr.grad, f"fftconv dk L={L}")
    _close(Dg.grad, Dr.grad, f"fftconv dD L={L}")


def test_fftconv_impulse_and_linearity_full_length():
    """Size-independent properties at L = 2^20: an impulse returns the filter; the op is linear in u."""
    import hyena_dna_b200 as H
    dev = _dev()
    L, Hc = 1 << 20, 4
    g = torch.Generator().manual_seed(7)
    k = (torch.randn(Hc, L, generator=g) * torch.exp(-torch.arange(L) / 50000.0)[None]).to(dev)
    Dv = torch.zeros(Hc, device=dev)
    u = torch.zeros(1, Hc, L, device=dev)
    shift = 12345
    u[:, :, shift] = 1.0
    out = H.fftconv_func(u, k, Dv, gelu=False)
    expect = torch.zeros_like(out)
    expect[0, :, shift:] = k[:, : L - shift]
    _close(out, expect, "impulse response")
    assert float(out[0, :, :shift].abs().max()) < 1e-4          # causal: nothing before the impulse
    a = torch.randn(1, Hc, L, generator=g).to(dev)
    b = torch.randn(1, Hc, L, generator=g).to(dev)
    lhs = H.fftconv_func(2.0 * a - 3.0 * b, k, Dv, gelu=False)
    rhs = 2.0 * H.fftconv_func(a, k, Dv, gelu=False) - 3.0 * H.fftconv_func(b, k, Dv, gelu=False)
    _close(lhs, rhs, "linearity")


def test_fftconv_rejects_unsupported_and_cpu():
    import hyena_dna_b200 as H
    dev = _dev()
    u = torch.randn(1, 2, 64, device=dev); k = torch.randn(2, 64, device=dev); D = torch.randn(2, device=dev)
    with pytest.raises(H.HyenaB200Error):
        H.fftconv_func(u, k, D, gelu=True)
    with pytest.raises(H.HyenaB200Error):
        H.fftconv_func(u.cpu(), k.cpu(), D.cpu(), gelu=False)
    with pytest.raises(H.HyenaB200Error):
        H.ops.fftconv_forward(torch.randn(1, 1, (1 << 20) + 2, device=dev), torch.empty(1, 1 << 21, dtype=torch.complex64, device=dev),
                              torch.zeros(1, device=dev))


# ------------------------------------------------------------------------------------------ filter
@pytest.mark.parametrize("case", CASES)
def test_filter_matches_oracle(case):
    import hyena_dna_b200 as H
    dev = _dev()
    G = load(case)
    P = O.canonical(G["sd"])
    L = G["L"]
    ref = O.hyena_filter(L, O.to_dtype(P, torch.float64))[0].transpose(0, 1)
    op = _module_from_sd(G["sd"], G["D"], G["l_max"], G["E"], G["w"], dev)
    k = op.filter_fn.filter_channel_major(L)
    _close(k, ref, f"filter {case}", scale_abs=False)
    k3 = op.filter_fn.filter(L)
    assert tuple(k3.shape) == (1, L, G["D"])


def test_filter_backward_matches_oracle_including_z():
    import hyena_dna_b200 as H
    dev = _dev()
    D, L, E = 24, 333, 5
    g = torch.Generator().manual_seed(3)
    P = O.init_params(D, L, emb_dim=E, w=10.0, generator=g)
    dk = torch.randn(D, L, generator=g)
    names = [k for k in P if "implicit_filter" in k] + ["filter_fn.pos_emb.z"]
    Q = {k: v.double().clone().requires_grad_(k in names) for k, v in P.items()}
    kref = O.hyena_filter(L, Q)[0].transpose(0, 1)
    kref.backward(dk.double())
    f = H.HyenaFilter(D, emb_dim=E, order=64, seq_len=L, w=10.0, lr_pos_emb=1e-5).to(dev)
    sd = {k[len("filter_fn."):]: v for k, v in P.items() if k.startswith("filter_fn.")}
    for extra in ("implicit_filter.3.freq", "implicit_filter.5.freq"):
        sd[extra] = sd["implicit_filter.1.freq"]
    f.load_state_dict(sd)
    k = f.filter_channel_major(L)
    k.backward(dk.to(dev))
    _close(k, kref, "filter fwd", scale_abs=False)
    got = dict(f.named_parameters())
    for name in names:
        short = name[len("filter_fn."):]
        _close(got[short].grad, Q[name].grad, f"grad {short}")


# ------------------------------------------------------------------------------------------ operator
@pytest.mark.parametrize("case", CASES)
def test_operator_matches_reference_golden(case):
    dev = _dev()
    G = load(case)
    op = _module_from_sd(G["sd"], G["D"], G["l_max"], G["E"], G["w"], dev)
    u = G["u"].to(dev).requires_grad_(True)
    y = op(u)
    y.backward(G["dy"].to(dev))
    _close(stored(G, y), G["y"], f"{case} y", scale_abs=False, ref64=G.get("y64"))
    _close(stored(G, u.grad), G["du"], f"{case} du", scale_abs=False, ref64=G.get("du64"))
    got = dict(op.named_parameters())
    for name, gref in G["grad"].items():
        _close(got[name].grad, gref, f"{case} grad {name}", ref64=G["grad64"].get(name))


@pytest.mark.parametrize("case", CASES_OPTIONS)
def test_operator_filter_options_match_reference_golden(case):
    """normalized=True (hyena.py:235-236) and trainable modulation deltas (modulation_lr != 0, hyena.py:145-150), non-zero
    shift: fixture from the unmodified src module (tests/golden/make_golden.py); the deltas gradient is checked too."""
    dev = _dev()
    G = load(case)
    op = _module_from_sd(G["sd"], G["D"], G["l_max"], G["E"], G["w"], dev, **G["extra"])
    assert isinstance(op.filter_fn.modulation.deltas, torch.nn.Parameter)
    assert op.filter_fn.modulation.deltas._optim["lr"] == G["extra"]["modulation_lr"]
    u = G["u"].to(dev).requires_grad_(True)
    y = op(u)
    y.backward(G["dy"].to(dev))
    PU.check(y, G["y"], f"{case} y", ref64=G["y64"])
    PU.check(u.grad, G["du"], f"{case} du", ref64=G["du64"])
    got = dict(op.named_parameters())
    assert "filter_fn.modulation.deltas" in G["grad"]
    for name, gref in G["grad"].items():
        PU.check(got[name].grad, gref, f"{case} grad {name}", ref64=G["grad64"][name], param_grad=True)


@pytest.mark.parametrize("B,L,D,l_max", [(2, 1001, 8, 1001), (1, 5000, 16, 8192), (2, 32768, 16, 32768),
                                         (1, 160000, 8, 160000)])
def test_operator_matches_oracle_fp64(B, L, D, l_max):
    dev = _dev()
    g = torch.Generator().manual_seed(B * 1000 + D)
    P = O.init_params(D, l_max, emb_dim=5, w=10.0, generator=g, init_std=0.02)
    u, _ = O.nucleotide_activations(B, L, D, seed=2222)
    dy = torch.randn(B, L, D, generator=torch.Generator().manual_seed(1))
    y64, du64, g64 = O.operator_fwd_bwd(u.double(), O.to_dtype(P, torch.float64), dy.double())
    sd = dict(P)
    for extra in ("filter_fn.implicit_filter.3.freq", "filter_fn.implicit_filter.5.freq"):
        sd[extra] = sd["filter_fn.implicit_filter.1.freq"]
    op = _module_from_sd(sd, D, l_max, 5, 10.0, dev)
    ug = u.to(dev).requires_grad_(True)
    y = op(ug)
    y.backward(dy.to(dev))
    _close(y, y64, "y")
    _close(ug.grad, du64, "du")
    got = dict(op.named_parameters())
    for name, gref in g64.items():
        _close(got[name].grad, gref, f"grad {name}")


def test_operator_large_1m_sampled_channels():
    """large-1m shape on the sequence axis (L = 2^20) with a narrow model so the fp64 oracle stays fast."""
    dev = _dev()
    B, L, D = 1, 1 << 20, 8
    g = torch.Generator().manual_seed(11)
    P = O.init_params(D, L, emb_dim=5, w=10.0, generator=g, init_std=0.02)
    u, _ = O.nucleotide_activations(B, L, D, seed=2222)
    dy = torch.randn(B, L, D, generator=torch.Generator().manual_seed(1))
    y64, du64, g64 = O.operator_fwd_bwd(u.double(), O.to_dtype(P, torch.float64), dy.double())
    sd = dict(P)
    for extra in ("filter_fn.implicit_filter.3.freq", "filter_fn.implicit_filter.5.freq"):
        sd[extra] = sd["filter_fn.implicit_filter.1.freq"]
    op = _module_from_sd(sd, D, L, 5, 10.0, dev)
    ug = u.to(dev).requires_grad_(True)
    y = op(ug)
    y.backward(dy.to(dev))
    _close(y, y64, "y 1m")
    _close(ug.grad, du64, "du 1m")
    got = dict(op.named_parameters())
    for name in ("filter_fn.bias", "short_filter.weight", "filter_fn.implicit_filter.6.weight", "in_proj.bias"):
        _close(got[name].grad, g64[name], f"grad {name} 1m")


def test_operator_full_width_large_1m_runs_and_is_causal():
    """BASELINE.json configs[3] (L=1,048,576, d_model=256, batch=1): finite outputs + causality property."""
    dev = _dev()
    import hyena_dna_b200 as H
    torch.manual_seed(0)
    L, D = 1 << 20, 256
    op = H.HyenaOperator(D, L, emb_dim=5, w=10, lr_pos_emb=0.0).to(dev)
    u, _ = O.nucleotide_activations(1, L, D)
    u = u.to(dev)
    with torch.no_grad():
        y0 = op(u)
        u2 = u.clone()
        cut = 700_001
        u2[:, cut:] += 1.0
        y1 = op(u2)
    assert torch.isfinite(y0).all()
    scale = float(y0.abs().max())
    assert float((y0[:, :cut] - y1[:, :cut]).abs().max()) <= 2e-4 * max(scale, 1.0)
    assert float((y0[:, cut:] - y1[:, cut:]).abs().max()) > 1e-3 * scale
    u.requires_grad_(True)
    y = op(u)
    y.square().mean().backward()
    assert torch.isfinite(u.grad).all()
    for n, p in op.named_parameters():
        assert p.grad is not None and torch.isfinite(p.grad).all(), n


def test_state_dict_roundtrip_and_optim_attrs():
    import hyena_dna_b200 as H
    G = load("ref_L64_D8")
    op = H.HyenaOperator(G["D"], G["l_max"], emb_dim=G["E"], w=G["w"], lr=6e-4, lr_pos_emb=0.0)
    assert set(op.state_dict().keys()) == set(G["sd"].keys())
    for k, v in op.state_dict().items():
        assert tuple(v.shape) == tuple(G["sd"][k].shape), k
    assert op.filter_fn.implicit_filter[0].weight._optim == {"weight_decay": 0, "lr": 6e-4}
    assert H.registry.layer["hyena"] is H.HyenaOperator


# ------------------------------------------------------------------------------------------ projections
def test_projection_gemms_match_fp64():
    """in/out projections through csrc/gemm.cu (cuBLASLt BF16x9 fp32 emulation) vs float64 matmuls."""
    import hyena_dna_b200 as H
    from importlib import import_module
    hy = import_module("hyena_dna_b200.hyena")
    dev = _dev()
    g = torch.Generator().manual_seed(9)
    B, L, D = 2, 4096, 64
    u = torch.randn(B, L, D, generator=g).to(dev).requires_grad_(True)
    W = (torch.randn(3 * D, D, generator=g) * 0.05).to(dev).requires_grad_(True)
    p = hy._InProj.apply(u, W)
    ref = torch.matmul(W.double(), u.double().transpose(1, 2))
    _close(p, ref, f"in_proj ({H.ops.proj_mode()})")
    dp = torch.randn(B, 3 * D, L, generator=g).to(dev)
    p.backward(dp)
    _close(u.grad, torch.matmul(dp.double().transpose(1, 2), W.double()), "in_proj du")
    _close(W.grad, torch.matmul(dp.double(), u.double()).sum(0), "in_proj dW")
    yp = torch.randn(B, D, L, generator=g).to(dev).requires_grad_(True)
    Wo = (torch.randn(D, D, generator=g) * 0.05).to(dev).requires_grad_(True)
    bo = torch.randn(D, generator=g).to(dev).requires_grad_(True)
    y = hy._OutProj.apply(yp, Wo, bo)
    _close(y, torch.matmul(yp.double().transpose(1, 2), Wo.double().t()) + bo.double(), "out_proj")
    dy = torch.randn(B, L, D, generator=g).to(dev)
    y.backward(dy)
    _close(yp.grad, torch.matmul(Wo.double().t(), dy.double().transpose(1, 2)), "out_proj dy_pre")
    _close(Wo.grad, torch.matmul(dy.double().transpose(1, 2), yp.double().transpose(1, 2)).sum(0), "out_proj dW")
    _close(bo.grad, dy.double().sum((0, 1)), "out_proj db")


# ------------------------------------------------------------------------------------------ host-buffer entry point
@pytest.mark.parametrize("B,L,D", [(1, 8192, 32), (2, 5000, 16)])
def test_host_step_matches_autograd(B, L, D):
    """HostStep (pinned host buffers, pipelined copies) == module forward + autograd backward."""
    import hyena_dna_b200 as H
    dev = _dev()
    if H.ops.proj_mode() != "tc" and H.ops.gemm_mode() != "bf16x9":
        pytest.skip("needs the tcgen05 or the cuBLASLt 12.9 projection path")
    torch.manual_seed(5)
    op = H.HyenaOperator(D, L, emb_dim=5, w=10.0, lr_pos_emb=0.0).to(dev)
    u = torch.randn(B, L, D); dy = torch.randn(B, L, D)
    ug = u.to(dev).requires_grad_(True)
    y = op(ug)
    y.backward(dy.to(dev))
    params = [p for p in op.parameters() if p.requires_grad]
    hs = H.HostStep(op, B, L, chunks=3)
    uh, dyh = u.pin_memory(), dy.pin_memory()
    yh, duh = torch.empty(B, L, D).pin_memory(), torch.empty(B, L, D).pin_memory()
    gh = [torch.empty(p.shape).pin_memory() for p in params]
    for _ in range(2):                       # twice: buffers and events are reusable
        hs.step(uh, dyh, yh, duh, gh)
    torch.cuda.synchronize()
    _close(yh, y, "host y")
    _close(duh, ug.grad, "host du")
    for g, p in zip(gh, params):
        _close(g, p.grad, "host grad")


# ------------------------------------------------------------------------------------------ BASELINE.json configs
@pytest.mark.parametrize("name,B,L,D", [("small-32k", 8, 32768, 256), ("medium-160k", 4, 160000, 256)])
def test_baseline_configs_full_size_against_fp32_oracle(name, B, L, D):
    """BASELINE.json configs[1] and [2] at full size, fwd+bwd, against the oracle run in fp32 on the host (the
    reference's own path) -- judged with the north_star tolerance, normwise where cancellation dominates."""
    dev = _dev()
    torch.set_num_threads(min(16, torch.get_num_threads()))
    g = torch.Generator().manual_seed(42)
    P = O.init_params(D, L, emb_dim=5, w=10.0, generator=g, init_std=0.02)
    u, _ = O.nucleotide_activations(B, L, D, seed=2222)
    dy = torch.randn(B, L, D, generator=torch.Generator().manual_seed(1))
    y_ref, du_ref, g_ref = O.operator_fwd_bwd(u, P, dy)
    sd = dict(P)
    for extra in ("filter_fn.implicit_filter.3.freq", "filter_fn.implicit_filter.5.freq"):
        sd[extra] = sd["filter_fn.implicit_filter.1.freq"]
    op = _module_from_sd(sd, D, L, 5, 10.0, dev)
    ug = u.to(dev).requires_grad_(True)
    y = op(ug)
    y.backward(dy.to(dev))
    _close(y, y_ref, f"{name} y")
    _close(ug.grad, du_ref, f"{name} du")
    got = dict(op.named_parameters())
    for n in ("filter_fn.bias", "short_filter.weight", "short_filter.bias", "in_proj.weight", "out_proj.weight",
              "filter_fn.implicit_filter.6.weight", "filter_fn.implicit_filter.0.weight"):
        _close(got[n].grad, g_ref[n], f"{name} grad {n}")


def test_hyena_filter_forward_layouts():
    """HyenaFilter.forward on (B,D,L) and on the reference operator's 5-D (b,h,v,z,l) layout (hyena.py:396-423)."""
    import hyena_dna_b200 as H
    dev = _dev()
    torch.manual_seed(2)
    D, L = 12, 700
    f = H.HyenaFilter(D, emb_dim=5, order=64, seq_len=L, w=10.0, lr_pos_emb=0.0).to(dev)
    x = torch.randn(2, D, L, device=dev)
    with torch.no_grad():
        k = f.filter(L)                                     # (1, L, D) like the reference
        y3 = f(x, L)
        y3k = f(x, L, k=k, bias=f.bias)
        y5 = f(x.reshape(2, 1, D, 1, L), L, k=k[0].transpose(0, 1), bias=f.bias[None, :, None])
    ref = O.fftconv_ref(x.double().cpu(), k[0].transpose(0, 1).double().cpu(), f.bias.double().cpu())
    _close(y3, ref, "filter.forward 3-D")
    _close(y3k, ref, "filter.forward 3-D with k")
    _close(y5.reshape(2, D, L), ref, "filter.forward 5-D")


def test_wide_model_filter_paths():
    """d_model > 256 and not a multiple of 128: output-layer halves, channel chunks and the library fallback of the
    filter weight-gradient reduction."""
    import hyena_dna_b200 as H
    dev = _dev()
    D, L, E = 320, 1500, 5
    g = torch.Generator().manual_seed(8)
    P = O.init_params(D, L, emb_dim=E, w=10.0, generator=g)
    dk = torch.randn(D, L, generator=g)
    names = [k for k in P if "implicit_filter" in k]
    Q = {k: v.double().clone().requires_grad_(k in names) for k, v in P.items()}
    kref = O.hyena_filter(L, Q)[0].transpose(0, 1)
    kref.backward(dk.double())
    f = H.HyenaFilter(D, emb_dim=E, order=64, seq_len=L, w=10.0, lr_pos_emb=0.0).to(dev)
    sd = {k[len("filter_fn."):]: v for k, v in P.items() if k.startswith("filter_fn.")}
    for extra in ("implicit_filter.3.freq", "implicit_filter.5.freq"):
        sd[extra] = sd["implicit_filter.1.freq"]
    f.load_state_dict(sd)
    k = f.filter_channel_major(L)
    k.backward(dk.to(dev))
    # unit-scale init drives sin() with arguments of order 10-30: fp32 evaluation of the MLP itself is ~1e-5 from
    # the fp64 truth (the same holds for the reference in fp32), hence the wider absolute term here
    _close(k, kref, "wide filter fwd")
    got = dict(f.named_parameters())
    for name in names:
        short = name[len("filter_fn."):]
        _close(got[short].grad, Q[name].grad, f"wide grad {short}")


# ------------------------------------------------------------------------------------------ extension-level ABI
@pytest.mark.parametrize("L", [64, 250, 512, 1024, 4096, 8192, 65536])
def test_extension_abi_takes_reference_filter_convention(L):
    """fftconv_fwd / fftconv_bwd driven exactly as src/ops/fftconv.py:61-103 drives the reference extension:
    filter = rfft(k, n=fft_size) in, dfilter (H, fft_size/2+1) complex64 out (csrc/fftconv/fftconv.cpp:53-61,134-143,235)."""
    import hyena_dna_b200 as H
    from importlib import import_module
    F = import_module("hyena_dna_b200.fftconv")
    dev = _dev()
    B, Hc = 2, 3
    g = torch.Generator().manual_seed(100 + L)
    u = torch.randn(B, Hc, L, generator=g)
    k = torch.randn(Hc, L, generator=g) * torch.exp(-torch.arange(L) / (0.05 * L + 1))[None] / math.sqrt(0.05 * L + 1)
    Dv = torch.randn(Hc, generator=g)
    dout = torch.randn(B, Hc, L, generator=g)
    ur, kr, Dr = (x.double().clone().requires_grad_(True) for x in (u, k, Dv))
    ref = O.fftconv_ref(ur, kr, Dr)
    ref.backward(dout.double())
    out, du, dk, dD = O.reference_fftconv_protocol(F.fftconv_fwd, F.fftconv_bwd, u.to(dev), k.to(dev), Dv.to(dev),
                                                   dout.to(dev))
    fft_size = max(2 * 2 ** int(math.ceil(math.log2(L))), 16)
    _close(out, ref, f"ext out L={L}")
    _close(du, ur.grad, f"ext du L={L}")
    _close(dk, kr.grad, f"ext dk L={L}")
    _close(dD, Dr.grad, f"ext dD L={L}")
    # dtype dispatch of the reference extension (fftconv.cpp:12-31): half / bfloat16 I/O with fp32 math
    for dt, tol in ((torch.float16, 2e-3), (torch.bfloat16, 1.6e-2)):
        k_f = torch.fft.rfft(k.to(dev), n=fft_size).contiguous()
        o16 = F.fftconv_fwd(u.to(dev).to(dt), k_f, Dv.to(dev), None, 1, None, None, False, False, False, fft_size, False,
                            False, False)
        assert o16.dtype == dt
        ref16 = O.fftconv_ref(u.to(dt).double(), k.double(), Dv.double())
        # the output is rounded to the 16-bit type: half an ulp of fp16 (2^-11) / bf16 (2^-8) of the value, plus the same of max|y|
        PU.check(o16.float(), ref16, f"ext out {dt} L={L}", rtol=tol, atol=tol * max(1.0, float(ref16.abs().max())))


def test_validation_of_spectrum_and_filter_shapes():
    """ADVICE r1: mismatched k / kspec / D used to give silently wrong results."""
    import hyena_dna_b200 as H
    dev = _dev()
    u = torch.randn(1, 2, 3000, device=dev)
    D = torch.randn(2, device=dev)
    good = H.ops.filter_spectrum(torch.randn(2, 3000, device=dev))
    H.ops.fftconv_forward(u, good, D)
    with pytest.raises(H.HyenaB200Error):          # the reference's rfft(k, fft_size) handed to the packed-spectrum op
        H.ops.fftconv_forward(u, torch.fft.rfft(torch.randn(2, 3000, device=dev), n=8192), D)
    with pytest.raises(H.HyenaB200Error):          # spectrum of another length class
        H.ops.fftconv_forward(u, H.ops.filter_spectrum(torch.randn(2, 1000, device=dev)), D)
    with pytest.raises(H.HyenaB200Error):          # wrong number of rows
        H.ops.fftconv_forward(u, H.ops.filter_spectrum(torch.randn(3, 3000, device=dev)), D)
    with pytest.raises(H.HyenaB200Error):
        H.ops.fftconv_forward(u, good, torch.randn(3, device=dev))
    with pytest.raises(H.HyenaB200Error):
        H.fftconv_func(u, torch.randn(3, 3000, device=dev), D, gelu=False)
    # a shorter / longer k is zero-padded / truncated like rfft(k, n=fft_size) does
    k_short = torch.randn(2, 1000, device=dev)
    a = H.fftconv_func(u, k_short, D, gelu=False)
    b = H.fftconv_func(u, torch.nn.functional.pad(k_short, (0, 2000)), D, gelu=False)
    assert torch.equal(a, b)
    k_long = torch.randn(2, 5000, device=dev)
    assert torch.equal(H.fftconv_func(u, k_long, D, gelu=False), H.fftconv_func(u, k_long[:, :3000].contiguous(), D, gelu=False))
    f = H.HyenaFilter(8, emb_dim=5, order=64, seq_len=128, w=10.0).to(dev)
    with pytest.raises(H.HyenaB200Error):          # filter longer than the positional embedding
        f.filter(129)


# ------------------------------------------------------------------------------------------ own projection GEMM
@pytest.mark.parametrize("B,L,K,N", [(1, 128, 32, 128), (2, 1000, 64, 192), (1, 4096, 256, 768), (2, 777, 24, 8),
                                     (1, 2048, 768, 256), (1, 333, 40, 200)])
def test_proj_gemm_tcgen05_matches_fp64(B, L, K, N):
    """csrc/proj_gemm.cuh (tcgen05, 3xTF32, A operand in tensor memory) against float64 matmuls, all four layout
    combinations, bias epilogue, ragged shapes, and the fused transposed short filter."""
    import hyena_dna_b200 as H
    dev = _dev()
    g = torch.Generator().manual_seed(L + K + N)
    W = (torch.randn(N, K, generator=g) * 0.05)
    bias = torch.randn(N, generator=g)
    for act_layout in (0, 1):
        act = torch.randn((B, L, K) if act_layout == 0 else (B, K, L), generator=g)
        a64 = act.double() if act_layout == 0 else act.double().transpose(1, 2)          # (B, L, K)
        for out_layout in (0, 1):
            for wt in (False, True):
                Wd = W.t().contiguous() if wt else W
                ref = torch.matmul(a64, W.double().t()) + bias.double()                      # (B, L, N)
                if out_layout == 0:
                    ref = ref.transpose(1, 2)
                got = H.ops.proj_gemm(act.to(dev), act_layout, Wd.to(dev), wt, out_layout, bias=bias.to(dev))
                _close(got, ref, f"proj_gemm act{act_layout} out{out_layout} wt{wt} {B}x{L}x{K}x{N}")
    # fused transposed FIR on a channel-major activation
    ds = torch.randn(B, K, L, generator=g)
    taps = torch.randn(K, 3, generator=g)
    dsp = torch.nn.functional.pad(ds.double(), (0, 2))
    dp = taps[:, 2].double()[None, :, None] * dsp[..., :L] + taps[:, 1].double()[None, :, None] * dsp[..., 1:L + 1] \
        + taps[:, 0].double()[None, :, None] * dsp[..., 2:L + 2]
    ref = torch.matmul(dp.transpose(1, 2), W.double().t())
    got = H.ops.proj_gemm(ds.to(dev), 1, W.to(dev), False, 1, fir=taps.to(dev))
    _close(got, ref, f"proj_gemm fused FIR {B}x{L}x{K}x{N}")


@pytest.mark.parametrize("B,L,M,N", [(1, 64, 128, 256), (2, 1000, 192, 64), (1, 40000, 768, 256), (2, 777, 24, 8),
                                     (1, 5000, 256, 256), (1, 333, 200, 320)])
def test_proj_wgrad_tcgen05_matches_fp64(B, L, M, N):
    """Split-K weight-gradient GEMM (MN-major B operand, A in tensor memory) against float64, plain and with the fused
    transposed short filter, normal and transposed output."""
    import hyena_dna_b200 as H
    dev = _dev()
    g = torch.Generator().manual_seed(L + M + N)
    X = torch.randn(B, M, L, generator=g)
    Y = torch.randn(B, L, N, generator=g)
    ref = torch.einsum("bml,bln->mn", X.double(), Y.double())
    got = H.ops.proj_wgrad(X.to(dev), Y.to(dev))
    _close(got, ref, f"wgrad {B}x{L}x{M}x{N}")
    got_t = H.ops.proj_wgrad(X.to(dev), Y.to(dev), transposed_out=True)
    _close(got_t, ref.t(), f"wgrad transposed {B}x{L}x{M}x{N}")
    taps = torch.randn(M, 3, generator=g)
    Xp = torch.nn.functional.pad(X.double(), (0, 2))
    dp = taps[:, 2].double()[None, :, None] * Xp[..., :L] + taps[:, 1].double()[None, :, None] * Xp[..., 1:L + 1] \
        + taps[:, 0].double()[None, :, None] * Xp[..., 2:L + 2]
    ref_f = torch.einsum("bml,bln->mn", dp, Y.double())
    got_f = H.ops.proj_wgrad(X.to(dev), Y.to(dev), fir=taps.to(dev))
    _close(got_f, ref_f, f"wgrad fused FIR {B}x{L}x{M}x{N}")


# ------------------------------------------------------------------------------------------ order 3
@pytest.mark.parametrize("case", ["ref_order3_L256_D16", "ref_order3_L200_D8"])
def test_operator_order3_matches_reference_golden(case):
    """order = 3 (configs/model/layer/hyena_dna.yaml:3; recurrence loop hyena.py:414-423) against vectors generated by the
    unmodified src/models/sequence/hyena.py (filter channels ordered '(v o)', hyena.py:408-412)."""
    import hyena_dna_b200 as H
    dev = _dev()
    G = load(case)
    op = H.HyenaOperator(G["D"], G["l_max"], order=3, filter_order=64, emb_dim=G["E"], w=G["w"], lr_pos_emb=0.0)
    op.load_state_dict(G["sd"], strict=True)
    op = op.to(dev)
    u = G["u"].to(dev).requires_grad_(True)
    y = op(u)
    y.backward(G["dy"].to(dev))
    _close(y, G["y"], f"{case} y")
    _close(u.grad, G["du"], f"{case} du")
    got = dict(op.named_parameters())
    for name, gref in G["grad"].items():
        _close(got[name].grad, gref, f"{case} grad {name}")


def test_operator_order3_long_sequence_matches_oracle_fp64():
    dev = _dev()
    import hyena_dna_b200 as H
    B, L, D = 1, 65536, 16
    g = torch.Generator().manual_seed(33)
    P = O.init_params(D, L, order=3, emb_dim=5, w=10.0, generator=g, init_std=0.02)
    u, _ = O.nucleotide_activations(B, L, D, seed=2222)
    dy = torch.randn(B, L, D, generator=torch.Generator().manual_seed(1))
    y64, du64, g64 = O.operator_fwd_bwd(u.double(), O.to_dtype(P, torch.float64), dy.double())
    sd = dict(P)
    for extra in ("filter_fn.implicit_filter.3.freq", "filter_fn.implicit_filter.5.freq"):
        sd[extra] = sd["filter_fn.implicit_filter.1.freq"]
    op = H.HyenaOperator(D, L, order=3, filter_order=64, emb_dim=5, w=10.0, lr_pos_emb=0.0)
    op.load_state_dict(sd, strict=True)
    op = op.to(dev)
    ug = u.to(dev).requires_grad_(True)
    y = op(ug)
    y.backward(dy.to(dev))
    _close(y, y64, "order3 y")
    _close(ug.grad, du64, "order3 du")
    got = dict(op.named_parameters())
    for name, gref in g64.items():
        _close(got[name].grad, gref, f"order3 grad {name}")


# ------------------------------------------------------------------------------------------ checkpointed stack (f2)
def test_checkpointed_stack_reuses_filter_and_matches_plain_autograd():
    """Two operators with a residual connection, each in its own checkpoint region: same outputs and gradients as the plain
    stack, and the recompute forward launches NO filter / spectrum kernels (cache hit), cf. long_conv_lm.py:39-45."""
    import hyena_dna_b200 as H
    dev = _dev()
    torch.manual_seed(3)
    B, L, D = 1, 4096, 32
    layers = [H.HyenaOperator(D, L, emb_dim=5, w=10.0, lr_pos_emb=0.0) for _ in range(2)]
    plain = H.CheckpointedHyenaStack(layers, use_checkpoint=False, cache_filter=False).to(dev)
    u = torch.randn(B, L, D, device=dev)
    dy = torch.randn(B, L, D, device=dev)
    up = u.clone().requires_grad_(True)
    yp = plain(up)
    yp.backward(dy)
    ref = {n: p.grad.clone() for n, p in plain.named_parameters()}
    for p in plain.parameters():
        p.grad = None
    ck = H.CheckpointedHyenaStack(layers, use_checkpoint=True, cache_filter=True).to(dev)
    uc = u.clone().requires_grad_(True)
    yc = ck(uc)
    H._lib.profile_begin()
    yc.backward(dy)
    prof = H._lib.profile_end()
    _close(yc, yp, "checkpointed y")
    _close(uc.grad, up.grad, "checkpointed du")
    for n, p in ck.named_parameters():
        _close(p.grad, ref[n], f"checkpointed grad {n}")
    # the backward window contains the recompute forwards: no forward filter / filter-spectrum kernels in it
    assert "filter_tc_fwd" not in prof and "row_pass<filter>" not in prof and "col_fwd<filter>" not in prof, prof.keys()
    # an optimizer step invalidates the cache
    with torch.no_grad():
        for p in ck.parameters():
            p.add_(0.01 * torch.randn_like(p))
    H._lib.profile_begin()
    with torch.no_grad():
        ck(u)
    prof2 = H._lib.profile_end()
    assert "filter_tc_fwd" in prof2
    plan = H.memory_plan(1, 1 << 20, 256, 8)
    assert plan["total"] < 180e9


# ------------------------------------------------------------------------------------------ fftconv variants (S8 f4)
@pytest.mark.parametrize("name", ["krev_L100", "krev_L257", "bidir_L128", "bidir_L101"])
def test_fftconv_k_rev_and_bidirectional_match_reference_golden(name):
    """k_rev (src/ops/fftconv.py:66-67, hyena.py:63-65) and bidirectional (hyena.py:67-73): fixtures from the unmodified
    reference fftconv_ref (tests/golden/make_golden_fftconv.py), forward and all gradients, fp64 truth alongside."""
    import os
    import numpy as np
    import hyena_dna_b200 as H
    dev = _dev()
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "fftconv_variants.npz"))
    T = lambda k: torch.from_numpy(z[f"{name}/{k}"])
    B, Hh, L, with_rev, bidir = (int(v) for v in z[f"{name}/cfg"])
    u = T("u").to(dev).requires_grad_(True); k = T("k").to(dev).requires_grad_(True); D = T("D").to(dev).requires_grad_(True)
    kr = T("krev").to(dev).requires_grad_(True) if with_rev else None
    n0 = H.launch_count()
    y = H.fftconv_ref(u, k, D, None, gelu=False, k_rev=kr, bidirectional=bool(bidir))
    y.backward(T("dy").to(dev))
    assert H.launch_count() > n0
    PU.check(y, T("y"), f"{name} y", ref64=T("y64"))
    PU.check(u.grad, T("du"), f"{name} du", ref64=T("du64"))
    PU.check(k.grad, T("dk"), f"{name} dk", ref64=T("dk64"), param_grad=True)
    PU.check(D.grad, T("dD"), f"{name} dD", ref64=T("dD64"), param_grad=True)
    if with_rev:
        PU.check(kr.grad, T("dkrev"), f"{name} dk_rev", ref64=T("dkrev64"), param_grad=True)
        # the same through the op-level entry point of src/ops/fftconv.py:105-108
        y2 = H.fftconv_func(u.detach(), k.detach(), D.detach(), gelu=False, k_rev=kr.detach())
        PU.check(y2, T("y"), f"{name} fftconv_func y", ref64=T("y64"))
    with pytest.raises(H.HyenaB200Error):
        H.fftconv_ref(u, k, D, None, gelu=False, k_rev=k, bidirectional=True)


def test_bidirectional_filter_module_matches_oracle_fp64():
    """HyenaFilter(bidirectional=True) inside the operator (hyena.py:261 passes the flag to fftconv_ref): the operator runs the
    chained path with the delayed convolution; checked against an fp64 restatement built from the reference's formula."""
    dev = _dev()
    B, L, D = 2, 300, 8
    g = torch.Generator().manual_seed(11)
    P = O.init_params(D, L, emb_dim=5, w=10.0, generator=g, init_std=0.02)
    sd = dict(P)
    for extra in ("filter_fn.implicit_filter.3.freq", "filter_fn.implicit_filter.5.freq"):
        sd[extra] = sd["filter_fn.implicit_filter.1.freq"]
    op = _module_from_sd(sd, D, L, 5, 10.0, dev, bidirectional=True)
    u = torch.randn(B, L, D, generator=g)
    y = op(u.to(dev))
    # fp64 truth: the reference operator's formula with the bidirectional fftconv_ref restated (hyena.py:59-88)
    P64 = O.to_dtype(P, torch.float64)
    import torch.nn.functional as F
    p = F.linear(u.double(), P64["in_proj.weight"], P64["in_proj.bias"]).transpose(1, 2)
    uc = O.short_filter(p, P64["short_filter.weight"], P64["short_filter.bias"], L)
    x0, x1, v = uc.split(D, dim=1)
    k = O.hyena_filter(L, P64)[0].transpose(0, 1)
    gte = v * x1
    n = 2 * L
    pad_before = (L + 2 * (L // 2)) // 2 - L // 2
    pad_after = L + 2 * (L // 2) - L - pad_before
    gf = torch.fft.rfft(F.pad(gte, (pad_before, pad_after)), n=n)
    yc = torch.fft.irfft(gf * (torch.fft.rfft(k, n=n) / n), n=n, norm="forward")[..., :L] + gte * P64["filter_fn.bias"][:, None]
    y64 = F.linear((yc * x0).transpose(1, 2), P64["out_proj.weight"], P64["out_proj.bias"])
    PU.check(y, y64.float(), "bidirectional operator y", ref64=y64)


def test_projection_gemms_are_bitwise_deterministic_at_full_length():
    """Regression test for a slot-release race of the warp-specialised projection kernels (round 2): with the activation tiles
    refilled by TMA as soon as their barrier completed, ~1 run in 10 at L = 2^20 read a few rows the copy engine had already
    overwritten (an mbarrier arrive is not queued behind the LDS instructions that precede it: tc_prims.cuh
    mbar_arrive_after_loads).  Identical inputs must give identical bits, run after run."""
    import hyena_dna_b200 as H
    dev = _dev()
    L, D = 1 << 20, 256
    g = torch.Generator().manual_seed(0)
    u = torch.randn(1, L, D, generator=g).to(dev)
    Wi = (torch.randn(3 * D, D, generator=g) * 0.05).to(dev)
    ref = H.ops.proj_gemm(u, 0, Wi, False, 0).clone()
    for i in range(12):
        out = H.ops.proj_gemm(u, 0, Wi, False, 0)
        assert torch.equal(out, ref), f"in_proj run {i}: {int((out != ref).sum())} elements differ"
    del ref, out
    ych = torch.randn(1, D, L, generator=g).to(dev)
    dyr = torch.randn(1, L, D, generator=g).to(dev)
    refw = H.ops.proj_wgrad(ych, dyr).clone()
    for i in range(6):
        assert torch.equal(H.ops.proj_wgrad(ych, dyr), refw), f"wgrad run {i} differs"
