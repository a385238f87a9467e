"""Paths the library chooses from its input rather than from a setting: the kernel-class names, the batch-1 backward row
pass on a misaligned filter spectrum, and the cuBLASLt projections a user gets by opting into TF32."""
import pytest
import torch

from tests import parity_util as PU


def test_kind_names_are_set_and_distinct():
    """bench.py keys per-kernel bytes on these names: every kernel class has one, and no two share it."""
    from importlib import import_module
    L = import_module("hyena_dna_b200._lib").lib()
    names = [L.hyena_b200_kind_name(i) for i in range(L.hyena_b200_kind_count())]
    assert all(n for n in names), names
    assert len(set(names)) == len(names), names


def _dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    return torch.device("cuda:0")


@pytest.mark.gpu
def test_core_backward_batch1_misaligned_spectrum():
    """B = 1 with the saved g spectrum runs the staged row kernel only when kspec and gspec are 16-byte aligned; an
    8-byte aligned kspec takes the generic backward row pass, which must give the same gradients."""
    import hyena_dna_b200 as H
    dev = _dev()
    g = torch.Generator().manual_seed(21)
    B, D, L = 1, 32, 1 << 14
    p = torch.randn(B, 3 * D, L, generator=g).to(dev)
    ib = (torch.randn(3 * D, generator=g) * 0.1).to(dev)
    sw = (torch.randn(3 * D, 3, generator=g) * 0.5).to(dev)
    sb = (torch.randn(3 * D, generator=g) * 0.1).to(dev)
    fb = torch.randn(D, generator=g).to(dev)
    k = (torch.randn(D, L, generator=g) * torch.exp(-torch.arange(L) / 2000.0)).to(dev)
    dy = torch.randn(B, D, L, generator=g).to(dev)
    kspec = H.ops.filter_spectrum(k)
    _, c, gs = H.ops.core_forward(p, ib, sw, sb, kspec, fb, True)
    assert gs is not None and gs.data_ptr() % 16 == 0
    buf = torch.empty(kspec.numel() + 1, dtype=kspec.dtype, device=dev)
    kmis = buf[1:].view(kspec.shape)
    kmis.copy_(kspec)
    assert kspec.data_ptr() % 16 == 0 and kmis.data_ptr() % 16 == 8 and kmis.is_contiguous()
    ref = H.ops.core_backward(dy, p, ib, sw, sb, kspec, fb, c, gs)
    got = H.ops.core_backward(dy, p, ib, sw, sb, kmis, fb, c, gs)
    for name, a, b in zip(("dp", "dk", "dsw", "dsb", "dfbias", "d_in_bias"), got, ref):
        PU.check(a, b, f"core_backward B=1 misaligned kspec: {name}", param_grad=name not in ("dp", "dk"))


def _normwise(got, ref):
    return float((got.double() - ref).norm() / ref.norm())


@pytest.mark.gpu
def test_tf32_opt_in_projections_match_fp64():
    """allow_tf32 = True moves the projections to cuBLASLt in TF32 (mode 'lt'); forward and backward stay within a
    TF32-sized normwise error of float64 matmuls."""
    import hyena_dna_b200 as H
    from importlib import import_module
    hy = import_module("hyena_dna_b200.hyena")
    dev = _dev()
    if H.ops.gemm_mode() != "bf16x9":
        pytest.skip("cuBLASLt 12.9 is not available")
    g = torch.Generator().manual_seed(22)
    B, L, D = 2, 4096, 64
    u = torch.randn(B, L, D, generator=g).to(dev).requires_grad_(True)
    W = (torch.randn(3 * D, D, generator=g) * 0.05).to(dev).requires_grad_(True)
    dp = torch.randn(B, 3 * D, L, generator=g).to(dev)
    yp = torch.randn(B, D, L, generator=g).to(dev).requires_grad_(True)
    Wo = (torch.randn(D, D, generator=g) * 0.05).to(dev).requires_grad_(True)
    bo = torch.randn(D, generator=g).to(dev).requires_grad_(True)
    dy = torch.randn(B, L, D, generator=g).to(dev)
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        assert H.ops.proj_mode() == "lt"
        p = hy._InProj.apply(u, W)
        p.backward(dp)
        y = hy._OutProj.apply(yp, Wo, bo)
        y.backward(dy)
        torch.cuda.synchronize()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = False
    assert H.ops.proj_mode() == "tc"
    u64, W64, dp64 = u.detach().double(), W.detach().double(), dp.double()
    yp64, Wo64, dy64 = yp.detach().double(), Wo.detach().double(), dy.double()
    checks = {
        "in_proj": (p, torch.matmul(W64, u64.transpose(1, 2))),
        "in_proj du": (u.grad, torch.matmul(dp64.transpose(1, 2), W64)),
        "in_proj dW": (W.grad, torch.matmul(dp64, u64).sum(0)),
        "out_proj": (y, torch.matmul(yp64.transpose(1, 2), Wo64.t()) + bo.detach().double()),
        "out_proj dy_pre": (yp.grad, torch.matmul(Wo64.t(), dy64.transpose(1, 2))),
        "out_proj dW": (Wo.grad, torch.matmul(dy64.transpose(1, 2), yp64.transpose(1, 2)).sum(0)),
        "out_proj db": (bo.grad, dy64.sum((0, 1))),
    }
    for what, (got, ref) in checks.items():
        err = _normwise(got.detach(), ref)
        assert err <= 2e-3, f"{what}: normwise error {err:.2e} vs float64"
