"""Raw device ops (thin wrappers over the C ABI) and the autograd Functions built on them.

PyTorch provides device memory, streams and autograd plumbing; all arithmetic of the custom-kernel
span runs in libhyena_b200.so.  Inputs must be CUDA fp32 tensors -- anything else raises.
"""
import torch

from . import _lib

_ws_cache = {}


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _need_cuda(*ts):
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise _lib.HyenaB200Error("hyena_b200 ops need CUDA tensors (there is no CPU path)")
        if t.dtype != torch.float32:
            raise _lib.HyenaB200Error(f"hyena_b200 ops compute in fp32; got {t.dtype}")


def workspace(B, D, L, backward, device):
    """Cached scratch buffer for the FFT passes, one per (device, stream): two operators driven from different streams
    (DDP bucket hooks, checkpoint recompute on a side stream) never share scratch, so the op stays re-entrant across
    streams as the reference extension is (csrc/fftconv/fftconv.cpp allocates per call)."""
    n = int(_lib.lib().hyena_b200_workspace_bytes(B, D, L, int(backward)))
    key = (device.index if device.index is not None else torch.cuda.current_device(), _stream())
    buf = _ws_cache.get(key)
    if buf is None or buf.numel() < n:
        buf = torch.empty(n, dtype=torch.uint8, device=device)
        _ws_cache[key] = buf
    # hand the library exactly the bytes this call asked for: the group size (rows in flight, sized to
    # stay L2-resident) is derived from the workspace size
    return buf[:n]


def spectrum_elems(L):
    return int(_lib.lib().hyena_b200_spectrum_elems(int(L)))


# ------------------------------------------------------------------------------------------ filter
def _filter_args(z, t, W0, b0, W1, b1, W2, b2, W3, freq, deltas, shift, modulate, L):
    E = z.shape[-1]
    N = W1.shape[0]
    D = W3.shape[0]
    rows = z.shape[-2]
    if L < 1 or L > rows or L > t.shape[-2 if t.dim() == 3 else 0]:
        raise _lib.HyenaB200Error(f"filter length {L} exceeds the positional embedding ({rows} rows); the reference "
                                  "returns a seq_len-long filter, callers clamp with min(L, l_max)")
    zz = z[0, :L] if z.dim() == 3 else z[:L]
    tt = (t[0, :L, 0] if t.dim() == 3 else t[:L]).contiguous()
    if zz.stride(-1) != 1:
        zz = zz.contiguous()
    return zz, tt, E, N, D


def filter_forward(z, t, W0, b0, W1, b1, W2, b2, W3, freq, deltas, shift, modulate, L):
    """k (D, L) channel-major == HyenaFilter.filter(L)[0].T  (hyena.py:229-238)."""
    _need_cuda(z, t, W0, b0, W1, b1, W2, b2, W3, freq, deltas)
    zz, tt, E, N, D = _filter_args(z, t, W0, b0, W1, b1, W2, b2, W3, freq, deltas, shift, modulate, L)
    k = torch.empty(D, L, dtype=torch.float32, device=z.device)
    ws = [x.contiguous() for x in (W0, b0, W1, b1, W2, b2, W3)]
    fr = freq.reshape(-1).contiguous()
    dl = deltas.reshape(-1).contiguous()
    with torch.cuda.device(z.device):
        _lib.check(_lib.lib().hyena_b200_filter_fwd(
            _ptr(zz), zz.stride(0), _ptr(tt), *[_ptr(w) for w in ws], _ptr(fr), _ptr(dl),
            float(shift), int(bool(modulate)), int(L), E, N, D, _ptr(k), _stream()))
    return k


def filter_backward(z, t, W0, b0, W1, b1, W2, b2, W3, freq, deltas, shift, modulate, L, dk, need_dz):
    """Tensor-core backward: stage 1 on tcgen05 (csrc/filter_tc.cuh), stage 2 = sequence-length reductions."""
    _need_cuda(z, t, W0, b0, W1, b1, W2, b2, W3, freq, deltas, dk)
    zz, tt, E, N, D = _filter_args(z, t, W0, b0, W1, b1, W2, b2, W3, freq, deltas, shift, modulate, L)
    ws = [x.contiguous() for x in (W0, b0, W1, b1, W2, b2, W3)]
    fr = freq.reshape(-1).contiguous()
    dl = deltas.reshape(-1).contiguous()
    dk = dk.contiguous()
    dev = z.device
    dh = torch.empty(D, L, dtype=torch.float32, device=dev)
    sc = torch.empty(7, 64, L, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().hyena_b200_filter_bwd_stage1(
            _ptr(zz), zz.stride(0), _ptr(tt), *[_ptr(w) for w in ws], _ptr(fr), _ptr(dl),
            float(shift), int(bool(modulate)), int(L), E, N, D, _ptr(dk), _ptr(dh), _ptr(sc), _stream()))
    a1, a2, a3, dp1, dp2, dp3, X = sc.unbind(0)          # feature-major (64, L) each
    if D <= 256 and E <= 8:
        grads = [torch.zeros_like(w) for w in ws]
        dfreq = torch.zeros(64, dtype=torch.float32, device=dev)
        zT = zz.t().contiguous()
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().hyena_b200_filter_bwd_stage2(
                _ptr(dh), _ptr(sc), _ptr(zT), *[_ptr(g) for g in grads], _ptr(dfreq), int(L), E, D, _stream()))
    else:                                             # wide models: library GEMMs with K = L
        sums = sc[3:7].sum(dim=2)
        grads = [dp1 @ zz, sums[0], dp2 @ a1.t(), sums[1], dp3 @ a2.t(), sums[2], dh @ a3.t()]
        dfreq = sums[3]
    dz = (dp1.t() @ ws[0]) if need_dz else None
    return grads, dfreq, dz


class HyenaFilterFn(torch.autograd.Function):
    """Differentiable implicit filter: parameters -> k (D, L)."""

    @staticmethod
    def forward(ctx, z, t, W0, b0, W1, b1, W2, b2, W3, freq, deltas, shift, modulate, L, cached=None):
        ctx.cfg = (shift, modulate, L)
        if cached is not None:                 # same inputs as the call that produced it (HyenaFilter.filter_channel_major)
            k = cached.detach()
        else:
            k = filter_forward(z, t, W0, b0, W1, b1, W2, b2, W3, freq, deltas, shift, modulate, L)
        # trainable deltas (modulation_lr != 0): their gradient needs the filter itself
        need_k = modulate and torch.is_tensor(deltas) and deltas.requires_grad
        ctx.save_for_backward(z, t, W0, b0, W1, b1, W2, b2, W3, freq, deltas, k if need_k else None)
        return k

    @staticmethod
    def backward(ctx, dk):
        z, t, W0, b0, W1, b1, W2, b2, W3, freq, deltas, ksaved = ctx.saved_tensors
        shift, modulate, L = ctx.cfg
        ddelta = None
        if ctx.needs_input_grad[10]:
            if not modulate or ksaved is None:
                ddelta = torch.zeros_like(deltas)
            else:                                      # ExponentialModulation with modulation_lr != 0 (hyena.py:145-155)
                D = ksaved.shape[0]
                dkc = dk.contiguous()
                tt = (t[0, :L, 0] if t.dim() == 3 else t[:L]).contiguous()
                dl = deltas.reshape(-1).contiguous()
                dd = torch.empty(D, dtype=torch.float32, device=dk.device)
                with torch.cuda.device(dk.device):
                    _lib.check(_lib.lib().hyena_b200_filter_ddelta(_ptr(dkc), _ptr(ksaved), _ptr(tt), _ptr(dl), float(shift),
                                                                    D, int(L), _ptr(dd), _stream()))
                ddelta = dd.reshape(deltas.shape)
        need_dz = ctx.needs_input_grad[0]
        grads, dfreq, dz = filter_backward(z, t, W0, b0, W1, b1, W2, b2, W3, freq, deltas, shift, modulate, L,
                                           dk, need_dz)
        gz = None
        if need_dz:
            gz = torch.zeros_like(z)
            (gz[0, :L] if z.dim() == 3 else gz[:L]).copy_(dz)
        return (gz, None, *grads, dfreq.reshape(freq.shape), ddelta, None, None, None, None)


class FilterL1NormFn(torch.autograd.Function):
    """k (D, L) -> k / sum_c |k[c, t]|: HyenaFilter(normalized=True), hyena.py:235-236 (L1 norm over the channel dim of the
    reference's (1, L, D) layout)."""

    @staticmethod
    def forward(ctx, k):
        _need_cuda(k)
        k = k.contiguous()
        D, L = k.shape
        out = torch.empty_like(k)
        norm = torch.empty(L, dtype=torch.float32, device=k.device)
        with torch.cuda.device(k.device):
            _lib.check(_lib.lib().hyena_b200_filter_l1norm_fwd(_ptr(k), _ptr(out), _ptr(norm), D, L, _stream()))
        ctx.save_for_backward(out, norm)
        return out

    @staticmethod
    def backward(ctx, dout):
        out, norm = ctx.saved_tensors
        dout = dout.contiguous()
        _need_cuda(dout)
        D, L = out.shape
        dk = torch.empty_like(out)
        with torch.cuda.device(out.device):
            _lib.check(_lib.lib().hyena_b200_filter_l1norm_bwd(_ptr(dout), _ptr(out), _ptr(norm), _ptr(dk), D, L, _stream()))
        return dk


# ------------------------------------------------------------------------------------------ spectrum / core
def filter_spectrum(k):
    """Opaque packed spectrum of k (D, L) -> (D, M) complex64 (replaces rfft(k, 2L)/2L, hyena.py:62)."""
    _need_cuda(k)
    k = k.contiguous()
    D, L = k.shape
    M = spectrum_elems(L)
    spec = torch.empty(D, M, dtype=torch.complex64, device=k.device)
    ws = workspace(1, D, L, False, k.device)
    with torch.cuda.device(k.device):
        _lib.check(_lib.lib().hyena_b200_filter_spectrum(_ptr(k), _ptr(spec), D, L, _ptr(ws), ws.numel(), _stream()))
    return spec


def _check_spectrum(kspec, H, L, what):
    """The packed spectrum is opaque but its type and shape are not: (H, spectrum_elems(L)) complex64, contiguous, on the
    same device -- anything else (e.g. the reference's rfft(k, fft_size), src/ops/fftconv.py:65) would be read out of
    bounds or silently misinterpreted by the kernels."""
    M = spectrum_elems(L)
    if not (torch.is_tensor(kspec) and kspec.is_cuda and kspec.dtype == torch.complex64 and kspec.dim() == 2
            and tuple(kspec.shape) == (H, M) and kspec.is_contiguous()):
        got = (tuple(kspec.shape), kspec.dtype) if torch.is_tensor(kspec) else type(kspec)
        raise _lib.HyenaB200Error(f"{what}: filter spectrum must be the packed form from filter_spectrum(): contiguous "
                                  f"complex64 ({H}, {M}) on the GPU; got {got}.  For the reference's rfft(k, fft_size) "
                                  "use fftconv.fftconv_fwd / fftconv_bwd, which convert it")


def spectrum_from_rfft(filt, L, fft_size):
    """rfft(k, n=fft_size) (H, fft_size/2+1) complex64 -- the filter the reference extension takes
    (src/ops/fftconv.py:64-65) -- to the packed spectrum the kernels consume."""
    if not (torch.is_tensor(filt) and filt.is_cuda and filt.dtype == torch.complex64 and filt.dim() == 2
            and filt.shape[1] == fft_size // 2 + 1):
        raise _lib.HyenaB200Error(f"filter must be a CUDA complex64 (H, fft_size/2+1 = {fft_size // 2 + 1}) tensor")
    filt = filt.contiguous()
    H = filt.shape[0]
    M = spectrum_elems(L)
    spec = torch.empty(H, M, dtype=torch.complex64, device=filt.device)
    ksc = torch.empty(H, L, dtype=torch.float32, device=filt.device) if fft_size < 2 * M else None
    ws = workspace(1, H, L, False, filt.device)
    with torch.cuda.device(filt.device):
        _lib.check(_lib.lib().hyena_b200_spectrum_from_rfft(_ptr(filt), int(fft_size), _ptr(spec), _ptr(ksc), H, int(L),
                                                            _ptr(ws), ws.numel(), _stream()))
    return spec


def spectrum_to_rfft(dk, fft_size):
    """dk (H, L) time domain -> dfilter (H, fft_size/2+1) complex64 with irfft(dfilter, n=fft_size, norm='forward')[:L]
    == dk: what csrc/fftconv/fftconv.cpp:235 returns and src/ops/fftconv.py:98 consumes."""
    _need_cuda(dk)
    dk = dk.contiguous()
    H, L = dk.shape
    M = spectrum_elems(L)
    out = torch.empty(H, fft_size // 2 + 1, dtype=torch.complex64, device=dk.device)
    ssc = torch.empty(H, M, dtype=torch.complex64, device=dk.device) if fft_size == 2 * M else None
    ws = workspace(1, H, L, False, dk.device)
    with torch.cuda.device(dk.device):
        _lib.check(_lib.lib().hyena_b200_spectrum_to_rfft(_ptr(dk), int(fft_size), _ptr(out), _ptr(ssc), H, int(L),
                                                          _ptr(ws), ws.numel(), _stream()))
    return out


def _save_spectrum():
    import os
    return os.environ.get("HYENA_B200_SAVE_SPECTRUM", "1") != "0"


def core_forward(p, in_bias, sw, sb, kspec, fbias, save_c):
    _need_cuda(p, in_bias, sw, sb, fbias)
    B, C3, L = p.shape
    D = C3 // 3
    if C3 != 3 * D or not p.is_contiguous():
        raise _lib.HyenaB200Error("core_forward: p must be contiguous (B, 3D, L)")
    _check_spectrum(kspec, D, L, "core_forward")
    if sw.numel() != 3 * C3 or sb.numel() != C3 or fbias.numel() != D or (in_bias is not None and in_bias.numel() != C3):
        raise _lib.HyenaB200Error("core_forward: short filter / bias shapes do not match p")
    y = torch.empty(B, D, L, dtype=torch.float32, device=p.device)
    c = torch.empty(B, D, L, dtype=torch.float32, device=p.device) if save_c else None
    # spectrum of the gated input, rows ordered (c, b): saves a column pass + a row FFT per row in backward
    gs = (torch.empty(D * B, kspec.shape[-1], dtype=torch.complex64, device=p.device)
          if (save_c and _save_spectrum()) else None)
    ws = workspace(B, D, L, False, p.device)
    with torch.cuda.device(p.device):
        _lib.check(_lib.lib().hyena_b200_core_fwd(
            _ptr(p), _ptr(in_bias), _ptr(sw), _ptr(sb), _ptr(kspec), _ptr(fbias), _ptr(y), _ptr(c), _ptr(gs),
            B, D, L, _ptr(ws), ws.numel(), _stream()))
    return y, c, gs


def core_backward(dy_pre, p, in_bias, sw, sb, kspec, fbias, c_saved, gspec=None, return_ds=False):
    _need_cuda(dy_pre, p, in_bias, sw, sb, fbias, c_saved)
    B, C3, L = p.shape
    D = C3 // 3
    dev = p.device
    _check_spectrum(kspec, D, L, "core_backward")
    if tuple(dy_pre.shape) != (B, D, L) or tuple(c_saved.shape) != (B, D, L):
        raise _lib.HyenaB200Error("core_backward: dy_pre / c_saved must be (B, D, L)")
    dy_pre = dy_pre.contiguous()
    dp = None if return_ds else torch.empty_like(p)
    ds = torch.empty_like(p)
    dk = torch.empty(D, L, dtype=torch.float32, device=dev)
    dsw = torch.zeros(C3, 3, dtype=torch.float32, device=dev)
    dsb = torch.zeros(C3, dtype=torch.float32, device=dev)
    dfb = torch.zeros(D, dtype=torch.float32, device=dev)
    dib = torch.zeros(C3, dtype=torch.float32, device=dev) if in_bias is not None else None
    ws = workspace(B, D, L, True, dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().hyena_b200_core_bwd(
            _ptr(dy_pre), _ptr(p), _ptr(in_bias), _ptr(sw), _ptr(sb), _ptr(kspec), _ptr(fbias), _ptr(c_saved),
            _ptr(gspec), _ptr(dp), _ptr(dk), _ptr(dsw), _ptr(dsb), _ptr(dfb), _ptr(dib), _ptr(ds),
            B, D, L, _ptr(ws), ws.numel(), _stream()))
    if return_ds:
        # d in_proj.bias = sum_t dp[t] = (w0 + w1 + w2) sum_t ds[t] - w1 ds[0] - w0 (ds[0] + ds[1])   (conv padding edge)
        if in_bias is not None:
            e0 = ds[:, :, 0].sum(0)
            e1 = ds[:, :, 1].sum(0) if L > 1 else torch.zeros_like(e0)
            dib = sw.sum(1) * dsb - sw[:, 1] * e0 - sw[:, 0] * (e0 + e1)
        return ds, dk, dsw, dsb, dfb, dib
    del ds
    return dp, dk, dsw, dsb, dfb, dib


class HyenaCoreFn(torch.autograd.Function):
    """(p, in_bias, short filter, k, filter bias) -> y_pre (B, D, L); hyena.py:394-432 for order 2."""

    @staticmethod
    def forward(ctx, p, in_bias, sw, sb, k, fbias, kspec=None):
        p = p.contiguous()
        sw2 = sw.reshape(sw.shape[0], -1).contiguous()
        sb = sb.contiguous(); fbias = fbias.contiguous()
        ib = in_bias.contiguous() if in_bias is not None else None
        if kspec is None:
            kspec = filter_spectrum(k)
        need = any(ctx.needs_input_grad)
        y, c, gs = core_forward(p, ib, sw2, sb, kspec, fbias, need)
        ctx.save_for_backward(p, ib, sw2, sb, kspec, fbias, c, gs)
        ctx.sw_shape = sw.shape
        return y

    @staticmethod
    def backward(ctx, dy):
        p, ib, sw2, sb, kspec, fbias, c, gs = ctx.saved_tensors
        dp, dk, dsw, dsb, dfb, dib = core_backward(dy, p, ib, sw2, sb, kspec, fbias, c, gs)
        return dp, dib, dsw.reshape(ctx.sw_shape), dsb, dk, dfb, None


class HyenaInCoreFn(torch.autograd.Function):
    """in_proj + operator core as ONE autograd node (tcgen05 projections): u (B, L, D) -> y_pre (B, D, L).

    Forward: p = W u^T channel-major (proj_gemm), then the fused core.  Backward: the core returns ds (gradient w.r.t. the
    short-filter outputs) and the two projection-backward GEMMs apply the transposed 3-tap filter to it on the fly, so
    neither dp nor a separate short-filter backward pass exists (hyena.py:391-432 and its autograd)."""

    @staticmethod
    def forward(ctx, u, W, in_bias, sw, sb, k, fbias, kspec=None):
        u = u.contiguous(); W = W.contiguous()
        sw2 = sw.reshape(sw.shape[0], -1).contiguous()
        sb = sb.contiguous(); fbias = fbias.contiguous()
        ib = in_bias.contiguous() if in_bias is not None else None
        p = proj_gemm(u, 0, W, False, 0)
        if kspec is None:
            kspec = filter_spectrum(k)
        need = any(ctx.needs_input_grad)
        y, c, gs = core_forward(p, ib, sw2, sb, kspec, fbias, need)
        ctx.save_for_backward(u, W, p, ib, sw2, sb, kspec, fbias, c, gs)
        ctx.sw_shape = sw.shape
        return y

    @staticmethod
    def backward(ctx, dy):
        u, W, p, ib, sw2, sb, kspec, fbias, c, gs = ctx.saved_tensors
        ds, dk, dsw, dsb, dfb, dib = core_backward(dy, p, ib, sw2, sb, kspec, fbias, c, gs, return_ds=True)
        du = proj_gemm(ds, 1, W, True, 1, fir=sw2) if ctx.needs_input_grad[0] else None
        dW = proj_wgrad(ds, u, fir=sw2) if ctx.needs_input_grad[1] else None
        return du, dW, dib, dsw.reshape(ctx.sw_shape), dsb, dk, dfb, None


# ------------------------------------------------------------------------------------------ incremental decoding
def decode_workspace_bytes(B, D, max_len):
    return int(_lib.lib().hyena_b200_decode_workspace_bytes(int(B), int(D), int(max_len)))


def decode_prefill(p, in_bias, sw, sb, g_hist, fir):
    """Decode state from a prompt: g_hist[:, :, :Lp] (gated history) and fir (last two biased in_proj outputs) from the
    prompt's p (B, 3D, Lp), the in_proj output without its bias."""
    _need_cuda(p, in_bias, sw, sb, g_hist, fir)
    B, C3, Lp = p.shape
    D = C3 // 3
    max_len = g_hist.shape[-1]
    if not (p.is_contiguous() and g_hist.is_contiguous() and fir.is_contiguous() and C3 == 3 * D
            and tuple(g_hist.shape) == (B, D, max_len) and tuple(fir.shape) == (B, C3, 2)):
        raise _lib.HyenaB200Error("decode_prefill: p (B, 3D, Lp), g_hist (B, D, max_len), fir (B, 3D, 2), contiguous")
    with torch.cuda.device(p.device):
        _lib.check(_lib.lib().hyena_b200_decode_prefill(_ptr(p), _ptr(in_bias), _ptr(sw), _ptr(sb), _ptr(g_hist), _ptr(fir),
                                                        B, D, Lp, max_len, _stream()))


def decode_step(u_t, W_in, in_bias, sw, sb, k, fbias, W_out, out_bias, g_hist, fir, t, ws):
    """One token at position t: u_t (B, D) -> y_t (B, D); appends g_t to g_hist and advances fir (csrc/k_decode.cu)."""
    _need_cuda(u_t, W_in, in_bias, sw, sb, k, fbias, W_out, out_bias, g_hist, fir)
    B, D = u_t.shape
    max_len = g_hist.shape[-1]
    for x in (u_t, W_in, in_bias, sw, sb, k, fbias, W_out, out_bias, g_hist, fir):
        if x is not None and not x.is_contiguous():
            raise _lib.HyenaB200Error("decode_step: every tensor must be contiguous")
    if (tuple(W_in.shape) != (3 * D, D) or tuple(W_out.shape) != (D, D) or tuple(k.shape) != (D, max_len)
            or tuple(g_hist.shape) != (B, D, max_len) or tuple(fir.shape) != (B, 3 * D, 2)):
        raise _lib.HyenaB200Error("decode_step: shapes do not match u_t (B, D) and g_hist (B, D, max_len)")
    y = torch.empty(B, D, dtype=torch.float32, device=u_t.device)
    with torch.cuda.device(u_t.device):
        _lib.check(_lib.lib().hyena_b200_decode_step(
            _ptr(u_t), _ptr(W_in), _ptr(in_bias), _ptr(sw), _ptr(sb), _ptr(k), _ptr(fbias), _ptr(W_out), _ptr(out_bias),
            _ptr(g_hist), _ptr(fir), _ptr(y), B, D, int(t), max_len, _ptr(ws), ws.numel(), _stream()))
    return y


# ------------------------------------------------------------------------------------------ plain fftconv
def fftconv_forward(u, kspec, Dvec):
    _need_cuda(u, Dvec)
    if u.dim() != 3 or not u.is_contiguous():
        raise _lib.HyenaB200Error("fftconv_forward: u must be contiguous (B, H, L)")
    B, H, L = u.shape
    _check_spectrum(kspec, H, L, "fftconv_forward")
    if Dvec.numel() != H or not Dvec.is_contiguous():
        raise _lib.HyenaB200Error(f"fftconv_forward: D must have {H} contiguous elements, got {tuple(Dvec.shape)}")
    out = torch.empty_like(u)
    ws = workspace(B, H, L, False, u.device)
    with torch.cuda.device(u.device):
        _lib.check(_lib.lib().hyena_b200_fftconv_fwd(_ptr(u), _ptr(kspec), _ptr(Dvec), _ptr(out), B, H, L,
                                                     _ptr(ws), ws.numel(), _stream()))
    return out


def fftconv_backward(dout, u, kspec, Dvec):
    _need_cuda(dout, u, Dvec)
    if u.dim() != 3 or not u.is_contiguous() or tuple(dout.shape) != tuple(u.shape) or not dout.is_contiguous():
        raise _lib.HyenaB200Error("fftconv_backward: u and dout must be contiguous (B, H, L) of the same shape")
    B, H, L = u.shape
    _check_spectrum(kspec, H, L, "fftconv_backward")
    if Dvec.numel() != H or not Dvec.is_contiguous():
        raise _lib.HyenaB200Error(f"fftconv_backward: D must have {H} contiguous elements, got {tuple(Dvec.shape)}")
    du = torch.empty_like(u)
    dk = torch.empty(H, L, dtype=torch.float32, device=u.device)
    dD = torch.zeros(H, dtype=torch.float32, device=u.device)
    ws = workspace(B, H, L, True, u.device)
    with torch.cuda.device(u.device):
        _lib.check(_lib.lib().hyena_b200_fftconv_bwd(_ptr(dout), _ptr(u), _ptr(kspec), _ptr(Dvec), _ptr(du), _ptr(dk),
                                                     _ptr(dD), B, H, L, _ptr(ws), ws.numel(), _stream()))
    return du, dk, dD


# ------------------------------------------------------------------------------------------ projections
_gemm_ws = {}
_gemm_mode = None


def gemm_mode():
    """'bf16x9' when the CUDA 12.9 cuBLASLt with fp32 emulation is usable, else 'torch' (no such library: the
    projections then stay on the tcgen05 kernels even with the TF32 opt-in, see proj_mode)."""
    global _gemm_mode
    if _gemm_mode is None:
        _gemm_mode = "torch"
        if torch.cuda.is_available() and _lib.lib().hyena_b200_gemm_available():
            _gemm_mode = "bf16x9"
    return _gemm_mode


def gemm(transa, transb, m, n, k, A, lda, strideA, B, ldb, strideB, C, ldc, strideC, batch=1, beta=0.0, bias=None,
         emulate=None):
    """Column-major strided-batched C = op(A) op(B) + beta*C (+bias) on cuBLASLt 12.9 (see csrc/gemm.cu).

    Precision follows PyTorch's own switch, like the reference's nn.Linear does: fp32-accurate BF16x9 emulation by
    default, TF32 tensor cores when the user set ``torch.backends.cuda.matmul.allow_tf32 = True`` (the reference
    training script does, train.py:34-35)."""
    if emulate is None:
        emulate = 2 if torch.backends.cuda.matmul.allow_tf32 else 1
    dev = C.device
    # one workspace per (device, stream): GEMMs issued on different streams may run concurrently
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), _stream())
    ws = _gemm_ws.get(key)
    if ws is None:
        ws = torch.empty(64 << 20, dtype=torch.uint8, device=dev)
        _gemm_ws[key] = ws
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().hyena_b200_gemm(int(transa), int(transb), m, n, k, 1.0, _ptr(A), lda, strideA,
                                              _ptr(B), ldb, strideB, float(beta), _ptr(C), ldc, strideC, batch,
                                              _ptr(bias), int(emulate), _ptr(ws), ws.numel(), _stream()))
    return C


_wimg_cache = {}


def proj_mode():
    """'tc': the projections run on this library's tcgen05 3xTF32 kernels (csrc/proj_gemm.cuh) -- the default;
    'lt': cuBLASLt 12.9 in plain TF32 (csrc/gemm.cu), when the user opted into TF32 via
    torch.backends.cuda.matmul.allow_tf32 and that library is usable: one MMA per product."""
    if torch.backends.cuda.matmul.allow_tf32 and gemm_mode() == "bf16x9":
        return "lt"
    return "tc"


def proj_gemm(act, act_layout, W, w_transposed, out_layout, bias=None, fir=None, out=None, l_range=None):
    """OUT[pos][n] = sum_k ACT[pos][k] Wl[n][k] (+ bias) on this library's tcgen05 kernel (csrc/proj_gemm.cuh, 3xTF32).
    act_layout 0: act (B, L, K); 1: act (B, K, L).  out_layout 0: (B, N, L); 1: (B, L, N).  Wl = W.T if w_transposed."""
    _need_cuda(act, W, bias, fir)
    if act.dim() != 3 or W.dim() != 2 or not act.is_contiguous() or not W.is_contiguous():
        raise _lib.HyenaB200Error("proj_gemm: act must be contiguous 3-D, W contiguous 2-D")
    B = act.shape[0]
    L, K = (act.shape[1], act.shape[2]) if act_layout == 0 else (act.shape[2], act.shape[1])
    N = W.shape[1] if w_transposed else W.shape[0]
    if (W.shape[0] if w_transposed else W.shape[1]) != K:
        raise _lib.HyenaB200Error(f"proj_gemm: weight {tuple(W.shape)} does not match K = {K}")
    dev = act.device
    oshape = (B, N, L) if out_layout == 0 else (B, L, N)
    if out is None:
        out = torch.empty(oshape, dtype=torch.float32, device=dev)
    elif tuple(out.shape) != oshape or not out.is_contiguous() or out.dtype != torch.float32:
        raise _lib.HyenaB200Error(f"proj_gemm: out must be contiguous fp32 {oshape}")
    l0, ln = (0, 0) if l_range is None else (int(l_range[0]), int(l_range[1] - l_range[0]))
    need = int(_lib.lib().hyena_b200_proj_wimg_bytes(N, K))
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), _stream())
    wimg = _wimg_cache.get(key)
    if wimg is None or wimg.numel() < need:
        wimg = torch.empty(max(need, 4 << 20), dtype=torch.uint8, device=dev)
        _wimg_cache[key] = wimg
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().hyena_b200_proj_gemm(
            _ptr(act), int(act_layout), _ptr(W), W.shape[1], int(bool(w_transposed)), _ptr(bias), _ptr(fir), _ptr(out),
            int(out_layout), B, L, K, N, l0, ln, _ptr(wimg), wimg.numel(), _stream()))
    return out


_wgrad_cache = {}


def proj_wgrad(X, Y, fir=None, transposed_out=False):
    """dW (M, N) [(N, M) if transposed_out] = sum_{b,pos} X[b][m][pos] Y[b][pos][n]; X (B, M, L), Y (B, L, N)
    (csrc/proj_gemm.cuh wgrad_kernel: tcgen05 3xTF32, split-K, deterministic)."""
    _need_cuda(X, Y, fir)
    if X.dim() != 3 or Y.dim() != 3 or not X.is_contiguous() or not Y.is_contiguous() or X.shape[0] != Y.shape[0] \
            or X.shape[2] != Y.shape[1]:
        raise _lib.HyenaB200Error(f"proj_wgrad: X (B, M, L) / Y (B, L, N) expected, got {tuple(X.shape)} / {tuple(Y.shape)}")
    B, M, L = X.shape
    N = Y.shape[2]
    dev = X.device
    dW = torch.empty((N, M) if transposed_out else (M, N), dtype=torch.float32, device=dev)
    need = int(_lib.lib().hyena_b200_proj_wgrad_scratch_bytes(M, N))
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), _stream())
    sc = _wgrad_cache.get(key)
    if sc is None or sc.numel() < need:
        sc = torch.empty(need, dtype=torch.uint8, device=dev)
        _wgrad_cache[key] = sc
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().hyena_b200_proj_wgrad(_ptr(X), _ptr(Y), _ptr(fir), _ptr(dW), int(bool(transposed_out)), 0.0,
                                                    B, L, M, N, _ptr(sc), sc.numel(), _stream()))
    return dW


# ------------------------------------------------------------------------------------------ block glue: add + LayerNorm
_ln_scratch = {}


class AddLayerNormFn(torch.autograd.Function):
    """(y, res_out) = (LayerNorm(x + res) * w + b, x + res) in one pass over HBM (csrc/layernorm.cuh), fp32.

    The pre-norm step of the Block that wraps the mixer (flash-attention/flash_attn/modules/block.py:111-148; with
    fused_dropout_add_ln it is flash_attn.ops.layer_norm.dropout_add_layer_norm(prenorm=True, residual_in_fp32=True),
    dropout p = 0).  ``res`` may be None (first block): res_out is then a copy of x."""

    @staticmethod
    def forward(ctx, x, res, w, b, eps):
        _need_cuda(x, res, w, b)
        if not x.is_contiguous() or (res is not None and (not res.is_contiguous() or res.shape != x.shape)):
            raise _lib.HyenaB200Error("add_layer_norm: x and res must be contiguous and of the same shape")
        D = x.shape[-1]
        if w.numel() != D or (b is not None and b.numel() != D):
            raise _lib.HyenaB200Error(f"add_layer_norm: weight / bias must have {D} elements")
        rows = x.numel() // D
        y = torch.empty_like(x)
        res_out = torch.empty_like(x)
        mean = torch.empty(rows, dtype=torch.float32, device=x.device)
        rstd = torch.empty(rows, dtype=torch.float32, device=x.device)
        w = w.contiguous()
        b = b.contiguous() if b is not None else None
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().hyena_b200_add_layernorm_fwd(
                _ptr(x), _ptr(res), _ptr(w), _ptr(b), float(eps), _ptr(res_out), _ptr(y),
                _ptr(mean), _ptr(rstd), rows, D, _stream()))
        ctx.save_for_backward(res_out, w, mean, rstd)
        ctx.has_res, ctx.has_b, ctx.D, ctx.rows = res is not None, b is not None, D, rows
        return y, res_out

    @staticmethod
    def backward(ctx, dy, dres):
        r, w, mean, rstd = ctx.saved_tensors
        D, rows = ctx.D, ctx.rows
        dy = dy.contiguous()
        dres = dres.contiguous() if dres is not None else None
        _need_cuda(dy, dres)
        dx = torch.empty_like(r)
        dw = torch.empty(D, dtype=torch.float32, device=r.device)
        db = torch.empty(D, dtype=torch.float32, device=r.device) if ctx.has_b else None
        need = int(_lib.lib().hyena_b200_add_layernorm_scratch_bytes(rows, D))
        key = (r.device.index if r.device.index is not None else torch.cuda.current_device(), _stream())
        sc = _ln_scratch.get(key)
        if sc is None or sc.numel() < need:
            sc = torch.empty(need, dtype=torch.uint8, device=r.device)
            _ln_scratch[key] = sc
        with torch.cuda.device(r.device):
            _lib.check(_lib.lib().hyena_b200_add_layernorm_bwd(
                _ptr(dy), _ptr(dres), _ptr(r), _ptr(w), _ptr(mean), _ptr(rstd), _ptr(dx), _ptr(dw), _ptr(db), rows, D,
                _ptr(sc), sc.numel(), _stream()))
        # the gradient of x and of the incoming residual are the same tensor values
        return dx, (dx if ctx.has_res else None), dw.reshape(w.shape), db, None


def add_layer_norm(x, res, weight, bias, eps):
    return AddLayerNormFn.apply(x, res, weight, bias, eps)
