"""Drop-in HyenaOperator / HyenaFilter backed by the sm_100a library.

Mirrors the public surface of /root/reference/src/models/sequence/hyena.py (same class names,
constructor keywords, state_dict keys and shapes, ``_optim`` attributes, ``filter(L)`` /
``forward`` semantics) for the configuration the HyenaDNA models use -- order=2, num_heads=1,
num_blocks=1, inner_factor=1, activation="id", dropout=0 -- and raises a clear error for options
outside that scope instead of silently diverging.  There is no CPU fallback.
"""
import math

import torch
import torch.nn as nn

from . import ops
from ._lib import HyenaB200Error


class OptimModule(nn.Module):
    """register(name, tensor, lr): lr == 0 -> buffer, else Parameter carrying ``_optim`` hyper-parameters
    (src/utils/train.py:142-155)."""

    def register(self, name, tensor, lr=None, wd=0.0):
        if lr == 0.0:
            self.register_buffer(name, tensor)
        else:
            self.register_parameter(name, nn.Parameter(tensor))
            optim = {}
            if lr is not None:
                optim["lr"] = lr
            if wd is not None:
                optim["weight_decay"] = wd
            setattr(getattr(self, name), "_optim", optim)


class Sin(nn.Module):
    """sin(freq * x) with one trainable frequency per feature (hyena.py:96-106).  Kept as a module so
    the state_dict carries ``implicit_filter.{1,3,5}.freq``; evaluated inside the fused filter kernel."""

    def __init__(self, dim, w=10, train_freq=True):
        super().__init__()
        self.freq = nn.Parameter(w * torch.ones(1, dim)) if train_freq else w * torch.ones(1, dim)

    def forward(self, x):
        return torch.sin(self.freq * x)


class PositionalEmbedding(OptimModule):
    """z (1, L, emb_dim) = [t, cos(f w), -sin(f w)], t (1, L, 1) = linspace(0, 1, L)  (hyena.py:109-131)."""

    def __init__(self, emb_dim, seq_len, lr_pos_emb=1e-5, **kwargs):
        super().__init__()
        self.seq_len = seq_len
        t = torch.linspace(0, 1, seq_len)[None, :, None]
        bands = (emb_dim - 1) // 2
        pos = torch.linspace(0, seq_len - 1, seq_len)[None, :, None]
        w = 2 * math.pi * pos / seq_len
        f = torch.linspace(1e-4, bands - 1, bands)[None, None]
        zc = torch.exp(-1j * f * w)
        self.register("z", torch.cat([t, zc.real, zc.imag], dim=-1), lr=lr_pos_emb)
        self.register("t", t, lr=0.0)

    def forward(self, L):
        return self.z[:, :L], self.t[:, :L]


class ExponentialModulation(OptimModule):
    """h * (exp(-t |deltas|) + shift)  (hyena.py:134-155); evaluated inside the fused filter kernel."""

    def __init__(self, d_model, fast_decay_pct=0.3, slow_decay_pct=1.5, target=1e-2, modulation_lr=0.0,
                 shift=0.0, **kwargs):
        super().__init__()
        self.shift = shift
        max_decay = math.log(target) / fast_decay_pct
        min_decay = math.log(target) / slow_decay_pct
        self.register("deltas", torch.linspace(min_decay, max_decay, d_model)[None, None], lr=modulation_lr)

    def forward(self, t, x):
        return x * (torch.exp(-t * self.deltas.abs()) + self.shift)


class HyenaFilter(OptimModule):
    """Implicit long filter (hyena.py:158-267).  ``filter(L)`` -> (1, L, D); ``forward(x, L, k, bias)`` ->
    causal FFT convolution of x (..., D, L) with k plus the bias skip term."""

    def __init__(self, d_model, emb_dim=3, order=16, fused_fft_conv=False, seq_len=1024, lr=1e-3, lr_pos_emb=1e-5,
                 dropout=0.0, w=1, wd=0, bias=True, num_inner_mlps=2, linear_mixer=False, modulate=True,
                 normalized=False, bidirectional=False, **kwargs):
        super().__init__()
        if linear_mixer or num_inner_mlps != 2 or dropout != 0.0:
            raise HyenaB200Error("HyenaFilter: linear_mixer / num_inner_mlps != 2 / "
                                 "dropout are outside the sm_100a hot path (no fallback)")
        if order != 64:
            raise HyenaB200Error(f"HyenaFilter: filter order {order} not supported by the fused kernel (64 only)")
        assert emb_dim % 2 != 0 and emb_dim >= 3, "emb_dim must be odd and greater or equal to 3 (time, sine and cosine)"
        self.d_model, self.emb_dim, self.seq_len, self.modulate = d_model, emb_dim, seq_len, modulate
        self.use_bias = bias
        self.fused_fft_conv = fused_fft_conv      # accepted for config compatibility; the fused path is always on
        self.bias = nn.Parameter(torch.randn(d_model))
        self.dropout = nn.Dropout(dropout)
        self.bidirectional = bidirectional
        self.normalized = normalized

        act = Sin(dim=order, w=w)
        self.pos_emb = PositionalEmbedding(emb_dim, seq_len, lr_pos_emb)
        self.implicit_filter = nn.Sequential(nn.Linear(emb_dim, order), act)
        for _ in range(num_inner_mlps):
            self.implicit_filter.append(nn.Linear(order, order))
            self.implicit_filter.append(act)
        self.implicit_filter.append(nn.Linear(order, d_model, bias=False))
        self.modulation = ExponentialModulation(d_model, **kwargs)
        for c in self.implicit_filter.children():
            for name, _ in c.state_dict().items():
                setattr(getattr(c, name), "_optim", {"weight_decay": wd, "lr": lr})

    def filter_channel_major(self, L):
        """k (D, L): the layout the convolution kernels consume.

        With ``self.cache_filter`` set (see stack.CheckpointedHyenaStack) the generated filter is kept and reused while
        none of the tensors it depends on has changed (torch's per-tensor version counters: an optimizer step or any
        in-place write invalidates it).  Under activation checkpointing every layer's forward runs twice per step
        (long_conv_lm.py:39-45,196-199): the recompute then skips the filter kernels -- at batch 1 they are a third of
        the custom-kernel time of a forward."""
        f = self.implicit_filter
        args = (self.pos_emb.z, self.pos_emb.t, f[0].weight, f[0].bias, f[2].weight, f[2].bias, f[4].weight, f[4].bias,
                f[6].weight, f[1].freq, self.modulation.deltas)
        cached = None
        if getattr(self, "cache_filter", False):
            key = (int(L), float(self.modulation.shift), bool(self.modulate)) + tuple((a.data_ptr(), a._version) for a in args)
            c = getattr(self, "_filter_cache", None)
            if c is not None and c[0] == key:
                cached = c[1]
        k = ops.HyenaFilterFn.apply(*args, float(self.modulation.shift), bool(self.modulate), int(L), cached)
        if getattr(self, "cache_filter", False) and cached is None:
            self._filter_cache = (key, k.detach())
        if self.normalized:                     # hyena.py:235-236: L1 norm over the channels of every position
            k = ops.FilterL1NormFn.apply(k)
        return k

    def filter(self, L, *args, **kwargs):
        return self.filter_channel_major(L).transpose(0, 1).unsqueeze(0)

    def forward(self, x, L, k=None, bias=None, *args, **kwargs):
        from .fftconv import fftconv_func, fftconv_ref
        if self.bidirectional:                 # hyena.py:261: fftconv_ref(..., bidirectional=self.bidirectional)
            if k is None:
                k = self.filter_channel_major(L)
            else:
                k = k[0] if type(k) is tuple else k
                if k.dim() == 3:
                    k = k[0].transpose(0, 1)
            b = self.bias if bias is None else bias
            b = b if self.use_bias else 0 * b
            if x.dim() == 5:
                bb, h, v, zz, l = x.shape
                x3 = x.permute(0, 3, 1, 2, 4).reshape(bb * zz, h * v, l)
                y = fftconv_ref(x3, k, b.reshape(-1), None, gelu=False, bidirectional=True)
                return y.reshape(bb, zz, h, v, l).permute(0, 2, 3, 1, 4).to(dtype=x.dtype)
            return fftconv_ref(x, k, b.reshape(-1), None, gelu=False, bidirectional=True)
        if k is None:
            k = self.filter_channel_major(L)
        else:
            k = k[0] if type(k) is tuple else k
            if k.dim() == 3:
                k = k[0].transpose(0, 1)
        if bias is None:
            bias = self.bias
        bias = bias if self.use_bias else 0 * bias
        bias = bias.reshape(-1).to(torch.float32)
        if x.dim() == 5:        # the reference operator's layout (b, heads, v, blocks, l)  (hyena.py:396-402, :423)
            b, h, v, z, l = x.shape
            x3 = x.permute(0, 3, 1, 2, 4).reshape(b * z, h * v, l)
            y = fftconv_func(x3.to(torch.float32), k, bias, gelu=False)
            return y.reshape(b, z, h, v, l).permute(0, 2, 3, 1, 4).to(dtype=x.dtype)
        shape = x.shape
        y = fftconv_func(x.reshape(-1, shape[-2], shape[-1]).to(torch.float32), k, bias, gelu=False)
        return y.reshape(shape).to(dtype=x.dtype)


class _InProj(torch.autograd.Function):
    """p = W u^T written channel-major (B, 3D, L) straight from the GEMM: no transpose pass
    (replaces hyena.py:391-392).  The bias is added inside the fused kernels."""

    @staticmethod
    def forward(ctx, u, W):
        u = u.contiguous(); W = W.contiguous()
        ctx.save_for_backward(u, W)
        B, L, D = u.shape
        C3 = W.shape[0]
        if ops.proj_mode() == "tc":
            return ops.proj_gemm(u, 0, W, False, 0)                       # p (B, 3D, L) = W u^T, channel-major
        p = torch.empty(B, C3, L, dtype=torch.float32, device=u.device)
        # col-major: P^T (L x 3D, ld L) = U (L x D) W^T (D x 3D);  U stored (D x L, ld D) -> op T
        ops.gemm(1, 0, L, C3, D, u, D, L * D, W, D, 0, p, L, C3 * L, batch=B)
        return p

    @staticmethod
    def backward(ctx, dp):
        u, W = ctx.saved_tensors
        B, L, D = u.shape
        C3 = W.shape[0]
        dp = dp.contiguous()
        if ops.proj_mode() == "tc":
            du = ops.proj_gemm(dp, 1, W, True, 1) if ctx.needs_input_grad[0] else None      # du = dp^T W
            dW = ops.proj_wgrad(dp, u) if ctx.needs_input_grad[1] else None                 # dW = sum dp u
            return du, dW
        du = dW = None
        if ctx.needs_input_grad[1]:
            dW = torch.empty_like(W)
            # dW^T (D x 3D, ld D) = sum_b U_b^T (D x L, stored, op N) dP_b^T (L x 3D, stored ld L, op N)
            for b in range(B):
                ops.gemm(0, 0, D, C3, L, u[b], D, 0, dp[b], L, 0, dW, D, 0, batch=1, beta=0.0 if b == 0 else 1.0)
        if ctx.needs_input_grad[0]:
            du = torch.empty_like(u)
            # dU^T (D x L, ld D) = W^T (D x 3D, stored ld D, op N) dP (3D x L; stored (L x 3D, ld L) -> op T)
            ops.gemm(0, 1, D, L, C3, W, D, 0, dp, L, C3 * L, du, D, L * D, batch=B)
        return du, dW


class _OutProj(torch.autograd.Function):
    """y = y_pre^T W^T + b consuming channel-major y_pre (B, D, L) (replaces hyena.py:432-440)."""

    @staticmethod
    def forward(ctx, y_pre, W, b):
        y_pre = y_pre.contiguous(); W = W.contiguous()
        ctx.save_for_backward(y_pre, W)
        ctx.has_bias = b is not None
        B, C, L = y_pre.shape
        Do = W.shape[0]
        if ops.proj_mode() == "tc":
            return ops.proj_gemm(y_pre, 1, W, False, 1, bias=b.contiguous() if b is not None else None)
        y = torch.empty(B, L, Do, dtype=torch.float32, device=y_pre.device)
        # Y^T (Do x L, ld Do) = W (Do x C; stored (C x Do, ld C) -> op T) Ypre (C x L; stored (L x C, ld L) -> op T)
        ops.gemm(1, 1, Do, L, C, W, C, 0, y_pre, L, C * L, y, Do, L * Do, batch=B,
                 bias=b.contiguous() if b is not None else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        y_pre, W = ctx.saved_tensors
        B, C, L = y_pre.shape
        Do = W.shape[0]
        dy = dy.contiguous()
        if ops.proj_mode() == "tc":
            d_pre = ops.proj_gemm(dy, 0, W, True, 0) if ctx.needs_input_grad[0] else None          # (B, C, L) = W^T dy^T
            dW = ops.proj_wgrad(y_pre, dy, transposed_out=True) if ctx.needs_input_grad[1] else None   # (Do, C)
            db = dy.sum((0, 1)) if (ctx.has_bias and ctx.needs_input_grad[2]) else None
            return d_pre, dW, db
        d_pre = dW = db = None
        if ctx.needs_input_grad[1]:
            dW = torch.empty_like(W)
            # dW^T (C x Do, ld C) = sum_b Ypre_b (C x L; stored (L x C, ld L) -> op T) dY_b (L x Do; stored (Do x L) -> op T)
            for b in range(B):
                ops.gemm(1, 1, C, Do, L, y_pre[b], L, 0, dy[b], Do, 0, dW, C, 0, batch=1, beta=0.0 if b == 0 else 1.0)
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = dy.sum((0, 1))
        if ctx.needs_input_grad[0]:
            d_pre = torch.empty_like(y_pre)
            # dYpre^T (L x C, ld L) = dY (L x Do; stored (Do x L, ld Do) -> op T) W (Do x C; stored (C x Do, ld C) -> op T)
            ops.gemm(1, 1, L, C, Do, dy, Do, L * Do, W, C, 0, d_pre, L, C * L, batch=B)
        return d_pre, dW, db


class HyenaInferenceCache:
    """Decode state of one HyenaOperator (see HyenaOperator.allocate_inference_cache), all fp32 on the module's device:
    g_hist (B, D, max_seqlen) gated history, fir (B, 3D, 2) short-filter state, k (D, max_seqlen) filter, fbias (D),
    workspace (bytes), seqlen_offset = the position the next step writes."""

    def __init__(self, g_hist, fir, k, fbias, workspace):
        self.g_hist, self.fir, self.k, self.fbias, self.workspace = g_hist, fir, k, fbias, workspace
        self.batch_size, self.max_seqlen = g_hist.shape[0], g_hist.shape[-1]
        self.seqlen_offset = 0

    def check_batch(self, B):
        if B != self.batch_size:
            raise HyenaB200Error(f"batch {B} does not match the inference cache ({self.batch_size})")


class HyenaOperator(nn.Module):
    """Hyena operator (hyena.py:270-448): order 2 as one fused pass on sm_100a, order >= 3 as a chain of its kernels.

    forward(u: (B, L, D)) -> (B, L, D) (or ``(y, None)`` when return_state).  Unknown keyword arguments
    (layer_idx, device, dtype, ...) fall through to the filter exactly as in the reference."""

    def __init__(self, d_model, l_max, order=2, filter_order=64, num_heads=1, inner_factor=1, num_blocks=1,
                 fused_bias_fc=False, outer_mixing=False, dropout=0.0, filter_dropout=0.0, filter_cls="hyena-filter",
                 post_order_ffn=False, jit_filter=False, short_filter_order=3, activation="id", return_state=False,
                 **filter_args):
        super().__init__()
        unsupported = {"order": order < 2, "num_heads": num_heads != 1, "inner_factor": inner_factor != 1,
                       "num_blocks": num_blocks != 1, "outer_mixing": outer_mixing, "dropout": dropout != 0.0,
                       "filter_dropout": filter_dropout != 0.0, "post_order_ffn": post_order_ffn,
                       "jit_filter": jit_filter, "short_filter_order": short_filter_order != 3,
                       "activation": activation not in ("id", "identity", None),
                       "filter_cls": filter_cls != "hyena-filter", "fused_bias_fc": fused_bias_fc}
        bad = [k for k, v in unsupported.items() if v]
        if bad:
            raise HyenaB200Error(f"HyenaOperator options outside the sm_100a hot path (no fallback): {bad}")
        self.d_model, self.l_max, self.order = d_model, l_max, order
        self.num_heads, self.inner_factor, self.num_blocks = num_heads, inner_factor, num_blocks
        self.block_dim, self.head_dim = l_max // num_blocks, d_model // num_heads
        self.filter_order, self.short_filter_order = filter_order, short_filter_order
        self.post_order_ffn, self.jit_filter, self.outer_mixing = post_order_ffn, jit_filter, outer_mixing
        self.filter_dropout, self.return_state = filter_dropout, return_state
        self.activation = nn.Identity()
        self.dropout = nn.Dropout(dropout)
        self.out_proj = nn.Linear(d_model * inner_factor, d_model)
        self.in_proj = nn.Linear(d_model, (order + 1) * d_model)
        total_width = d_model * inner_factor * (order + 1)
        self.short_filter = nn.Conv1d(total_width, total_width, short_filter_order, groups=total_width,
                                      padding=short_filter_order - 1)
        filter_args.pop("channels", None)
        self.filter_fn = HyenaFilter(self.head_dim * inner_factor * (order - 1), order=filter_order, seq_len=l_max,
                                     channels=1, dropout=filter_dropout, **filter_args)

    def forward(self, u, *args, **kwargs):
        if not u.is_cuda:
            raise HyenaB200Error("HyenaOperator (hyena_b200) runs on CUDA sm_100a only; there is no CPU fallback")
        in_dtype = u.dtype
        u = u.to(torch.float32)
        l = u.size(-2)
        l_filter = min(l, self.l_max)
        k = self.filter_fn.filter_channel_major(l_filter)                           # (D*(order-1), l_filter)
        fb = self.filter_fn.bias if self.filter_fn.use_bias else 0 * self.filter_fn.bias
        kspec = None
        if self.order == 2 and getattr(self.filter_fn, "cache_filter", False):
            # spectrum of the cached filter, kept with it (same invalidation: it is keyed on the cached k tensor)
            c = getattr(self, "_kspec_cache", None)
            kkey = (k.data_ptr(), k._version, tuple(k.shape))
            if c is not None and c[0] == kkey:
                kspec = c[1]
            else:
                kspec = ops.filter_spectrum(k.detach())
                self._kspec_cache = (kkey, kspec)
        if self.order > 2 or self.filter_fn.bidirectional:
            y_pre = self._forward_chained(u, k, fb, l_filter)
        elif ops.proj_mode() == "tc" and l_filter == l:
            # one autograd node: in_proj GEMM + fused core; backward feeds ds straight into the projection GEMMs
            y_pre = ops.HyenaInCoreFn.apply(u, self.in_proj.weight, self.in_proj.bias, self.short_filter.weight,
                                            self.short_filter.bias, k, fb, kspec)
        else:
            p = _InProj.apply(u, self.in_proj.weight)                               # (B, 3D, l)
            if l_filter < l:
                p = p[..., :l_filter].contiguous()
            y_pre = ops.HyenaCoreFn.apply(p, self.in_proj.bias, self.short_filter.weight, self.short_filter.bias, k, fb,
                                          kspec)
        y = _OutProj.apply(y_pre, self.out_proj.weight, self.out_proj.bias).to(in_dtype)
        if self.return_state:
            return y, None
        return y

    # ---------------------------------------------------------------------------------------- incremental decoding
    def allocate_inference_cache(self, batch_size, max_seqlen, dtype=None, **kwargs):
        """Decode state for ``batch_size`` sequences of up to ``max_seqlen`` positions, for ``prefill`` / ``step``.

        The reference has no recurrent mode (hyena.py:384-386).  This one is exact: each step computes the causal
        convolution over the whole stored history.  The state holds the filter k (D, max_seqlen), generated here once,
        and the filter bias, so it is valid only while the parameters are unchanged: allocate a new one after an
        optimizer step or a state_dict load.  The state is fp32 whatever ``dtype`` says."""
        if self.order != 2 or self.filter_fn.bidirectional:
            raise HyenaB200Error("incremental decoding covers the causal order-2 operator only "
                                 f"(order={self.order}, bidirectional={self.filter_fn.bidirectional})")
        max_seqlen, batch_size = int(max_seqlen), int(batch_size)
        lim = min(self.l_max, 1 << 20)
        if not 1 <= max_seqlen <= lim:
            raise HyenaB200Error(f"max_seqlen {max_seqlen} outside [1, {lim}] (l_max = {self.l_max}, library limit 2^20)")
        dev = self.in_proj.weight.device
        if dev.type != "cuda":
            raise HyenaB200Error("HyenaOperator (hyena_b200) runs on CUDA sm_100a only; there is no CPU fallback")
        D = self.d_model
        with torch.no_grad():
            k = self.filter_fn.filter_channel_major(max_seqlen).detach().contiguous()
            fb = self.filter_fn.bias if self.filter_fn.use_bias else torch.zeros_like(self.filter_fn.bias)
            fb = fb.detach().to(torch.float32).contiguous()
        ws = torch.empty(ops.decode_workspace_bytes(batch_size, D, max_seqlen), dtype=torch.uint8, device=dev)
        return HyenaInferenceCache(
            g_hist=torch.zeros(batch_size, D, max_seqlen, dtype=torch.float32, device=dev),
            fir=torch.zeros(batch_size, 3 * D, 2, dtype=torch.float32, device=dev), k=k, fbias=fb, workspace=ws)

    def prefill(self, u, cache):
        """Run the prompt u (B, Lp, D) through the full-sequence kernels and fill ``cache`` from it.  Returns exactly what
        ``forward(u)`` returns; the next ``step`` is position Lp.  Gradients are not tracked."""
        B, Lp, D = u.shape
        cache.check_batch(B)
        if not 1 <= Lp <= cache.max_seqlen:
            raise HyenaB200Error(f"prompt length {Lp} outside [1, max_seqlen = {cache.max_seqlen}]")
        if not u.is_cuda:
            raise HyenaB200Error("HyenaOperator (hyena_b200) runs on CUDA sm_100a only; there is no CPU fallback")
        in_dtype = u.dtype
        with torch.no_grad():
            u = u.to(torch.float32).contiguous()
            k = self.filter_fn.filter_channel_major(Lp)
            fb = self.filter_fn.bias if self.filter_fn.use_bias else 0 * self.filter_fn.bias
            W = self.in_proj.weight.contiguous()
            # the projection and the core of forward(), run apart so that p can also feed the decode state
            p = ops.proj_gemm(u, 0, W, False, 0) if ops.proj_mode() == "tc" else _InProj.apply(u, W)
            y_pre = ops.HyenaCoreFn.apply(p, self.in_proj.bias, self.short_filter.weight, self.short_filter.bias, k, fb)
            ops.decode_prefill(p, self.in_proj.bias, self.short_filter.weight.reshape(3 * D, 3), self.short_filter.bias,
                               cache.g_hist, cache.fir)
            y = _OutProj.apply(y_pre, self.out_proj.weight, self.out_proj.bias).to(in_dtype)
        cache.seqlen_offset = Lp
        return (y, None) if self.return_state else y

    def step(self, u_t, cache):
        """One token u_t (B, 1, D) at position ``cache.seqlen_offset`` -> (B, 1, D) in u_t's dtype; advances the cache.
        Equals, to fp32 rounding, the matching row of ``forward`` over the whole sequence so far.  Gradients are not tracked."""
        B, one, D = u_t.shape
        cache.check_batch(B)
        if one != 1 or D != self.d_model:
            raise HyenaB200Error(f"step takes one token (B, 1, {self.d_model}); got {tuple(u_t.shape)}")
        t = cache.seqlen_offset
        if t >= cache.max_seqlen:
            raise HyenaB200Error(f"inference cache is full: {cache.max_seqlen} positions")
        if not u_t.is_cuda:
            raise HyenaB200Error("HyenaOperator (hyena_b200) runs on CUDA sm_100a only; there is no CPU fallback")
        with torch.no_grad():
            y = ops.decode_step(u_t.reshape(B, D).to(torch.float32).contiguous(), self.in_proj.weight, self.in_proj.bias,
                                self.short_filter.weight.reshape(3 * D, 3), self.short_filter.bias, cache.k, cache.fbias,
                                self.out_proj.weight, self.out_proj.bias, cache.g_hist, cache.fir, t, cache.workspace)
        cache.seqlen_offset = t + 1
        y = y.reshape(B, 1, D).to(u_t.dtype)
        return (y, None) if self.return_state else y

    def _forward_chained(self, u, k, fb, l_filter):
        """order >= 3 (the shipped HyenaDNA layer default is 3, configs/model/layer/hyena_dna.yaml:3): the recurrence of
        hyena.py:414-423 as a chain of this library's long convolutions.  Projections and every FFT convolution
        (forward and backward) run on the sm_100a kernels; the gates and the 3-tap short filter between them are
        plain elementwise / depthwise torch ops here -- the fully fused pass exists for order 2 only."""
        D, O1 = self.d_model, self.order - 1
        from .fftconv import fftconv_func
        p = _InProj.apply(u, self.in_proj.weight)                                   # (B, (order+1) D, l)
        if l_filter < p.shape[-1]:
            p = p[..., :l_filter]
        p = p + self.in_proj.bias[None, :, None]
        uc = torch.nn.functional.conv1d(p, self.short_filter.weight, self.short_filter.bias,
                                        padding=self.short_filter_order - 1, groups=p.shape[1])[..., :l_filter]
        *x, v = uc.split(D, dim=1)
        kk = k.reshape(D, O1, l_filter)                                             # filter channels are ordered (v o): :408-412
        bb = fb.reshape(D, O1)
        bidir = self.filter_fn.bidirectional
        for o, x_i in enumerate(reversed(x[1:])):
            if bidir:
                from .fftconv import fftconv_ref
                v = fftconv_ref((v * x_i).contiguous(), kk[:, o].contiguous(), bb[:, o].contiguous(), None, gelu=False,
                                bidirectional=True)
            else:
                v = fftconv_func((v * x_i).contiguous(), kk[:, o].contiguous(), bb[:, o].contiguous(), gelu=False)
        return (v * x[0]).contiguous()

    @property
    def d_output(self):
        return self.d_model
