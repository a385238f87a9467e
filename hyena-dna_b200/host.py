"""Host-buffer entry point: one forward + backward of a HyenaOperator with inputs and outputs in pinned HOST
memory, copies pipelined against the compute.

This is what a caller that lives on the host side of PCIe uses (the reference-facing "plugin" call of
bench.py's `e2e` leg): `u` and `dy` come from pinned host tensors, `y`, `du` and all parameter gradients go back
to pinned host tensors.  Same arithmetic as `HyenaOperator.forward` + autograd (tests/test_gpu_parity.py
::test_host_step_matches_autograd), issued by hand so that

  * `u` is uploaded in sequence chunks and each chunk's slice of the in_proj GEMM starts as soon as it lands,
    while the implicit filter (which needs no input) is generated under the first upload,
  * `dy` is uploaded under the forward pass, `y` is downloaded in chunks under the backward pass,
  * `du` is produced first in the projection backward and downloaded in chunks under the weight-gradient GEMMs
    and the filter backward.

Three CUDA streams (compute, host->device, device->host) and events; no host synchronisation inside a step.
"""
import torch

from . import ops
from ._lib import HyenaB200Error


class HostStep:
    def __init__(self, op, batch, seqlen, chunks=4):
        self.tc = ops.proj_mode() == "tc"               # own tcgen05 projections (default) or cuBLASLt slices
        self.op = op
        dev = op.in_proj.weight.device
        self.dev = dev
        B, L, D = batch, seqlen, op.d_model
        if L > op.l_max:
            raise HyenaB200Error("HostStep: sequence longer than l_max")
        self.B, self.L, self.D = B, L, D
        self.nch = chunks
        self.bounds = [(i * L // chunks, (i + 1) * L // chunks) for i in range(chunks)]
        self.h2d = torch.cuda.Stream(device=dev)
        self.d2h = torch.cuda.Stream(device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        self.u = torch.empty(B, L, D, **f32)
        self.dy = torch.empty(B, L, D, **f32)
        self.p = torch.empty(B, 3 * D, L, **f32)
        self.y = torch.empty(B, L, D, **f32)
        self.du = torch.empty(B, L, D, **f32)
        self.d_pre = torch.empty(B, D, L, **f32)
        self.params = [p for p in op.parameters() if p.requires_grad]

    # ------------------------------------------------------------------ GEMM slices (column-major views, see hyena.py)
    def _in_proj_chunk(self, lo, hi):
        B, L, D = self.B, self.L, self.D
        W = self.op.in_proj.weight
        C3 = W.shape[0]
        if self.tc:
            ops.proj_gemm(self.u, 0, W, False, 0, out=self.p, l_range=(lo, hi))
            return
        # P^T[lo:hi] (n x 3D, ld L) = U[lo:hi] (n x D; stored (D x n), ld D -> op T) W^T (D x 3D, stored, op N)
        ops.gemm(1, 0, hi - lo, C3, D, self.u[:, lo:], D, L * D, W, D, 0, self.p[:, :, lo:], L, C3 * L, batch=B)

    def _out_proj_chunk(self, y_pre, lo, hi):
        B, L, D = self.B, self.L, self.D
        W, b = self.op.out_proj.weight, self.op.out_proj.bias
        if self.tc:
            ops.proj_gemm(y_pre, 1, W, False, 1, bias=b, out=self.y, l_range=(lo, hi))
            return
        ops.gemm(1, 1, D, hi - lo, D, W, D, 0, y_pre[:, :, lo:], L, D * L, self.y[:, lo:], D, L * D, batch=B, bias=b)

    def _du_chunk(self, dp, lo, hi):
        B, L, D = self.B, self.L, self.D
        W = self.op.in_proj.weight
        C3 = W.shape[0]
        if self.tc:
            ops.proj_gemm(dp, 1, W, True, 1, out=self.du, l_range=(lo, hi))
            return
        ops.gemm(0, 1, D, hi - lo, C3, W, D, 0, dp[:, :, lo:], L, C3 * L, self.du[:, lo:], D, L * D, batch=B)

    # ------------------------------------------------------------------ one step
    @torch.no_grad()
    def step(self, u_host, dy_host, y_host, du_host, grads_host, reduce_fn=None):
        """u_host, dy_host, y_host, du_host: pinned (B, L, D) fp32; grads_host: list of pinned tensors shaped like
        ``[p for p in op.parameters() if p.requires_grad]`` (same order).  Returns nothing; all results are in the
        host tensors once the current stream has been synchronised.  ``reduce_fn(list_of_device_grads)``, when
        given, runs before the gradients leave the device (data-parallel all-reduce)."""
        op, B, L, D = self.op, self.B, self.L, self.D
        main = torch.cuda.current_stream(self.dev)
        h2d, d2h = self.h2d, self.d2h
        ff = op.filter_fn
        f = ff.implicit_filter
        # ---- uploads: u in chunks, then dy (under the forward pass)
        h2d.wait_stream(main)
        d2h.wait_stream(main)
        ev_u = []
        with torch.cuda.stream(h2d):
            for lo, hi in self.bounds:
                for b in range(B):                                      # contiguous pieces: plain async memcpys
                    self.u[b, lo:hi].copy_(u_host[b, lo:hi], non_blocking=True)
                e = torch.cuda.Event(); e.record(h2d); ev_u.append(e)
            self.dy.copy_(dy_host, non_blocking=True)
            ev_dy = torch.cuda.Event(); ev_dy.record(h2d)
        # ---- forward
        fargs = (ff.pos_emb.z, ff.pos_emb.t, f[0].weight, f[0].bias, f[2].weight, f[2].bias, f[4].weight, f[4].bias,
                 f[6].weight, f[1].freq, ff.modulation.deltas, float(ff.modulation.shift), bool(ff.modulate), L)
        k = ops.filter_forward(*fargs)                                  # needs no input: runs under the first upload
        kspec = ops.filter_spectrum(k)
        for (lo, hi), e in zip(self.bounds, ev_u):
            main.wait_event(e)
            self._in_proj_chunk(lo, hi)
        sw = op.short_filter.weight.reshape(3 * D, -1).contiguous()
        sb = op.short_filter.bias
        fb = ff.bias if ff.use_bias else torch.zeros_like(ff.bias)
        ib = op.in_proj.bias
        y_pre, c, gs = ops.core_forward(self.p, ib, sw, sb, kspec, fb, True)
        for lo, hi in self.bounds:
            self._out_proj_chunk(y_pre, lo, hi)
            e = torch.cuda.Event(); e.record(main)
            with torch.cuda.stream(d2h):
                d2h.wait_event(e)
                for b in range(B):
                    y_host[b, lo:hi].copy_(self.y[b, lo:hi], non_blocking=True)
        # ---- backward
        main.wait_event(ev_dy)
        Wo = op.out_proj.weight
        if self.tc:
            ops.proj_gemm(self.dy, 0, Wo, True, 0, out=self.d_pre)
            dWo = ops.proj_wgrad(y_pre, self.dy, transposed_out=True)
        else:
            # d_pre^T (L x D, ld L) = dY (L x D; stored (D x L) -> op T) Wo (D x D; stored (D x D)^T -> op T)
            ops.gemm(1, 1, L, D, D, self.dy, D, L * D, Wo, D, 0, self.d_pre, L, D * L, batch=B)
            dWo = torch.empty_like(Wo)
            for b in range(B):
                ops.gemm(1, 1, D, D, L, y_pre[b], L, 0, self.dy[b], D, 0, dWo, D, 0, beta=0.0 if b == 0 else 1.0)
        dbo = self.dy.sum((0, 1))
        dp, dk, dsw, dsb, dfb, dib = ops.core_backward(self.d_pre, self.p, ib, sw, sb, kspec, fb, c, gs)
        for lo, hi in self.bounds:                                       # du first, so that it can leave early
            self._du_chunk(dp, lo, hi)
            e = torch.cuda.Event(); e.record(main)
            with torch.cuda.stream(d2h):
                d2h.wait_event(e)
                for b in range(B):
                    du_host[b, lo:hi].copy_(self.du[b, lo:hi], non_blocking=True)
        Wi = op.in_proj.weight
        if self.tc:
            dWi = ops.proj_wgrad(dp, self.u)
        else:
            dWi = torch.empty_like(Wi)
            for b in range(B):
                ops.gemm(0, 0, D, 3 * D, L, self.u[b], D, 0, dp[b], L, 0, dWi, D, 0, beta=0.0 if b == 0 else 1.0)
        need_dz = ff.pos_emb.z.requires_grad
        fgrads, dfreq, dz = ops.filter_backward(*fargs, dk, need_dz)
        # ---- parameter gradients, keyed by parameter identity, then copied out in op.parameters() order
        g = {id(op.in_proj.weight): dWi, id(op.in_proj.bias): dib, id(op.out_proj.weight): dWo,
             id(op.out_proj.bias): dbo, id(op.short_filter.weight): dsw.reshape(op.short_filter.weight.shape),
             id(op.short_filter.bias): dsb, id(ff.bias): dfb if ff.use_bias else torch.zeros_like(dfb),
             id(f[0].weight): fgrads[0], id(f[0].bias): fgrads[1], id(f[2].weight): fgrads[2],
             id(f[2].bias): fgrads[3], id(f[4].weight): fgrads[4], id(f[4].bias): fgrads[5],
             id(f[6].weight): fgrads[6], id(f[1].freq): dfreq.reshape(f[1].freq.shape)}
        missing = [n for n, prm in op.named_parameters() if prm.requires_grad and id(prm) not in g
                   and not (need_dz and prm is ff.pos_emb.z)]
        if missing:     # e.g. modulation deltas registered as a Parameter (modulation_lr != 0)
            raise HyenaB200Error(f"HostStep: no gradient is produced for trainable parameter(s) {missing}")
        if need_dz:
            gz = torch.zeros_like(ff.pos_emb.z)
            gz[0, :L].copy_(dz)
            g[id(ff.pos_emb.z)] = gz
        glist = [g[id(prm)].contiguous() for prm in self.params]
        if reduce_fn is not None:
            reduce_fn(glist)
        for gh, gd in zip(grads_host, glist):
            gh.copy_(gd, non_blocking=True)
        main.wait_stream(d2h)
