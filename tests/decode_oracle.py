"""TEST INFRASTRUCTURE ONLY -- token-by-token restatement of the order-2 HyenaOperator, the way a cached-state decoder
computes it.  Built from the pieces of oracle/hyena_oracle.py (filter, short filter, full forward); citations are
relative to the reference repository (src/models/sequence/hyena.py)."""
import torch
import torch.nn.functional as F

from oracle.hyena_oracle import hyena_filter, hyena_operator, short_filter


def hyena_operator_decode(u, P, prompt_len, shift=0.0, modulate=True, normalized=False, prompt_outputs=True):
    """Positions [0, prompt_len) form the prompt: their gated history is built in one go, and their outputs (when
    prompt_outputs) are hyena_operator's.  Every later position t is then computed from the stored state alone, with
    direct sums (no FFT):
      p_t = W_in u_t + b_in                                                            hyena.py:391
      s_t = w0 p_{t-2} + w1 p_{t-1} + w2 p_t + sb, p_{<0} = 0 (padding after the bias)  :363-369, :394
      x0, x1, v = split(s_t);  g_t = v x1                                               :404, :420
      c_t = sum_{j=0..t} k[:, j] g_{t-j} + fbias g_t                                    :423 via :261, :59-88
      y_t = W_out (c_t x0) + b_out                                                      :432-440
    u (B, L, D) -> y (B, L, D), or (B, L - prompt_len, D) without prompt_outputs.  fp32 or fp64, any device."""
    B, L, D = u.shape
    assert P["in_proj.weight"].shape[0] == 3 * D, "order 2 only"
    Lp = int(prompt_len)
    W_in, b_in = P["in_proj.weight"], P["in_proj.bias"]
    sw, sb = P["short_filter.weight"][:, 0, :], P["short_filter.bias"]
    k = hyena_filter(L, P, shift, modulate, normalized)[0].transpose(0, 1)            # (D, L), :405-408
    fb = P["filter_fn.bias"]
    g_hist = torch.zeros(B, D, L, dtype=u.dtype, device=u.device)
    fir = torch.zeros(B, 3 * D, 2, dtype=u.dtype, device=u.device)                   # p_{t-2}, p_{t-1}
    ys = []
    if Lp > 0:
        p = F.linear(u[:, :Lp], W_in, b_in).transpose(1, 2)                           # (B, 3D, Lp)
        x0, x1, v = short_filter(p, P["short_filter.weight"], sb, Lp).split(D, dim=1)
        g_hist[:, :, :Lp] = v * x1
        fir[:, :, 2 - min(Lp, 2):] = p[:, :, -min(Lp, 2):]
        if prompt_outputs:
            ys.append(hyena_operator(u[:, :Lp], P, shift, modulate, normalized=normalized))
    for t in range(Lp, L):
        p_t = F.linear(u[:, t], W_in, b_in)                                           # (B, 3D)
        s = sw[:, 0] * fir[:, :, 0] + sw[:, 1] * fir[:, :, 1] + sw[:, 2] * p_t + sb
        fir = torch.stack([fir[:, :, 1], p_t], dim=-1)
        x0, x1, v = s.split(D, dim=1)
        g_hist[:, :, t] = v * x1
        c = (k[:, :t + 1].flip(-1) * g_hist[:, :, :t + 1]).sum(-1) + fb * g_hist[:, :, t]
        ys.append(F.linear(c * x0, P["out_proj.weight"], P["out_proj.bias"])[:, None])
    return torch.cat(ys, dim=1) if ys else u.new_zeros(B, 0, D)
