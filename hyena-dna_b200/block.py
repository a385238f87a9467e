"""Block glue either side of the mixer (SURVEY.md S8 f1): the pre-norm residual Block of the HyenaDNA backbone.

Mirrors flash-attention/flash_attn/modules/block.py:36-200 for the configuration src/models/sequence/long_conv_lm.py
uses (create_block :139-200: prenorm=True, residual_in_fp32, fused_dropout_add_ln optional; LMBackbone.forward :377-396
threads (hidden_states, residual) through the blocks and applies the same dropout -> add -> LayerNorm once more at the
end): same constructor keywords, attribute names (mixer, norm1, mlp, norm2, dropout1/2) and state_dict keys, so a
reference checkpoint's ``backbone.layers.N.*`` entries load unchanged.

The dropout -> add -> LayerNorm step runs as ONE sm_100a kernel (csrc/layernorm.cuh) in fp32 -- the residual stream is
kept in fp32 whatever the activation dtype, i.e. residual_in_fp32 semantics.  Dropout / stochastic depth with p > 0,
post-norm blocks and RMSNorm are outside the hot path and raise; there is no CPU fallback.
"""
import torch
import torch.nn as nn

from . import ops
from ._lib import HyenaB200Error


class Block(nn.Module):
    def __init__(self, dim, mixer_cls=None, mlp_cls=None, norm_cls=nn.LayerNorm, dropout_cls=nn.Dropout, prenorm=True,
                 resid_dropout1=0.0, resid_dropout2=0.0, drop_path1=0.0, drop_path2=0.0, fused_dropout_add_ln=False,
                 return_residual=False, residual_in_fp32=False, sequence_parallel=False, mark_shared_params=False):
        super().__init__()
        bad = {"prenorm": not prenorm, "resid_dropout1": resid_dropout1 != 0.0, "resid_dropout2": resid_dropout2 != 0.0,
               "drop_path1": drop_path1 != 0.0, "drop_path2": drop_path2 != 0.0, "return_residual": return_residual,
               "sequence_parallel": sequence_parallel, "mixer_cls": mixer_cls is None}
        bad = [k for k, v in bad.items() if v]
        if bad:
            raise HyenaB200Error(f"Block options outside the sm_100a hot path (no fallback): {bad}")
        self.prenorm = prenorm
        self.fused_dropout_add_ln = fused_dropout_add_ln      # accepted for config compatibility: the fused kernel always runs
        self.return_residual = return_residual
        self.residual_in_fp32 = residual_in_fp32
        self.mixer = mixer_cls(dim)
        self.dropout1 = dropout_cls(resid_dropout1)
        self.norm1 = norm_cls(dim)
        self.mlp = mlp_cls(dim) if mlp_cls is not None else nn.Identity()
        if not isinstance(self.mlp, nn.Identity):
            self.dropout2 = dropout_cls(resid_dropout2)
            self.norm2 = norm_cls(dim)
        for n in (self.norm1, getattr(self, "norm2", None)):
            if n is not None and not isinstance(n, nn.LayerNorm):
                raise HyenaB200Error("Block: only nn.LayerNorm is supported by the fused add + norm kernel")
        if mark_shared_params:
            for p in list(self.norm1.parameters()) + (list(self.norm2.parameters()) if hasattr(self, "norm2") else []):
                p._shared_params = True

    @staticmethod
    def _add_norm(hidden_states, residual, norm):
        if not hidden_states.is_cuda:
            raise HyenaB200Error("Block (hyena_b200) runs on CUDA sm_100a only; there is no CPU fallback")
        x = hidden_states.to(torch.float32).contiguous()
        r = residual.to(torch.float32).contiguous() if residual is not None else None
        return ops.add_layer_norm(x, r, norm.weight.to(torch.float32), norm.bias.to(torch.float32) if norm.bias is not None
                                  else None, norm.eps)

    def forward(self, hidden_states, residual=None, mixer_subset=None, mixer_kwargs=None):
        """(hidden_states, residual) -> (mlp(LN2(.)) or mixer output, new residual); block.py:111-180, prenorm branch."""
        if mixer_subset is not None:
            raise HyenaB200Error("Block: mixer_subset is not supported")
        return self._run(hidden_states, residual, lambda y: self.mixer(y, **(mixer_kwargs or {})))

    def allocate_inference_cache(self, batch_size, max_seqlen, dtype=None, **kwargs):
        """The mixer's decode state (HyenaOperator.allocate_inference_cache)."""
        return self.mixer.allocate_inference_cache(batch_size, max_seqlen, dtype=dtype, **kwargs)

    def prefill(self, hidden_states, residual, cache):
        """forward() over a prompt (B, Lp, D) that also fills the mixer's decode state ``cache``."""
        fn = self._mixer_fn("prefill")
        return self._run(hidden_states, residual, lambda y: fn(y, cache))

    def step(self, hidden_states, residual, cache):
        """forward() for one token (B, 1, D) at the cache's position, using and advancing the mixer's decode state."""
        fn = self._mixer_fn("step")
        return self._run(hidden_states, residual, lambda y: fn(y, cache))

    def _mixer_fn(self, name):
        fn = getattr(self.mixer, name, None)
        if fn is None:
            raise HyenaB200Error(f"Block: the mixer {type(self.mixer).__name__} has no incremental decoding ({name})")
        return fn

    def _run(self, hidden_states, residual, mix):
        in_dtype = hidden_states.dtype
        y, residual = self._add_norm(hidden_states, residual, self.norm1)
        hidden_states = mix(y.to(in_dtype))
        if isinstance(hidden_states, tuple):                # mixers built with return_state
            hidden_states = hidden_states[0]
        if not isinstance(self.mlp, nn.Identity):
            y, residual = self._add_norm(hidden_states, residual, self.norm2)
            hidden_states = self.mlp(y.to(in_dtype))
        if not self.residual_in_fp32:
            residual = residual.to(in_dtype)
        return hidden_states, residual


class Backbone(nn.Module):
    """Stack of Blocks + the final dropout -> add -> LayerNorm (LMBackbone without the embedding: long_conv_lm.py:377-396).
    Attribute names follow the reference (``layers``, ``ln_f``) so that its state_dict keys map one to one."""

    def __init__(self, d_model, n_layer, mixer_cls, mlp_cls=None, layer_norm_epsilon=1e-5, residual_in_fp32=False):
        super().__init__()
        self.residual_in_fp32 = residual_in_fp32
        self.layers = nn.ModuleList([
            Block(d_model, mixer_cls=mixer_cls, mlp_cls=mlp_cls, norm_cls=lambda d: nn.LayerNorm(d, eps=layer_norm_epsilon),
                  prenorm=True, residual_in_fp32=residual_in_fp32) for _ in range(n_layer)])
        self.ln_f = nn.LayerNorm(d_model, eps=layer_norm_epsilon)

    def forward(self, hidden_states):
        residual = None
        for layer in self.layers:
            hidden_states, residual = layer(hidden_states, residual)
        y, _ = Block._add_norm(hidden_states, residual, self.ln_f)
        return y.to(hidden_states.dtype)

    def allocate_inference_cache(self, batch_size, max_seqlen, dtype=None, **kwargs):
        """{layer index: decode state} for ``prefill`` / ``step``, keyed like flash_attn's InferenceParams memory dict."""
        return {i: layer.allocate_inference_cache(batch_size, max_seqlen, dtype=dtype, **kwargs)
                for i, layer in enumerate(self.layers)}

    def prefill(self, hidden_states, caches):
        """forward() over a prompt (B, Lp, D) that also fills every layer's decode state."""
        residual = None
        for i, layer in enumerate(self.layers):
            hidden_states, residual = layer.prefill(hidden_states, residual, caches[i])
        y, _ = Block._add_norm(hidden_states, residual, self.ln_f)
        return y.to(hidden_states.dtype)

    def step(self, hidden_states, caches):
        """forward() for one token (B, 1, D) at the caches' position; advances every layer's decode state."""
        residual = None
        for i, layer in enumerate(self.layers):
            hidden_states, residual = layer.step(hidden_states, residual, caches[i])
        y, _ = Block._add_norm(hidden_states, residual, self.ln_f)
        return y.to(hidden_states.dtype)
