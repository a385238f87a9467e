"""Generate golden vectors from the UNMODIFIED reference code (run in the build container only).

    python tests/golden/make_golden.py

Imports /root/reference/standalone_hyenadna.py as-is and /root/reference/src/models/sequence/hyena.py
behind four import shims (hydra, omegaconf, pytorch_lightning, opt_einsum are absent here; none of
them is touched by the hot path).  Writes tests/golden/*.npz: reference state_dict, input u,
upstream grad dy, reference output y, reference input grad du and parameter grads, plus the
float64 "truth" output of the same module (.double()).  /root/reference does not exist on the
GPU box, so these files are what the tests there compare against.
"""
import copy
import os
import sys
import types

import numpy as np
import torch

REF = "/root/reference"
OUT = os.path.dirname(os.path.abspath(__file__))

CASES = {
    # name: (B, L, D, emb_dim, w, l_max, init_std)
    "ref_L64_D8":     (2, 64, 8, 3, 1.0, 64, None),
    "ref_L256_D16":   (2, 256, 16, 5, 10.0, 256, 0.02),
    "ref_L250_lmax300_D8": (1, 250, 8, 5, 10.0, 300, None),   # L < l_max, L not a power of two
    "tiny_1k":        (2, 1024, 128, 5, 10.0, 1024, 0.02),   # BASELINE.json configs[0]
    # order = 3: the shipped HyenaDNA layer default (configs/model/layer/hyena_dna.yaml:3), two chained recurrences
    "ref_order3_L256_D16": (2, 256, 16, 5, 10.0, 256, 0.02, 3),
    "ref_order3_L200_D8":  (1, 200, 8, 5, 10.0, 256, None, 3),
    # filter options outside the shipped configs: L1-normalised filter (hyena.py:235-236) and trainable modulation deltas
    # (modulation_lr != 0, hyena.py:145-150), with a non-zero shift
    "ref_norm_modlr_L256_D16": (2, 256, 16, 5, 10.0, 256, 0.02, 2, {"normalized": True, "modulation_lr": 1e-3, "shift": 0.05}),
}
TINY_SAMPLE = 8192      # stored entries of tiny_1k's y and du (of 2 * 1024 * 128 each)


def _shim():
    def mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m
    def get_method(path):
        import importlib
        m, _, attr = path.rpartition(".")
        return getattr(importlib.import_module(m), attr)
    hy = mod("hydra"); hy.utils = mod("hydra.utils", get_method=get_method)
    class _Cfg(dict): pass
    mod("omegaconf", DictConfig=_Cfg, ListConfig=list, OmegaConf=types.SimpleNamespace(to_container=lambda c, **k: c))
    pl = mod("pytorch_lightning"); pl.utilities = mod("pytorch_lightning.utilities", rank_zero_only=lambda f: f)
    mod("opt_einsum", contract=torch.einsum)


def build(case, which):
    B, L, D, E, w, l_max, init_std = CASES[case][:7]
    order = CASES[case][7] if len(CASES[case]) > 7 else 2
    extra = dict(CASES[case][8]) if len(CASES[case]) > 8 else {}
    torch.manual_seed(1234)
    if which == "standalone":
        import standalone_hyenadna as S
        kw = {"shift": 0.0}
        kw.update(extra)
        op = S.HyenaOperator(D, l_max, order=order, filter_order=64, emb_dim=E, w=w, lr_pos_emb=0.0, **kw)
        init = S._init_weights
    else:
        from src.models.sequence.hyena import HyenaOperator
        op = HyenaOperator(D, l_max, order=order, filter_order=64, emb_dim=E, w=w, lr_pos_emb=0.0,
                           layer_idx=0, device=None, dtype=None, **extra)
        import standalone_hyenadna as S
        init = S._init_weights
    if init_std is not None:
        from functools import partial
        op.apply(partial(init, n_layer=8, initializer_range=init_std))
    return op


def main():
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.set_num_threads(8)
    sys.path.insert(0, REF)
    _shim()
    only = sys.argv[1:]
    for case, spec in CASES.items():
        if only and case not in only:
            continue
        B, L, D, E, w, l_max, init_std = spec[:7]
        order = spec[7] if len(spec) > 7 else 2
        op = build(case, "standalone")
        op_src = build(case, "src")
        op_src.load_state_dict(op.state_dict())
        if order > 2 or len(spec) > 8:
            # (options case: standalone_hyenadna.py's filter ignores `normalized` (:192-214), the src module implements it)
            # the two copies of the operator in the reference disagree beyond order 2: standalone_hyenadna.py:283-284
            # orders the filter channels '(o d)', src/models/sequence/hyena.py:408-412 '(v o)'.  The drop-in target is
            # the src module (SURVEY.md S8a), so the fixture comes from it.
            op, op_src = op_src, None
        g = torch.Generator().manual_seed(0)
        u = torch.randn(B, L, D, generator=g)
        dy = torch.randn(B, L, D, generator=torch.Generator().manual_seed(1))
        u1 = u.clone().requires_grad_(True)
        y = op(u1)
        y.backward(dy)
        if op_src is not None:
            y_src = op_src(u)
            assert torch.equal(y, y_src), "standalone and src/ HyenaOperator disagree"
        op64 = copy.deepcopy(op).double()
        op64.zero_grad()
        u64 = u.double().requires_grad_(True)
        y64 = op64(u64)
        y64.backward(dy.double())
        out = {"u": u.numpy(), "dy": dy.numpy(), "y": y.detach().numpy(), "du": u1.grad.numpy(),
               "y64": y64.detach().numpy(), "du64": u64.grad.numpy(),
               "meta": np.array([B, L, D, E, l_max], dtype=np.int64), "w": np.float64(w), "order": np.int64(order)}
        if len(spec) > 8:
            import json
            out["extra_json"] = np.array(json.dumps(spec[8]))
        for k, v in op.state_dict().items():
            out["sd/" + k] = v.numpy()
        for k, p in op.named_parameters():
            out["grad/" + k] = p.grad.numpy()
        for k, p in op64.named_parameters():
            out["grad64/" + k] = p.grad.numpy()
        if case == "tiny_1k":
            # keep the fixture small (under 1 MB): u / dy are regenerated from their seeds by the tests
            # (checked against the checksums stored here); y / du are kept at a fixed seeded sample of
            # TINY_SAMPLE flat indices (sample_idx); fp64 truth kept for the filter grads only
            out["u_sum"] = np.float64(u.double().sum()); out["dy_sum"] = np.float64(dy.double().sum())
            out["u_head"] = u[0, :4, :4].numpy(); out["dy_head"] = dy[0, :4, :4].numpy()
            idx = np.sort(np.random.default_rng(0).choice(out["y"].size, TINY_SAMPLE, replace=False)).astype(np.int32)
            out["sample_idx"] = idx
            out["y"], out["du"] = out["y"].reshape(-1)[idx], out["du"].reshape(-1)[idx]
            for k in ("u", "dy", "y64", "du64"):
                del out[k]
            for k in list(out):
                if k.startswith("grad64/") and "implicit_filter" not in k and "filter_fn.bias" not in k:
                    del out[k]
        path = os.path.join(OUT, case + ".npz")
        np.savez_compressed(path, **out)
        print(case, "->", path, os.path.getsize(path) // 1024, "KiB",
              "max|y-y64|", float((y.detach().double() - y64.detach()).abs().max()))


if __name__ == "__main__":
    main()
