"""Helpers to load the committed golden fixtures (tests/golden/*.npz)."""
import json
import os

import numpy as np
import torch

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
CASES = ["ref_L64_D8", "ref_L256_D16", "ref_L250_lmax300_D8", "tiny_1k"]      # order = 2
CASES_ORDER3 = ["ref_order3_L256_D16", "ref_order3_L200_D8"]
CASES_OPTIONS = ["ref_norm_modlr_L256_D16"]     # normalized=True, modulation_lr != 0, shift != 0


def load(case):
    z = np.load(os.path.join(GOLDEN_DIR, case + ".npz"))
    B, L, D, E, l_max = [int(x) for x in z["meta"]]
    out = {"B": B, "L": L, "D": D, "E": E, "l_max": l_max, "w": float(z["w"])}
    out["extra"] = json.loads(str(z["extra_json"])) if "extra_json" in z.files else {}
    out["sd"] = {k[3:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("sd/")}
    out["grad"] = {k[5:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("grad/")}
    out["grad64"] = {k[7:]: torch.from_numpy(z[k]) for k in z.files if k.startswith("grad64/")}
    if "u" in z.files:
        out["u"] = torch.from_numpy(z["u"]); out["dy"] = torch.from_numpy(z["dy"])
    else:   # regenerated from the seeds make_golden.py used, verified against stored checksums
        u = torch.randn(B, L, D, generator=torch.Generator().manual_seed(0))
        dy = torch.randn(B, L, D, generator=torch.Generator().manual_seed(1))
        assert abs(float(u.double().sum()) - float(z["u_sum"])) < 1e-6
        assert abs(float(dy.double().sum()) - float(z["dy_sum"])) < 1e-6
        assert torch.equal(u[0, :4, :4], torch.from_numpy(z["u_head"]))
        assert torch.equal(dy[0, :4, :4], torch.from_numpy(z["dy_head"]))
        out["u"], out["dy"] = u, dy
    for k in ("y", "du", "y64", "du64"):
        if k in z.files:
            out[k] = torch.from_numpy(z[k])
    if "sample_idx" in z.files:     # outputs stored at a fixed sample of their flat indices only
        out["sample_idx"] = torch.from_numpy(z["sample_idx"].astype(np.int64))
    return out


def stored(G, t):
    """The entries of an output tensor (y, du) that fixture G stores: all of them, or its fixed sample."""
    idx = G.get("sample_idx")
    return t if idx is None else t.reshape(-1)[idx.to(t.device)]
