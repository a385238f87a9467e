"""CPU checks of bench.py's pure logic (roofline assembly, algorithmic byte counts, argument defaults)."""
import importlib.util
import json
import os

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_span_bytes_match_survey_formula():
    b = _bench()
    r = b.build_roofline({"row_pass<conv_bwd>": (40.0, 10), "col_fwd<gate>": (12.5, 10)}, 10, 1, 256, 1 << 20, 39.0)
    assert r["algorithmic_bytes_per_step"] == (44 + 16) * 256 * (1 << 20)          # 15,360 B/nt (SURVEY.md S8(d))
    assert abs(r["span_ms_per_step"] - 5.25) < 1e-9
    assert r["dominant_kernel"]["name"] == "row_pass<conv_bwd>"
    assert abs(sum(k["share_of_span"] for k in r["kernels"].values()) - 1.0) < 1e-3
    k = r["kernels"]["col_fwd<gate>"]
    assert k["algorithmic_bytes_per_step"] == 8 * 256 * (1 << 20)
    assert abs(k["achieved_gbs"] - 8 * 256 * (1 << 20) / 1.25e-3 / 1e9) < 0.1
    assert 0 < r["frac"] == round(r["achieved"] / r["peak"], 4)
    json.dumps(r)                                                                   # serialisable


def test_roofline_handles_unknown_and_empty_profiles():
    b = _bench()
    r = b.build_roofline({}, 5, 2, 128, 4096, 1.0)
    assert r["dominant_kernel"] is None and r["achieved"] == 0.0 and r["traffic"] is None
    r = b.build_roofline({"twiddle_init": (0.01, 1)}, 1, 1, 8, 1024, 1.0)
    assert "achieved_gbs" not in r["kernels"]["twiddle_init"]


def test_dump_outputs_writes_whole_or_seeded_samples_within_budget(tmp_path):
    import numpy as np
    import torch
    b = _bench()
    b.DUMP_BYTES = 3 * 4 * 1000                     # 1000 float32 elements per output
    g = torch.Generator().manual_seed(0)
    outs = {"y": torch.randn(2, 50, 40, generator=g), "du": torch.randn(2, 50, 40, generator=g),
            "grad.w": torch.randn(30, 20, generator=g)}
    for d in ("a", "b"):
        b.dump_outputs(str(tmp_path / d), outs)
    total = 0
    for name, t in outs.items():
        a = np.load(tmp_path / "a" / (name + ".npy"))
        assert a.dtype == np.float32 and np.array_equal(a, np.load(tmp_path / "b" / (name + ".npy")))
        total += a.nbytes
        if name == "grad.w":
            assert np.array_equal(a, t.numpy())                     # fits its share: written whole
        else:
            assert a.ndim == 1 and 800 < a.size <= 1000                # 1000 draws of 4000 indices, duplicates dropped
            assert np.isin(a, t.numpy().reshape(-1)).all()          # entries of the output, not something else
    assert total <= b.DUMP_BYTES
    assert np.array_equal(np.isin(outs["y"].numpy().reshape(-1), np.load(tmp_path / "a" / "y.npy")),
                          np.isin(outs["du"].numpy().reshape(-1), np.load(tmp_path / "a" / "du.npy")))   # same indices


def test_synthetic_inputs_match_the_oracle_recipe():
    import torch
    from oracle import hyena_oracle as O
    b = _bench()
    a = b.nucleotide_activations(2, 100, 16, seed=7)
    ref, ids = O.nucleotide_activations(2, 100, 16, seed=7)
    assert torch.equal(a, ref) and int(ids.min()) >= 7 and int(ids.max()) <= 10
