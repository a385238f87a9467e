#!/usr/bin/env python
"""Per-token cost of incremental decoding (HyenaOperator.step) against a full forward, one operator layer.

    python tools/bench_decode.py [--steps 200] [--warmup 20] [--out FILE]

d_model = 256, batch B in {1, 8}, history length t in {2^10, 2^14, 2^17, 2^20}.  For each case:
  step_ms          wall time of one step (CUDA events around --steps consecutive steps at positions t - steps .. t - 1,
                   host overhead of the Python call included)
  kernel_ms        device time of the step's three kernels per step (the library's per-launch event timing, in a
                   separate pass over the same positions)
  bytes            4 D t (B + 1) (the filter k[:, :t] and the B histories g[:, :, :t]) + the in_proj / out_proj weights
  kernel_TBps      bytes / kernel_ms, and its share of the 7.7 TB/s HBM3e data-sheet figure of one B200.  Below 126 MB of
                   bytes (t = 2^10, and 2^14 at B = 1) the data is L2-resident between steps, so the share can exceed 1.
  forward_ms       one no-grad forward of the same operator over t positions: the per-token cost without a decode state
The history values do not change the work, so the cache is positioned at t - steps directly instead of by a prompt.
Prints one JSON line per case and a summary table; the GPU name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

HBM_TBPS = 7.7
L2_BYTES = 126 << 20


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                              "0"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        out = ""
    return {"nvidia_smi": out or None, "torch_name": torch.cuda.get_device_name(0)}


def time_steps(op, u, cache, t0, n):
    cache.seqlen_offset = t0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        op.step(u[:, i:i + 1], cache)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def kernel_ms(op, u, cache, t0, n, lib):
    cache.seqlen_offset = t0
    torch.cuda.synchronize()
    lib.profile_begin()
    for i in range(n):
        op.step(u[:, i:i + 1], cache)
    prof = lib.profile_end()
    kinds = {k: v for k, v in prof.items() if k.startswith("decode_step")}
    assert all(c == n for _, c in kinds.values()), kinds
    return sum(ms for ms, _ in kinds.values()) / n, {k: ms / n for k, (ms, _) in kinds.items()}


def forward_ms(op, x, reps):
    with torch.no_grad():
        op(x)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            op(x)
        e1.record()
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--forward-reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="also write the JSON lines and the table to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_decode.py measures on the GPU; no CUDA device found")
    import hyena_dna_b200 as H
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda:0")
    D, L_MAX = 256, 1 << 20
    n = a.warmup + a.steps
    op = H.HyenaOperator(D, L_MAX, emb_dim=5, w=10.0, lr_pos_emb=0.0).to(dev)
    weights = 4 * (4 * D * D + 5 * D)          # in_proj (3D x D) + out_proj (D x D) + biases
    lines = [json.dumps({"gpu": gpu_info(), "d_model": D, "steps": a.steps, "warmup": a.warmup})]
    print(lines[0], flush=True)
    rows = []
    for B in (1, 8):
        for lg in (10, 14, 17, 20):
            t = 1 << lg
            g = torch.Generator(device=dev).manual_seed(lg)
            cache = op.allocate_inference_cache(B, t)
            cache.g_hist.normal_(generator=g)
            u = torch.randn(B, n, D, device=dev, generator=g)
            t0 = t - n
            time_steps(op, u[:, :a.warmup], cache, t0, a.warmup)
            step = time_steps(op, u[:, a.warmup:], cache, t0 + a.warmup, a.steps)
            kms, split = kernel_ms(op, u[:, a.warmup:], cache, t0 + a.warmup, a.steps, H._lib)
            del cache
            torch.cuda.empty_cache()
            x = torch.randn(B, t, D, device=dev, generator=g)
            fwd = forward_ms(op, x, a.forward_reps)
            del x
            torch.cuda.empty_cache()
            nbytes = 4 * D * t * (B + 1) + weights
            r = {"B": B, "t": t, "step_ms": round(step, 5), "kernel_ms": round(kms, 5),
                 "kernel_split_ms": {k: round(v, 5) for k, v in split.items()}, "bytes": nbytes,
                 "kernel_TBps": round(nbytes / kms / 1e9, 3), "share_of_7.7TBps": round(nbytes / kms / 1e9 / HBM_TBPS, 3),
                 "step_TBps": round(nbytes / step / 1e9, 3), "l2_resident": nbytes < L2_BYTES,
                 "forward_ms": round(fwd, 3), "speedup_vs_forward": round(fwd / step, 1)}
            rows.append(r)
            lines.append(json.dumps(r))
            print(lines[-1], flush=True)
    table = ["", f"{'B':>2} {'t':>8} {'step ms':>9} {'kernel ms':>10} {'TB/s':>6} {'of 7.7':>6} {'fwd ms':>9} {'fwd/step':>9}"]
    for r in rows:
        table.append(f"{r['B']:>2} {r['t']:>8} {r['step_ms']:>9.4f} {r['kernel_ms']:>10.4f} {r['kernel_TBps']:>6.2f} "
                     f"{r['share_of_7.7TBps']:>6.2f} {r['forward_ms']:>9.3f} {r['speedup_vs_forward']:>9.1f}"
                     + ("  (L2-resident)" if r["l2_resident"] else ""))
    print("\n".join(table))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write("\n".join(lines + table) + "\n")


if __name__ == "__main__":
    main()
