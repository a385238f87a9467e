#!/usr/bin/env python
"""bench.py -- nucleotides/s through HyenaOperator fwd+bwd at L=1,048,576, d_model=256 (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's sm_100a path
    python bench.py --steps K --dump-outputs DIR                   # ... and write the last timed step's outputs
    python bench.py --impl reference [--steps K] [--warmup W]      # the reference's CPU torch.fft path

A "step" is one forward + backward of the operator over one batch of synthetic single-nucleotide
activations (B = 1 sample of L tokens per GPU: BASELINE.json configs[3]/[4]; weak scaling, global
batch = N).  With N > 1 the driver launches one rank per GPU under torchrun; ranks are batch-sharded
replicas and the only collective is the all-reduce of the operator's parameter grads (NCCL).

One JSON line on stdout (rank 0).  Keys beyond the base contract:
  roofline      HBM roofline of the custom-kernel span (SURVEY.md S8(d): (44+16/B)*D bytes per
                nucleotide fwd+bwd, in_proj output -> out_proj input), achieved = those bytes / the
                summed CUDA-event time of this library's kernels inside the timed steps; "kernels"
                lists each kernel class' share so it can be checked against profiles/*launches*.csv
  cpu_baseline  the oracle (CPU restatement of the reference torch.fft path) timed on the host cores
                on a bounded sample of the same workload
  e2e           same metric through the public module API with HOST (pinned) buffers: u and dy are
                copied host->device and y, du and all parameter grads device->host inside the timed
                region, copies overlapped with compute on a side stream where the data flow allows
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly one JSON line: keep NCCL's own banner ("NCCL version ...", printed to stdout when the
# environment sets NCCL_DEBUG) on stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

import torch  # noqa: E402

L_FULL, D_MODEL, EMB, W_FREQ = 1 << 20, 256, 5, 10.0
METRIC = "nucleotides/sec through HyenaOperator fwd+bwd at L=1M d=256"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--seqlen", type=int, default=L_FULL, help="override L (debug only; invalidates the number)")
    ap.add_argument("--d-model", type=int, default=D_MODEL)
    ap.add_argument("--batch", type=int, default=1, help="samples per GPU")
    ap.add_argument("--cpu-threads", type=int, default=0,
                    help="host threads for the CPU arm (0 = min(cores, 16): torch CPU ops were ~40x SLOWER with all "
                         "128 hardware threads of the B200 host than the survey box was with 8)")
    ap.add_argument("--cpu-sample-len", type=int, default=1 << 17,
                    help="sequence length of the bounded CPU sample of the product arm's cpu_baseline leg")
    ap.add_argument("--ref-seconds", type=float, default=200.0,
                    help="time budget of the --impl reference arm: it runs the FULL workload (same L, D, batch) and "
                         "times as many of the requested steps as fit in this budget (at least one)")
    ap.add_argument("--no-gpu-reference", action="store_true",
                    help="skip the gpu_reference leg (the reference's torch.fft/cuFFT path timed on the same GPU)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-chunks", type=int, default=4, help="sequence chunks of the HostStep copy pipeline")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write y, du and the parameter grads of the last timed step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ----------------------------------------------------------------------------------------- output dump
DUMP_BYTES = 60 * 10 ** 6        # payload of --dump-outputs in all (npy headers stay well inside 64 MB)


def dump_outputs(outdir, outputs, seed=0):
    """outputs: {name: tensor}.  Writes DIR/<name>.npy (float32, float64 kept).  Each output gets an equal share of
    DUMP_BYTES: one that fits is written whole, a larger one as a 1-D array of its entries at a fixed seeded sample of
    its flat indices (sorted; the same indices for every output of one size), so that two runs with the same arguments
    are comparable array for array."""
    import numpy as np
    os.makedirs(outdir, exist_ok=True)
    for name, t in outputs.items():
        t = t.detach()
        share = DUMP_BYTES // len(outputs) // (8 if t.dtype == torch.float64 else 4)      # elements
        if t.numel() > share:
            idx = np.unique(np.random.default_rng(seed).integers(0, t.numel(), share))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        a = t.cpu().numpy()
        np.save(os.path.join(outdir, name + ".npy"), a if a.dtype == np.float64 else a.astype(np.float32))


# ----------------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def mark(self):
        """wall-clock marker: samples between two marks are the ones taken under load"""
        return time.time()

    def stop(self, t_begin=None, t_end=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        import datetime
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 10:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                if t_begin is not None and not (t_begin - 0.05 <= ts <= t_end + 0.05):
                    continue
            except ValueError:
                pass
            f = f[1:]
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for nm, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------- per-kernel algorithmic bytes
def kernel_algorithmic_bytes(B, D, L):
    """Compulsory HBM bytes per step of each kernel class under the current design (DESIGN.md S4: FFT scratch assumed
    on chip, every HBM tensor read or written once per kernel that needs it), fp32.  Keys = hyena_b200_kind_name()."""
    n = float(B) * D * L                 # (position, channel) pairs per step
    f = float(D) * L                     # per-channel (filter-side) pairs
    return {
        "col_fwd<gate>": 8 * n,                          # x1, v rows of p
        "col_fwd<dc>": 8 * n,                            # dy_pre, x0 row of p
        "col_fwd<filter>": 4 * f,                        # k
        "row_pass<filter>": 8 * f,                       # kspec out
        "row_pass<conv_fwd>": 8 * f + 8 * n,             # kspec in, saved g spectrum out
        "row_pass<conv_bwd>": 8 * f + 8 * n,             # kspec in, saved g spectrum in
        "col_inv<conv_fwd>": 12 * n,                     # x0 in; y_pre, c out (the skip term lives in the filter spectrum)
        "col_inv<bwd_dg>": 32 * n,                       # x0,x1,v, dy_pre, c in; ds (3 rows) out
        "col_inv<dk>": 4 * f,                            # dk out
        "short_conv_bwd": 24 * n,                        # ds in, dp out
        "filter_tc_fwd": 4 * f,                          # k out
        "filter_tc_bwd": 8 * f + 7 * 64 * 4.0 * L,       # dk in, dh out, seven (64, L) arrays out
        "filter_tc_red": 4 * f + 7 * 64 * 4.0 * L,       # dh and the seven arrays in
        # pipelined calls (HYENA_B200_PIPE: kernels of different row groups overlap, the call is timed as one record)
        "conv_fwd<pipelined>": 8 * n + 8 * f + 8 * n + 12 * n,
        "conv_bwd<pipelined>": 8 * n + 8 * f + 8 * n + 32 * n + 4 * f,
        "filter_spectrum<pipelined>": 4 * f + 8 * f,
    }


# ----------------------------------------------------------------------------------------- roofline assembly
def build_roofline(prof, steps, B, D, L, ms_step):
    """prof: {kernel class: (summed device ms over `steps` steps, launches)} from hyena_dna_b200._lib.profile_end().
    Pure function (unit-tested on CPU in tests/test_bench_logic.py)."""
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_gbs = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
    span_bytes = (44.0 + 16.0 / B) * D * B * L               # SURVEY.md S8(d), per step
    # the projections are this library's kernels too now (csrc/proj_gemm.cuh) but sit OUTSIDE the span of S8(d)
    # (in_proj output -> out_proj input): reported on their own, against the tensor-core roofline
    proj = {k: v for k, v in prof.items() if k.startswith("proj_")}
    prof = {k: v for k, v in prof.items() if not k.startswith("proj_")}
    tot_ms = sum(v[0] for v in prof.values())
    span_ms = tot_ms / steps
    achieved = span_bytes / (span_ms * 1e-3) / 1e9 if span_ms > 0 else 0.0
    kab = kernel_algorithmic_bytes(B, D, L)
    kernels = {}
    for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0]):
        ms_k = v[0] / steps
        ent = {"ms_per_step": round(ms_k, 4), "launches_per_step": v[1] / steps,
               "share_of_span": round(v[0] / max(tot_ms, 1e-9), 4)}
        if k in kab and ms_k > 0:
            ent["algorithmic_bytes_per_step"] = kab[k]
            ent["achieved_gbs"] = round(kab[k] / (ms_k * 1e-3) / 1e9, 1)
            ent["frac_of_peak"] = round(kab[k] / (ms_k * 1e-3) / 1e9 / peak_gbs, 4)
        kernels[k] = ent
    dominant = next(iter(kernels), None)
    traffic, traffic_src = None, None
    try:     # DRAM bytes of the same kernels from the committed ncu capture (same shape only)
        tj = json.load(open(os.path.join(ROOT, "profiles", "span_traffic.json")))
        if (L, D, B) == (L_FULL, D_MODEL, 1):
            traffic, traffic_src = tj["span_dram_bytes_per_step"], tj["source"]
    except Exception:
        pass
    projections = None
    if proj:
        pms = sum(v[0] for v in proj.values()) / steps
        flops = 3 * 2.0 * B * L * D * (3 * D + D)            # fwd + input grads + weight grads of in_proj and out_proj
        tf = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1590.0)))
        projections = {"ms_per_step": round(pms, 4), "fp32_equivalent_tflops": round(flops / (pms * 1e-3) / 1e12, 1),
                       "tf32_mma_tflops": round(3 * flops / (pms * 1e-3) / 1e12, 1),
                       "peak_tf32_dense_tflops_derived": round(tf / 2, 1),
                       "frac_of_tf32_peak": round(3 * flops / (pms * 1e-3) / 1e12 / (tf / 2), 4),
                       "note": "3xTF32: three tf32 MMAs per fp32 product; tf32 peak taken as half the measured bf16 peak",
                       "kernels": {k: {"ms_per_step": round(v[0] / steps, 4), "launches_per_step": v[1] / steps}
                                   for k, v in proj.items()}}
    return {"bound": "hbm", "kernel": "custom-kernel span (in_proj output -> out_proj input), fwd+bwd, per step",
            "projections": projections,
            "achieved": round(achieved, 1), "peak": peak_gbs, "unit": "GB/s",
            "frac": round(achieved / peak_gbs, 4), "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": peak_src, "algorithmic_bytes_per_step": span_bytes, "span_ms_per_step": round(span_ms, 4),
            "step_ms": round(ms_step, 4),
            "dominant_kernel": ({"name": dominant, **kernels[dominant]} if dominant else None),
            "kernels": kernels}


# ----------------------------------------------------------------------------------------- synthetic inputs
def nucleotide_activations(B, L, D, seed=2222):
    """SURVEY.md S8(d): token ids ~ U{7,8,9,10} (A,C,G,T; hg38_char_tokenizer.py:58-67), a 16-row embedding table
    ~ N(0, 0.02^2) and LayerNorm -> unit-scale rows drawn from four distinct vectors."""
    g = torch.Generator().manual_seed(seed)
    ids = torch.randint(7, 11, (B, L), generator=g)
    table = torch.randn(16, D, generator=g) * 0.02
    return torch.nn.functional.layer_norm(table[ids], (D,))


# ----------------------------------------------------------------------------------------- CPU arm
def cpu_reference_run(L, D, B, steps, warmup, threads=0, budget_s=None):
    """Time the oracle (reference torch.fft path restated, fp32) on the host cores.  With ``budget_s`` the number of
    timed steps is cut so that the whole call ends within the budget (at least one timed step)."""
    from oracle import hyena_oracle as O
    cores = threads if threads > 0 else min(os.cpu_count() or 1, 16)
    torch.set_num_threads(cores)
    g = torch.Generator().manual_seed(0)
    P = O.init_params(D, L, emb_dim=EMB, w=W_FREQ, generator=g, init_std=0.02)
    u, _ = O.nucleotide_activations(B, L, D)
    dy = torch.randn(B, L, D, generator=g)
    t_start = time.perf_counter()
    tw = time.perf_counter()
    for _ in range(warmup):
        O.operator_fwd_bwd(u, P, dy)
    tw = (time.perf_counter() - tw) / max(warmup, 1)
    done, t0 = 0, time.perf_counter()
    for _ in range(max(steps, 1)):
        O.operator_fwd_bwd(u, P, dy)
        done += 1
        per = (time.perf_counter() - t0) / done
        if budget_s is not None and (time.perf_counter() - t_start) + per > budget_s:
            break
    dt = (time.perf_counter() - t0) / done
    return {"value": B * L / dt, "unit": "nt/s", "cores": cores, "kind": "port",
            "host_cpus": os.cpu_count(),
            "sample": f"oracle fwd+bwd, fp32 torch CPU ({cores} threads of {os.cpu_count()} host CPUs), B={B} L={L} "
                      f"D={D}, {done} timed step(s) after {warmup} warm-up ({dt:.2f} s/step)"}, dt, done


def workload_config(L, D, B, world):
    return {"workload": f"large-1m: HyenaOperator fwd+bwd, L={L} d_model={D} order=2 filter_order=64 "
                        f"emb_dim={EMB}, batch {B}/GPU (global {world * B}), fp32, TF32 off",
            "parallelism": f"dp{world} (batch-sharded replicas, grad all-reduce)",
            "l2": "inputs larger than L2 (u, p, dy are 1-3 GB each; 126 MB L2), no explicit flush"}


def reference_arm(args):
    """The reference's own CPU path (oracle port of the torch.fft path) on the host cores, on the SAME workload
    (full L, D, batch).  One rank only; under torchrun the other ranks exit without work."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    L, D, B = args.seqlen, args.d_model, args.batch
    wu = min(args.warmup, 1)
    cb, dt, done = cpu_reference_run(L, D, B, args.steps, wu, args.cpu_threads, budget_s=args.ref_seconds)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "nt/s", "n_gpus": args.gpus,
            "steps": done, "steps_requested": args.steps, "warmup": wu, "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(L, D, B, world),
            "note": f"ONE host process on {cb['cores']} threads runs one sample of the workload per step regardless of "
                    f"--gpus (at N>1 the ratio to the N-GPU arm is not a per-GPU anchor); steps cut to the "
                    f"--ref-seconds budget ({args.ref_seconds:.0f} s)",
            "cpu_baseline": cb, "gpu_launches": 0,
            "e2e": {"value": cb["value"], "unit": "nt/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------- reference GPU path
def gpu_reference_run(op, u, dy, steps=3, warmup=1):
    """The reference's own GPU path (plain torch ops: F.linear, F.conv1d, torch.fft -> cuFFT; hyena.py:388-444), as the
    oracle restates it, on the same device, same weights, same inputs, fp32 with TF32 off: the >=10x denominator of
    north_star."""
    import gc
    from oracle import hyena_oracle as O
    B, L, D = u.shape
    P = O.canonical({k: v.detach() for k, v in op.state_dict().items()})
    which = "oracle restatement (oracle/hyena_oracle.py) of the reference torch.fft path on cuda (cuFFT)"

    def one():
        O.operator_fwd_bwd(u.detach(), P, dy)

    try:
        for _ in range(warmup):
            one()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            one()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
    finally:
        P = None
        gc.collect()
        torch.cuda.empty_cache()
    return {"ms_per_step": round(ms, 3), "value": B * L / (ms * 1e-3), "unit": "nt/s", "steps": steps,
            "warmup": warmup, "impl": which, "dtype": "f32, TF32 off"}


def bind_to_gpu_numa_node(local):
    """Pin this process (and hence the pinned host buffers it allocates next, first touch) to the CPUs of the NUMA node
    the GPU hangs off: with 8 ranks x 4.3 GB of PCIe traffic per step the e2e leg otherwise crosses the socket
    interconnect for half the GPUs (VERDICT r1: e2e scaling 0.665 at N = 8).  Best effort; returns a note for the line."""
    try:
        bus = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local)],
                             capture_output=True, text=True, timeout=20).stdout.strip().lower()
        if bus.startswith("0000"):
            bus = bus[4:]                                       # sysfs uses a 4-digit domain
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return "numa: single node"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
            return f"numa: GPU {local} on node {node}, process bound to its {len(allowed)} CPUs"
        return f"numa: node {node} has no allowed CPUs"
    except Exception as e:
        return f"numa: not bound ({type(e).__name__})"


# ----------------------------------------------------------------------------------------- GPU arm
def main():
    args = parse()
    if args.impl == "reference":
        return reference_arm(args)

    import hyena_dna_b200 as H
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU path for the product arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_note = bind_to_gpu_numa_node(local)
    if world > 1:
        # NCCL prints its version banner with printf on stdout when the environment sets NCCL_DEBUG; stdout must carry
        # exactly one JSON line, so communicator creation (eager with device_id, plus one barrier) runs with fd 1
        # pointing at stderr
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False

    L, D, B = args.seqlen, args.d_model, args.batch      # (oracle/ is imported by the cpu_baseline leg only)
    torch.manual_seed(1234)
    op = H.HyenaOperator(D, L, order=2, filter_order=64, emb_dim=EMB, w=W_FREQ, lr_pos_emb=0.0)
    # model-realistic init (standalone_hyenadna.py:612-641): Linear weights N(0, 0.02), biases 0
    g = torch.Generator().manual_seed(0)
    with torch.no_grad():
        for m in op.modules():
            if isinstance(m, torch.nn.Linear):
                m.weight.copy_(torch.randn(m.weight.shape, generator=g) * 0.02)
                if m.bias is not None:
                    m.bias.zero_()
        op.out_proj.weight.copy_(torch.randn(D, D, generator=g) * 0.02 / 4.0)
    op = op.to(dev)
    params = [p for p in op.parameters() if p.requires_grad]
    u_host = nucleotide_activations(B, L, D, seed=2222 + rank)
    dy_host = torch.randn(B, L, D, generator=torch.Generator().manual_seed(1 + rank))
    u_host, dy_host = u_host.pin_memory(), dy_host.pin_memory()
    u = u_host.to(dev).requires_grad_(True)
    dy = dy_host.to(dev)

    # N > 1: two-bucket gradient all-reduce driven by autograd hooks; the first (large) bucket is reduced on a side stream
    # while the filter backward still runs (hyena-dna_b200/distributed.py)
    reducer = H.distributed.OverlappedGradReducer(params, named=[(n, p) for n, p in op.named_parameters()
                                                                 if p.requires_grad]) if world > 1 else None

    def step():
        for p in params:
            p.grad = None
        u.grad = None
        y = op(u)
        y.backward(dy)
        if reducer is not None:
            reducer.finish()
        return y

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()              # running through warm-up so that samples exist when the timed region starts
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()

    # ---------------- timed region (device-resident inputs)
    n0 = H.launch_count()
    H._lib.profile_begin()
    barrier(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_begin = sampler.mark()
    e0.record()
    for _ in range(args.steps - 1):
        step()
    y = step()
    e1.record()
    torch.cuda.synchronize()
    t_end = sampler.mark()
    barrier()
    ms = e0.elapsed_time(e1)
    prof = H._lib.profile_end()
    launches = H.launch_count() - n0
    clocks = sampler.stop(t_begin, t_end) if rank == 0 else None
    if args.dump_outputs and rank == 0:     # before the legs below overwrite the grads
        dump_outputs(args.dump_outputs, {"y": y, "du": u.grad,
                                         **{"grad." + n: p.grad for n, p in op.named_parameters() if p.grad is not None}})
    del y
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = world * B * L / (ms_step * 1e-3)

    # ---------------- roofline of the custom-kernel span (rank 0's kernels)
    roofline = build_roofline(prof, args.steps, B, D, L, ms_step)

    # ---------------- e2e: host buffers in, host buffers out
    e2e = None
    if not args.no_e2e:
        y_host = torch.empty(B, L, D).pin_memory()
        du_host = torch.empty(B, L, D).pin_memory()
        g_host = [torch.empty(p.shape).pin_memory() for p in params]
        hs = H.HostStep(op, B, L, chunks=args.e2e_chunks)

        reduce_fn = H.distributed.allreduce_tensors if world > 1 else None

        def e2e_step():
            hs.step(u_host, dy_host, y_host, du_host, g_host, reduce_fn)
        for _ in range(2):
            e2e_step()
        torch.cuda.synchronize(); barrier()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(args.steps):
            e2e_step()
        a1.record()
        torch.cuda.synchronize(); barrier()
        t2 = torch.tensor([a0.elapsed_time(a1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        e2e_ms = float(t2.item()) / args.steps
        pbytes = sum(p.numel() for p in params) * 4
        e2e = {"value": world * B * L / (e2e_ms * 1e-3), "unit": "nt/s", "ms_per_step": round(e2e_ms, 3),
               "h2d_bytes_per_step": 2 * B * L * D * 4, "d2h_bytes_per_step": 2 * B * L * D * 4 + pbytes,
               "note": "per GPU, through hyena_dna_b200.HostStep: u,dy pinned host -> device; y, du, param grads device -> "
                       f"pinned host; u uploaded in {args.e2e_chunks} sequence chunks under the in_proj GEMM slices, dy under the forward, "
                       "y and du downloaded in chunks under the backward"}

    # ---------------- informational: the same step with TF32 projections (the reference's training setting,
    # train.py:34-35; NOT the matched-numerics number, reported separately and never used for `value`)
    tf32_ms = None
    if world == 1 and not args.no_e2e:
        torch.backends.cuda.matmul.allow_tf32 = True
        for _ in range(2):
            step()
        torch.cuda.synchronize()
        b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        b0.record()
        for _ in range(args.steps):
            step()
        b1.record()
        torch.cuda.synchronize()
        tf32_ms = b0.elapsed_time(b1) / args.steps
        torch.backends.cuda.matmul.allow_tf32 = False

    # ---------------- the reference's own GPU path on the same device (rank 0, N = 1 only)
    gpu_ref = None
    if rank == 0 and world == 1 and not args.no_gpu_reference:
        try:
            gpu_ref = gpu_reference_run(op, u.detach(), dy)
            gpu_ref["speedup"] = round(value / gpu_ref["value"], 3)
        except Exception as e:       # out of memory on a smaller device etc.: report, do not fail the bench line
            gpu_ref = {"unavailable": repr(e)[:200]}

    # ---------------- CPU baseline (rank 0, N = 1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu, _, _ = cpu_reference_run(min(args.cpu_sample_len, L), D, 1, 1, 1, args.cpu_threads)

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "nt/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(L, D, B, world),
                "gpu_launches": int(launches), "host_affinity": numa_note, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
                "gpu_reference": gpu_ref,
                "speedup_vs_gpu_reference": (gpu_ref or {}).get("speedup"),
                "tf32_projections_ms_per_step": tf32_ms,
                "impl": "b200"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
