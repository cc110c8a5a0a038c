"""Heat rollouts with sources per sample and per step on rectangle(32, 32) (961 unknowns), N = 100 steps recorded every 10,
one JSON line per (route, B, source form, checkpoint).

    python tools/heat_src_bench.py [--batches 64,1024,4096] [--checkpoints none,10] [--reps 3] [--profile-batch 4096]

Routes: kappa shared by the batch (n_el,) and one field per sample (B, n_el).  Source forms: constructor f (n,) (the
baseline, no new kernel), f (B, n), source (N, n), source (B, N, n).  Per configuration: the forward call (no gradient) and
the forward + backward call (L = sum(W * U), gradients to u0, kappa and every source), timed with CUDA events around work
that ends in a synchronisation, one warm-up call, median of --reps.  The new kernels' times (dfe_heat_src_load and
dfe_heat_src_grad, each with its small table kernel) come from KernelTimer events in the timed forward + backward call;
their bytes are counted from the shapes (src_bytes()) and given as a fraction of 6.5 TB/s, the copy bandwidth measured on
a B200 (DESIGN.md).  A separate torch.profiler run at --profile-batch gives the per-kernel split of the (B, N, n) form.
The GPU's name and power limit are read in the same run.  Needs a CUDA device (no CPU fallback).
"""
import argparse
import json
import pathlib
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parents[1]))
from difffe_physics_lab_b200 import DifferentiableHeatSolver, FEMesh, _native   # noqa: E402
from difffe_physics_lab_b200.solver import KernelTimer                           # noqa: E402

N, EVERY, DT = 100, 10, 1e-3
COPY_BW = 6.5e12
FORMS = ["f_n", "f_B", "src_N", "src_BN"]


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def src_bytes(n, npad, B, form, per_sample_kappa, n_fwd):
    """Global-memory bytes of the new kernels over one forward + backward call, from the shapes.  dfe_heat_src_load:
    per row the source row (n doubles) and the c row written (npad), plus the base row (npad) when it is per sample;
    dfe_heat_src_grad: per row the lambda row (npad) and the gradient row written (n).  n_fwd: forward rollouts of the
    call (2 with checkpointing: the backward recomputes every segment)."""
    per_base = per_sample_kappa or form == "f_B"
    if form == "f_n":
        return {"load": 0, "grad": 0}
    if form == "f_B":
        # one load of B rows at set-up; dL/df from lam_sum (B rows)
        return {"load": B * (n + npad + (npad if per_sample_kappa else 0)) * 8, "grad": B * (npad + n) * 8}
    nb = 1 if form == "src_N" and not per_base else B
    load = n_fwd * N * nb * (n + npad + (npad if per_base else 0)) * 8
    rows = N if form == "src_N" else N * B
    return {"load": load, "grad": rows * (npad + n) * 8}


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def inputs(m, B, form, per_sample, gen):
    n = m.n_nodes
    r = lambda *s: torch.rand(s, dtype=torch.float64, device="cuda", generator=gen) * 2 - 1
    kap = torch.exp(torch.rand((B, m.n_elements) if per_sample else (m.n_elements,), dtype=torch.float64, device="cuda",
                               generator=gen) * 2.3 - 1.2)
    f = r(B, n) if form == "f_B" else r(n)
    src = r(N, n) if form == "src_N" else r(B, N, n) if form == "src_BN" else None
    return kap, f, src, r(B, n), r(B, N // EVERY, n)


def run(m, kap, f, src, u0, W, checkpoint, backward):
    leaf = lambda t: None if t is None else t.clone().requires_grad_(backward)
    k, fs, ss, u = leaf(kap), leaf(f), leaf(src), leaf(u0)
    s = DifferentiableHeatSolver(m, k, DT, fs, checkpoint=checkpoint)
    if not backward:
        with torch.no_grad():
            return s(u, N, every=EVERY, source=ss)
    (W * s(u, N, every=EVERY, source=ss)).sum().backward()
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="64,1024,4096")
    ap.add_argument("--checkpoints", default="none,10")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--profile-batch", type=int, default=4096)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("heat_src_bench.py needs a CUDA device")
    gpu, power = gpu_identity()
    m = FEMesh.rectangle(32, 32, bc_value=0.1)
    nm = m._native(torch.cuda.current_device())
    n, npad = m.n_nodes, _native.lib().dfe_band_npad(nm.handle)
    gen = torch.Generator(device="cuda").manual_seed(0)
    cks = [None if c == "none" else int(c) for c in args.checkpoints.split(",")]
    for per_sample in (False, True):
        for B in [int(x) for x in args.batches.split(",")]:
            for form in FORMS:
                kap, f, src, u0, W = inputs(m, B, form, per_sample, gen)
                for c in cks:
                    run(m, kap, f, src, u0, W, c, False)
                    run(m, kap, f, src, u0, W, c, True)
                    t_f, t_fb, split = [], [], {}
                    for _ in range(args.reps):
                        t_f.append(timed(lambda: run(m, kap, f, src, u0, W, c, False))[0])
                        with KernelTimer() as kt:
                            t_fb.append(timed(lambda: run(m, kap, f, src, u0, W, c, True))[0])
                        for name, (_, ms) in kt.summary().items():
                            split.setdefault(name, []).append(ms)
                    med = {k: float(np.median(v)) for k, v in split.items()}
                    sb = src_bytes(n, npad, B, form, per_sample, 2 if c is not None else 1)
                    new = {}
                    for k, key in (("load", "heat_src_load"), ("grad", "heat_src_grad")):
                        if key in med and sb[k]:
                            new[k] = {"ms": med[key], "bytes": sb[k], "TB_per_s": sb[k] / (med[key] * 1e-3) / 1e12,
                                      "frac_of_6.5TB_s": sb[k] / (med[key] * 1e-3) / COPY_BW}
                    print(json.dumps({"kappa": "(B, n_el)" if per_sample else "(n_el,)", "B": B, "form": form,
                                      "checkpoint": c, "N": N, "every": EVERY, "mesh": "rectangle(32, 32)",
                                      "fwd_ms_per_step": float(np.median(t_f)) / N,
                                      "fwd_bwd_ms_per_step": float(np.median(t_fb)) / N,
                                      "new_kernels": new, "kernel_ms": med, "gpu": gpu, "power_limit": power}), flush=True)
                del kap, f, src, u0, W
                torch.cuda.empty_cache()

    from torch.profiler import ProfilerActivity, profile
    B = args.profile_batch
    for per_sample in (False, True):
        kap, f, src, u0, W = inputs(m, B, "src_BN", per_sample, gen)
        run(m, kap, f, src, u0, W, None, True)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run(m, kap, f, src, u0, W, None, True)
            torch.cuda.synchronize()
        per = {}
        for e in prof.events():
            if e.device_type != torch.autograd.DeviceType.CUDA:
                continue
            us = e.device_time if hasattr(e, "device_time") else e.cuda_time
            cnt, t = per.get(e.name, (0, 0.0))
            per[e.name] = (cnt + 1, t + us)
        for name, (cnt, us) in sorted(per.items(), key=lambda kv: -kv[1][1])[:12]:
            print(json.dumps({"profile_B": B, "kappa": "(B, n_el)" if per_sample else "(n_el,)", "form": "src_BN",
                              "kernel": name[:70], "launches": cnt, "ms": us / 1e3, "gpu": gpu, "power_limit": power}),
                  flush=True)
        del kap, f, src, u0, W
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
