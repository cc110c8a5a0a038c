"""Heat rollouts with one conductivity field per sample on rectangle(32, 32) (961 unknowns), kappa (B, n_el) log-uniform
in [0.3, 3], N = 100 steps recorded every 10: the per-sample route (dfe_heat_ps_*) against the per-sample loop of
shared-kappa solvers, one JSON line per configuration.

    python tools/heat_ps_bench.py [--batches 64,1024,4096] [--checkpoints none,10] [--reps 3] [--loop-max 1024]
                                  [--profile-batch 4096]

Per (B, checkpoint): the forward call (no gradient) and the forward + backward call (L = sum(W * U), gradients to u0, kappa
and f), timed with CUDA events around work that ends in a synchronisation, one warm-up call, median of --reps.  The
set-up (assembly + factorisation) and rollout kernel times come from KernelTimer events in the timed calls.  The loop
(B shared-route solvers, one sample each, forward + backward) alternates with the new route: every repetition below
B = 1024, one timed repetition from B = 1024 on, not run above --loop-max.  The outputs of both routes are compared
(states, dL/du0, dL/dkappa, dL/df).  Bytes per step are counted from the shapes (step_bytes()).  A separate
torch.profiler run at --profile-batch gives the per-kernel split.  The GPU's name and power limit are read in the same
run.  Needs a CUDA device (no CPU fallback).
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


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def step_bytes(nm):
    """Global-memory bytes per sample and time step of the rollout kernels, from the mesh's shapes: the factor is read
    once per sweep; the carry is read and written once per sweep; forward reads c_b and writes a node-layout state,
    the adjoint reads the recorded dL/du rows (1 / EVERY of the steps) and writes lambda and the running sum."""
    I = nm.info
    n = I.n_nodes
    npad = _native.lib().dfe_band_npad(nm.handle)
    fac = npad * 33 * 8
    fwd = 2 * fac + 2 * 2 * npad * 8 + npad * 8 + n * 8
    adj = 2 * fac + 2 * 2 * npad * 8 + n * 8 / EVERY + 3 * npad * 8
    grad = n * 8 + npad * 8                                 # k_hps_grad: u and lambda rows of every step
    return {"fwd": fwd, "adj": adj, "grad": grad}


def run(m, kap, f, u0, W, checkpoint, backward):
    k = kap.clone().requires_grad_(backward)
    fs = f.clone().requires_grad_(backward)
    u = u0.clone().requires_grad_(backward)
    s = DifferentiableHeatSolver(m, k, DT, fs, checkpoint=checkpoint)
    if not backward:
        with torch.no_grad():
            return (s(u, N, every=EVERY),)
    U = s(u, N, every=EVERY)
    (W * U).sum().backward()
    return U.detach(), u.grad, k.grad, fs.grad


def loop(m, kap, f, u0, W):
    """the per-sample loop: one shared-kappa solver per sample, forward + backward"""
    outs = [run(m, kap[b], f, u0[b:b + 1], W[b:b + 1], None, True) for b in range(kap.shape[0])]
    return (torch.cat([o[0] for o in outs]), torch.cat([o[1] for o in outs]), torch.stack([o[2] for o in outs]),
            torch.stack([o[3] for o in outs]).sum(0))


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="64,1024,4096")
    ap.add_argument("--checkpoints", default="none,10")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--loop-max", type=int, default=1024)
    ap.add_argument("--profile-batch", type=int, default=4096)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("heat_ps_bench.py needs a CUDA device")
    gpu, power = gpu_identity()
    m = FEMesh.rectangle(32, 32, bc_value=0.1)
    nm = m._native(torch.cuda.current_device())
    assert _native.lib().dfe_band_ps_supported(nm.handle) == 1
    sb = step_bytes(nm)
    rng = np.random.default_rng(0)
    cks = [None if c == "none" else int(c) for c in args.checkpoints.split(",")]
    for B in [int(x) for x in args.batches.split(",")]:
        kap = torch.tensor(np.exp(rng.uniform(np.log(0.3), np.log(3.0), (B, m.n_elements))), device="cuda")
        f = torch.tensor(rng.uniform(-1.0, 1.0, m.n_nodes), device="cuda")
        u0 = torch.tensor(rng.uniform(-1.0, 1.0, (B, m.n_nodes)), device="cuda")
        W = torch.tensor(rng.standard_normal((B, N // EVERY, m.n_nodes)), device="cuda")
        for c in cks:
            run(m, kap, f, u0, W, c, False)
            run(m, kap, f, u0, W, c, True)
            use_loop = c is None and B <= args.loop_max
            reps_loop = args.reps if B < 1024 else 1
            t_f, t_fb, t_loop, split, rel = [], [], [], {}, None
            for r in range(args.reps):
                t, _ = timed(lambda: run(m, kap, f, u0, W, c, False))
                t_f.append(t)
                with KernelTimer() as kt:
                    t, out_new = timed(lambda: run(m, kap, f, u0, W, c, True))
                t_fb.append(t)
                for name, (_, ms) in kt.summary().items():
                    split.setdefault(name, []).append(ms)
                if use_loop and r < reps_loop:
                    t, out_old = timed(lambda: loop(m, kap, f, u0, W))
                    t_loop.append(t)
                    if rel is None:
                        rel = {k: float((a - b).abs().max() / b.abs().max())
                               for k, a, b in zip(("U", "du0", "dkappa", "df"), out_new, out_old)}
                del out_new
            med = {k: float(np.median(v)) for k, v in split.items()}
            n_fwd = N * (2 if c is not None else 1)         # checkpointing recomputes every segment in the backward
            fwd_kernel_step = med["heat_ps_fwd"] / n_fwd
            adj_kernel_step = med["heat_ps_adj"] / N
            line = {"B": B, "checkpoint": c, "N": N, "every": EVERY, "kappa": "(B, n_el)", "mesh": "rectangle(32, 32)",
                    "setup_ms": med.get("heat_ps_setup"),
                    "fwd_ms_per_step": float(np.median(t_f)) / N,
                    "fwd_bwd_ms_per_step": float(np.median(t_fb)) / N,
                    "kernel_ms": med,
                    "fwd_kernel_ms_per_step": fwd_kernel_step, "adj_kernel_ms_per_step": adj_kernel_step,
                    "fwd_bytes_per_step": sb["fwd"] * B, "adj_bytes_per_step": sb["adj"] * B,
                    "fwd_GB_per_s": sb["fwd"] * B / (fwd_kernel_step * 1e-3) / 1e9,
                    "adj_GB_per_s": sb["adj"] * B / (adj_kernel_step * 1e-3) / 1e9,
                    "loop_fwd_bwd_ms_per_step": float(np.median(t_loop)) / N if t_loop else None,
                    "loop_reps": len(t_loop),
                    "speedup_fwd_bwd": float(np.median(t_loop) / np.median(t_fb)) if t_loop else None,
                    "relerr_vs_loop": rel,
                    "ok_vs_loop": None if rel is None else (rel["U"] <= 1e-12 and max(rel["du0"], rel["dkappa"],
                                                                                          rel["df"]) <= 1e-10),
                    "gpu": gpu, "power_limit": power}
            print(json.dumps(line), flush=True)
        del kap, f, u0, W
        torch.cuda.empty_cache()

    # per-kernel split, in a run of its own
    from torch.profiler import ProfilerActivity, profile
    B = args.profile_batch
    kap = torch.tensor(np.exp(rng.uniform(np.log(0.3), np.log(3.0), (B, m.n_elements))), device="cuda")
    f = torch.tensor(rng.uniform(-1.0, 1.0, m.n_nodes), device="cuda")
    u0 = torch.tensor(rng.uniform(-1.0, 1.0, (B, m.n_nodes)), device="cuda")
    W = torch.tensor(rng.standard_normal((B, N // EVERY, m.n_nodes)), device="cuda")
    run(m, kap, f, u0, W, None, True)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        run(m, kap, f, u0, W, None, True)
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = e.device_time if hasattr(e, "device_time") else e.cuda_time
        c, t = per.get(e.name, (0, 0.0))
        per[e.name] = (c + 1, t + us)
    for name, (c, us) in sorted(per.items(), key=lambda kv: -kv[1][1])[:14]:
        print(json.dumps({"profile_B": B, "checkpoint": None, "kernel": name[:70], "launches": c, "ms": us / 1e3,
                          "gpu": gpu, "power_limit": power}), flush=True)


if __name__ == "__main__":
    main()
