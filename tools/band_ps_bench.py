"""Per-sample-kappa batches on rectangle(32, 32) (961 unknowns), kappa (B, n_el): the batched banded route
(dfe_band_ps_fwd / _bwd) against the per-sample loop (assemble / eliminate / Jacobi-PCG per sample), one JSON line each.

    python tools/band_ps_bench.py [--batches 2,64,1024,4096,16384] [--loop-max 4096] [--reps 5] [--profile-batch 4096]

A step is forward + adjoint: u = solver(f), (u * gbar).sum().backward() with f and kappa requiring gradients.  CUDA
events around the step (which ends in a synchronisation), one warm-up step per configuration, median of --reps steps;
the two routes alternate inside each repetition.  The loop runs only for B <= --loop-max (B serial solves per direction),
and with one timed step from B = 1024 on.  A separate torch.profiler run at --profile-batch gives the per-kernel split,
turned into achieved GB/s and GFLOP/s with the bytes and flops per sample counted from the shapes (counts()).  The GPU's
name and power limit are read in the same run.  Needs a CUDA device (no CPU fallback).
"""
import argparse
import json
import pathlib
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parents[1]))
from difffe_physics_lab_b200 import DifferentiableFESolver, FEMesh, _native   # noqa: E402


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def counts(nm):
    """Global-memory bytes and flops per sample of each kernel of the new route, from the mesh's shapes."""
    I = nm.info
    n, ne, nf, nnz = I.n_nodes, I.n_elements, I.n_free, I.nnz_full
    npad = _native.lib().dfe_band_npad(nm.handle)
    nb = npad // 32
    fac = npad * 33 * 8                                    # invd | Lr of one sample
    # blocked Cholesky per block row: dense 32 x 32 Cholesky (32^3 / 3 fma), X = S L^-T (32 * 32^2 / 2 fma), lower half
    # of the rank-32 update (528 * 32 fma)
    chol = nb * 2 * (32 ** 3 / 3 + 32 * 32 ** 2 / 2 + 528 * 32)
    return {
        "k_bps_assemble": (ne * 8 + nnz * 8, 3 * 3 * ne * 6),            # kappa in, vals out; 6 flops per entry
        "k_bps_factor": (nnz * 8 + fac, chol),                            # vals in, factor out
        "k_band_rhs_fwd": (n * 8 + npad * 8, 3 * ne * 4),                 # f in, rhs out
        "k_bps_solve": (2 * (2 * fac + 2 * npad * 8 + n * 8), 2 * 2 * 2 * 32 * nf),   # fwd and adjoint: 2 sweeps each
        "k_band_grad2": (2 * n * 8 + npad * 8 + ne * 8, ne * 16 + n * 6),  # u, lambda in; dL/dkappa, dL/df out
    }


def make_step(m, f, kap, gbar, loop):
    def step():
        k = kap.clone().requires_grad_(True)
        ft = f.clone().requires_grad_(True)
        s = DifferentiableFESolver(m, kappa=k)
        if loop:
            s._opts["batch_min"] = 10 ** 9
        u = s(ft)
        (u * gbar).sum().backward()
        return u.detach(), k.grad, ft.grad
    return step


def time_once(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="2,64,1024,4096,16384")
    ap.add_argument("--loop-max", type=int, default=4096)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--profile-batch", type=int, default=4096)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("band_ps_bench.py needs a CUDA device")
    gpu, power = gpu_identity()
    m = FEMesh.rectangle(32, 32, bc_value=0.1)
    nm = m._native(torch.cuda.current_device())
    assert _native.lib().dfe_band_ps_supported(nm.handle) == 1
    rng = np.random.default_rng(0)
    for B in [int(x) for x in args.batches.split(",")]:
        f = torch.tensor(rng.uniform(-1.0, 1.0, (B, m.n_nodes)), device="cuda")
        gbar = torch.tensor(rng.standard_normal((B, m.n_nodes)), device="cuda")
        kap = torch.tensor(np.exp(rng.uniform(np.log(1e-3), 0.0, (B, m.n_elements))), device="cuda")
        new = make_step(m, f, kap, gbar, False)
        run_loop = B <= args.loop_max
        old = make_step(m, f, kap, gbar, True) if run_loop else None
        new()
        reps_old = args.reps if B < 1024 else 1
        t_new, t_old, rel = [], [], None
        if run_loop:
            old()
        for r in range(args.reps):
            t, out_new = time_once(new)
            t_new.append(t)
            if run_loop and r < reps_old:
                t, out_old = time_once(old)
                t_old.append(t)
                if rel is None:
                    rel = [float((a - b).abs().max() / b.abs().max()) for a, b in zip(out_new, out_old)]
        line = {"B": B, "kappa": "(B, n_el)", "mesh": "rectangle(32, 32)", "new_ms": float(np.median(t_new)),
                "new_samples_per_s": B / (float(np.median(t_new)) * 1e-3),
                "loop_ms": float(np.median(t_old)) if t_old else None, "loop_steps_timed": len(t_old),
                "speedup": float(np.median(t_old) / np.median(t_new)) if t_old else None,
                "relerr_u_gk_gf_vs_loop": rel, "gpu": gpu, "power_limit": power}
        print(json.dumps(line), flush=True)
        del f, gbar, kap, new, old
        torch.cuda.empty_cache()

    # per-kernel split, in a run of its own
    from torch.profiler import ProfilerActivity, profile
    B = args.profile_batch
    f = torch.tensor(rng.uniform(-1.0, 1.0, (B, m.n_nodes)), device="cuda")
    gbar = torch.tensor(rng.standard_normal((B, m.n_nodes)), device="cuda")
    kap = torch.tensor(np.exp(rng.uniform(np.log(1e-3), 0.0, (B, m.n_elements))), device="cuda")
    step = make_step(m, f, kap, gbar, False)
    step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        name = e.name
        for k in counts(nm):
            if k in name:
                name = k
        us = e.device_time if hasattr(e, "device_time") else e.cuda_time
        c, t = per.get(name, (0, 0.0))
        per[name] = (c + 1, t + us)
    cnt = counts(nm)
    for name, (c, us) in sorted(per.items(), key=lambda kv: -kv[1][1]):
        row = {"profile_B": B, "kernel": name[:60], "launches": c, "ms": us / 1e3, "gpu": gpu, "power_limit": power}
        if name in cnt:
            by, fl = cnt[name]
            row["GB_per_s"] = by * B / (us * 1e-6) / 1e9
            row["GFLOP_per_s"] = fl * B / (us * 1e-6) / 1e9
            row["bytes_per_sample"], row["flops_per_sample"] = by, fl
        print(json.dumps(row), flush=True)


if __name__ == "__main__":
    main()
