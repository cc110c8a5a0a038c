"""Throughput of DifferentiableHeatSolver: one JSON line per (B, checkpoint) on rectangle(32, 32), per-element kappa, N = 100.

    python tools/heat_bench.py [--steps 100] [--batches 1024,4096,16384] [--reps 3]

Fields: forward ms/step (rollout kernel, every 10th state returned), forward + adjoint + gradient ms/step, HeatStepper.step
ms/step on the same inputs (the forward baseline), state-steps/s of the forward, the DMMA flops and global-memory bytes per
step counted from the loop bounds and shapes, the CTA size the rollout kernels chose, and the GPU's name and power limit read
in the same run.  At B = 4096 the forward is also timed with 8 warps (128 states) per CTA, the CTA size of dfe_band_solve.
CUDA events, one warm-up call per configuration, median of --reps timed calls.  Needs a CUDA device (no CPU fallback).
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
from difffe_physics_lab_b200.timestepping import HeatStepper                     # noqa: E402

L2_BYTES = 126 * 2 ** 20


def gpu_identity():
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out


def timed(fn, reps):
    fn()                                                    # warm-up of this exact shape
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times))


def counts(B, nn, npad, N, every):
    """DMMA flops and global-memory bytes per time step, from the loop bounds of k_heat_roll / k_heat_grad."""
    nb, warps = npad // 32, -(-B // 16)
    # per warp and time step: 2 nb stage-2 products and 2 (nb - 1) stage-1 products, 40 m8n8k4 DMMAs (512 flops) each
    flops = warps * (4 * nb - 2) * 40 * 512
    carry = 4 * B * npad * 8                                # X read + written in each of the two passes
    fwd_bytes = carry + B * nn * 8                          # + the trajectory row
    adj_bytes = carry + 3 * B * npad * 8 + B * nn * 8 / every   # + lambda row, running sum, recorded dL/du_n
    grad_bytes = B * (nn + npad) * 8                        # u row + lambda row per (n, b) pair
    return flops, fwd_bytes, adj_bytes + grad_bytes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--batches", default="1024,4096,16384")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("heat_bench.py needs a CUDA device (difffe_physics_lab_b200 has no CPU fallback)")
    _native.build()
    name, power = gpu_identity()
    torch.cuda.set_device(0)
    rng = np.random.default_rng(0)
    mesh = FEMesh.rectangle(32, 32)
    nn = mesh.n_nodes
    N, every, dt = args.steps, 10, 1e-3
    kap = torch.tensor(np.exp(rng.uniform(np.log(0.3), np.log(3.0), mesh.n_elements)), device="cuda")
    h = mesh._native(0).handle
    lib = _native.lib()
    npad = int(lib.dfe_band_npad(h))
    for B in (int(b) for b in args.batches.split(",")):
        u0 = torch.rand((B, nn), dtype=torch.float64, device="cuda")
        hs = HeatStepper(mesh, kap, dt)
        t_hs = timed(lambda: hs.step(u0, N), args.reps)
        flops, fwd_b, bwd_b = counts(B, nn, npad, N, every)
        for ck in (None, 10):
            solver = DifferentiableHeatSolver(mesh, kap, dt, checkpoint=ck)
            with torch.no_grad():
                t_f = timed(lambda: solver(u0, N, every=every), args.reps)
            k = kap.clone().requires_grad_(True)
            u = u0.clone().requires_grad_(True)
            sg = DifferentiableHeatSolver(mesh, k, dt, checkpoint=ck)
            G = torch.randn((B, N // every, nn), dtype=torch.float64, device="cuda")

            def fwd_bwd():
                U = sg(u, N, every=every)
                torch.autograd.backward(U, G)

            t_fb = timed(fwd_bwd, args.reps)
            rec = {"mesh": "rectangle(32,32)", "n_free": mesh.n_nodes - len(mesh.dirichlet_nodes), "n_el": mesh.n_elements,
                   "kappa": "per-element", "N": N, "B": B, "every": every, "checkpoint": ck,
                   "cta_warps": int(lib.dfe_heat_warps(h, B)),
                   "fwd_ms_per_step": t_f / N, "fwd_adj_grad_ms_per_step": t_fb / N, "heatstepper_ms_per_step": t_hs / N,
                   "fwd_state_steps_per_s": B * N / (t_f * 1e-3),
                   "dmma_flops_per_step": flops, "fwd_tflops": flops / (t_f / N * 1e-3) / 1e12,
                   "fwd_bytes_per_step": fwd_b, "adj_grad_bytes_per_step": bwd_b,
                   "trajectory_bytes": B * N * nn * 8 if ck is None else B * (N // ck + ck) * nn * 8,
                   "gpu": name, "power_limit": power}
            rec["trajectory_exceeds_l2"] = rec["trajectory_bytes"] > L2_BYTES
            if B == 4096 and ck is None:                    # the CTA-size choice against 128 states per CTA
                try:
                    DifferentiableHeatSolver._cta_warps = 8
                    with torch.no_grad():
                        rec["fwd_ms_per_step_8warps"] = timed(lambda: solver(u0, N, every=every), args.reps) / N
                finally:
                    DifferentiableHeatSolver._cta_warps = 0
            print(json.dumps(rec), flush=True)
            del sg, G, u, k
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
