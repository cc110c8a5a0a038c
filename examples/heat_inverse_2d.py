"""Recover a conductivity field from transient temperature measurements: an inverse heat problem solved with Adam through
the discrete adjoint of a backward-Euler rollout (DifferentiableHeatSolver).

Setup: rectangle(32, 32) (2048 elements), a per-element kappa with a warm inclusion, a batch of 64 random initial states,
100 implicit steps of dt = 1e-3, and the states recorded every 10 steps as the data.  Starting from kappa = 1 everywhere, Adam
on log(kappa) fits the recorded states; every iteration runs the whole rollout in one kernel launch and its adjoint.  Printed
per iteration: the data misfit and the relative L2 error of the kappa field.  Asserted: the misfit drops monotonically over
the first iterations (a property of the problem and the exact gradient, not a speed).

    python examples/heat_inverse_2d.py            (needs a CUDA device)
"""
import pathlib
import sys

import numpy as np
import torch

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parents[1]))
from difffe_physics_lab_b200 import DifferentiableHeatSolver, FEMesh   # noqa: E402


def main():
    torch.manual_seed(0)
    mesh = FEMesh.rectangle(32, 32)
    el = mesh.elements
    cx = mesh.nodes[el][..., 0].mean(1)
    cy = mesh.nodes[el][..., 1].mean(1)
    inclusion = ((cx - 0.6) ** 2 + (cy - 0.4) ** 2) < 0.2 ** 2
    kappa_true = torch.where(inclusion, 3.0, 1.0).to(torch.float64).cuda()
    dt, N, every, B = 1e-3, 100, 10, 64
    u0 = torch.rand((B, mesh.n_nodes), dtype=torch.float64, device="cuda")
    with torch.no_grad():
        data = DifferentiableHeatSolver(mesh, kappa_true, dt)(u0, N, every=every)

    log_k = torch.zeros(mesh.n_elements, dtype=torch.float64, device="cuda", requires_grad=True)
    opt = torch.optim.Adam([log_k], lr=0.02)
    misfits = []
    for it in range(40):
        opt.zero_grad()
        kappa = log_k.exp()
        U = DifferentiableHeatSolver(mesh, kappa, dt)(u0, N, every=every)
        misfit = 0.5 * ((U - data) ** 2).sum() / B
        misfit.backward()
        opt.step()
        err = float((kappa.detach() - kappa_true).norm() / kappa_true.norm())
        misfits.append(float(misfit))
        print(f"iter {it:3d}  misfit {float(misfit):.6e}  kappa rel. error {err:.4f}")
    assert all(b < a for a, b in zip(misfits[:5], misfits[1:6])), "misfit did not drop monotonically over 5 iterations"
    print(f"misfit {misfits[0]:.3e} -> {misfits[-1]:.3e} in {len(misfits)} Adam iterations")


if __name__ == "__main__":
    main()
