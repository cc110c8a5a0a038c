"""Recover a moving heat source from recorded transients: an inverse source problem solved with Adam through the discrete
adjoint of a backward-Euler rollout with a time-dependent source (DifferentiableHeatSolver(...)(u0, N, source=q)).

Setup: rectangle(32, 32), kappa = 1, a Gaussian heater of width 0.08 moving along a circle of radius 0.25 around the
centre, 40 implicit steps of dt = 2e-3, a batch of 8 random initial states, and every state recorded as the data.  Starting
from q = 0, Adam on the per-step source q (40, n_nodes) fits the recorded states.  Printed per iteration: the data misfit
and the relative L2 error of the source.  Asserted: the misfit drops monotonically over the first iterations (a property of
the problem and the exact gradient, not a speed).

    python examples/heat_source_2d.py            (needs a CUDA device)
"""
import math
import pathlib
import sys

import torch

sys.path.insert(0, str(pathlib.Path(__file__).resolve().parents[1]))
from difffe_physics_lab_b200 import DifferentiableHeatSolver, FEMesh   # noqa: E402


def main():
    torch.manual_seed(0)
    mesh = FEMesh.rectangle(32, 32)
    x, y = mesh.nodes[:, 0].to(torch.float64).cuda(), mesh.nodes[:, 1].to(torch.float64).cuda()
    dt, N, B = 2e-3, 40, 8
    t = torch.arange(1, N + 1, dtype=torch.float64, device="cuda") * dt       # step n evaluates the source at t_{n+1}
    px, py = 0.5 + 0.25 * torch.cos(2 * math.pi * t / (N * dt)), 0.5 + 0.25 * torch.sin(2 * math.pi * t / (N * dt))
    q_true = 50.0 * torch.exp(-((x[None] - px[:, None]) ** 2 + (y[None] - py[:, None]) ** 2) / (2 * 0.08 ** 2))
    u0 = torch.rand((B, mesh.n_nodes), dtype=torch.float64, device="cuda")
    solver = DifferentiableHeatSolver(mesh, 1.0, dt)
    with torch.no_grad():
        data = solver(u0, N, every=1, source=q_true)

    q = torch.zeros((N, mesh.n_nodes), dtype=torch.float64, device="cuda", requires_grad=True)
    opt = torch.optim.Adam([q], lr=0.5)
    misfits = []
    for it in range(100):
        opt.zero_grad()
        U = solver(u0, N, every=1, source=q)
        misfit = 0.5 * ((U - data) ** 2).sum() / B
        misfit.backward()
        opt.step()
        err = float((q.detach() - q_true).norm() / q_true.norm())
        misfits.append(float(misfit.detach()))
        print(f"iter {it:3d}  misfit {misfits[-1]:.6e}  source rel. error {err:.4f}")
    assert all(b < a for a, b in zip(misfits[:5], misfits[1:6])), "misfit did not drop monotonically over 5 iterations"
    print(f"misfit {misfits[0]:.3e} -> {misfits[-1]:.3e} in {len(misfits)} Adam iterations")


if __name__ == "__main__":
    main()
