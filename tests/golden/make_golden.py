"""Generate golden vectors by running the UNMODIFIED reference implementation.

Needs a checkout of the original DiffFE-Physics-Lab (the directory that holds its ``diffhe`` package); the tests
only read the stored vectors:

    python tests/golden/make_golden.py --reference DIR          # small cases  (~1-2 min)
    python tests/golden/make_golden.py --reference DIR --big    # + 2D 64x64 / 128x128 forward (~3 min, ~7 GB RAM)

Outputs ``tests/golden/ref_small.npz`` and ``tests/golden/ref_big.npz``.  Every
array is float64/int64 stored bit-exactly.  Keys are ``<case>/<field>``.
"""
from __future__ import annotations

import argparse
import pathlib
import sys

import numpy as np
import torch

ap = argparse.ArgumentParser()
ap.add_argument("--reference", required=True, help="checkout of the original DiffFE-Physics-Lab")
ap.add_argument("--big", action="store_true")
a = ap.parse_args()
sys.path.insert(0, a.reference)
from diffhe.mesh import FEMesh  # noqa: E402  (reference)
from diffhe.solver import DifferentiableFESolver  # noqa: E402  (reference)

HERE = pathlib.Path(__file__).parent
out = {}


def put(case, **kw):
    for k, v in kw.items():
        out[f"{case}/{k}"] = np.asarray(v)


def mesh_arrays(mesh):
    keys = np.array(list(mesh.dirichlet_nodes.keys()), dtype=np.int64)
    vals = np.array(list(mesh.dirichlet_nodes.values()), dtype=np.float64)
    return dict(nodes=mesh.nodes.numpy(), elements=mesh.elements.numpy(), bc_idx=keys, bc_val=vals)


def run_case(case, mesh, kappa, f, gbar=None, loss="sum", backward=True, dense=False):
    """u = solver(f); L = sum(gbar*u); record u, dL/dkappa, dL/df."""
    kap = torch.tensor(float(kappa), dtype=torch.float64, requires_grad=backward)
    ft = torch.tensor(np.asarray(f), dtype=torch.float64, requires_grad=backward)
    solver = DifferentiableFESolver(mesh, kappa=kap)
    put(case, kappa=float(kappa), f=np.asarray(f, dtype=np.float64), **mesh_arrays(mesh))
    if not backward:
        with torch.no_grad():
            u = solver(ft)
        put(case, u=u.numpy())
        return
    u = solver(ft)
    if gbar is None:
        gbar = np.ones(mesh.n_nodes)
    L = (torch.tensor(gbar, dtype=torch.float64) * u).sum()
    L.backward()
    put(case, u=u.detach().numpy(), gbar=gbar, gkappa=kap.grad.numpy(), gf=ft.grad.numpy())
    if dense:
        # dense K, F exactly as the reference builds them (solver.py:79-96 / 109-145)
        K, F = capture_dense(mesh, float(kappa), np.asarray(f, dtype=np.float64))
        put(case, K=K, F=F)


def capture_dense(mesh, kappa, f):
    """Call the reference's own assembly, intercepting _apply_bc_and_solve."""
    grabbed = {}
    s = DifferentiableFESolver(mesh, kappa=kappa)

    def grab(K, F):
        grabbed["K"] = K.detach().numpy().copy()
        grabbed["F"] = F.detach().numpy().copy()
        return torch.zeros(mesh.n_nodes, dtype=torch.float64)

    s._apply_bc_and_solve = grab  # instance attribute shadows the method; reference code untouched
    with torch.no_grad():
        s(torch.tensor(f, dtype=torch.float64))
    return grabbed["K"], grabbed["F"]


def small():
    rng = np.random.default_rng(20261018)
    # --- C1: line(20), kappa=1, f=1 (BASELINE config 1)
    m = FEMesh.line(20)
    run_case("c1_line20", m, 1.0, np.ones(21), dense=True)
    # --- demo step 0 (examples/poisson_1d_demo.py:88-110)
    m = FEMesh.line(30)
    with torch.no_grad():
        u_data = DifferentiableFESolver(m, kappa=torch.tensor(2.0, dtype=torch.float64))(torch.ones(31, dtype=torch.float64))
    kest = torch.tensor(1.0, dtype=torch.float64, requires_grad=True)
    u = DifferentiableFESolver(m, kappa=kest.abs())(torch.ones(31, dtype=torch.float64))
    loss = ((u - u_data) ** 2).mean()
    loss.backward()
    put("demo_line30", u_data=u_data.numpy(), u=u.detach().numpy(), loss=float(loss), gkappa=kest.grad.numpy(), **mesh_arrays(m))
    # --- 1D with non-zero Dirichlet, random f / gbar
    m = FEMesh.line(10, bc_left=1.0, bc_right=2.0)
    run_case("line10_bc12_f0", m, 1.0, np.zeros(11), backward=False)
    run_case("line10_bc12_rand", m, 1.7, rng.uniform(-1, 2, 11), gbar=rng.standard_normal(11), dense=True)
    m = FEMesh.line(40, x_left=-0.3, x_right=2.1, bc_left=-0.5, bc_right=0.25)
    run_case("line40_rand", m, 0.37, rng.uniform(0, 1, 41), gbar=rng.standard_normal(41), dense=True)
    # --- mixed (one natural end)
    m = FEMesh.line(8, bc_left=1.0, bc_right=None)
    run_case("line8_left_only", m, 1.3, rng.uniform(0, 1, 9), gbar=rng.standard_normal(9), dense=True)
    m = FEMesh.line(8, bc_left=None, bc_right=-0.7)
    run_case("line8_right_only", m, 0.8, rng.uniform(0, 1, 9), gbar=rng.standard_normal(9), dense=True)
    # --- smallest meshes (edge cases): 2 elements -> 1 unknown, both BC lift into the same row
    m = FEMesh.line(2, bc_left=0.5, bc_right=-1.5)
    run_case("line2_bc", m, 1.1, np.array([0.3, 0.9, -0.2]), gbar=np.array([1.0, -2.0, 0.5]), dense=True)
    m = FEMesh.line(3, bc_left=0.5, bc_right=-1.5)
    run_case("line3_bc", m, 1.1, np.array([0.3, 0.9, -0.2, 0.4]), gbar=np.array([1.0, -2.0, 0.5, 0.1]), dense=True)
    # --- 1D scaling (SURVEY §8c): d(sum u)/dkappa
    for n in (100, 400):
        run_case(f"line{n}_ones", FEMesh.line(n), 1.0, np.ones(n + 1))
    run_case("line1600_ones", FEMesh.line(1600), 1.0, np.ones(1601), backward=False)
    # --- float32 forcing is promoted to float64 (SURVEY §7 quirks)
    m = FEMesh.line(12)
    f32 = torch.linspace(0, 1, 13, dtype=torch.float32)
    with torch.no_grad():
        u = DifferentiableFESolver(m)(f32)
    put("line12_f32", f=f32.numpy(), u=u.numpy(), **mesh_arrays(m))
    assert u.dtype == torch.float64
    # --- 2D, kappa=1, f=1, zero BC
    for n in (4, 8, 16):
        run_case(f"rect{n}_ones", FEMesh.rectangle(n, n), 1.0, np.ones((n + 1) ** 2), dense=(n <= 8))
    # --- 2D non-square, non-zero BC, random everything
    m = FEMesh.rectangle(7, 5, x_range=(0.0, 2.3), y_range=(-1.0, 0.7), bc_value=0.3)
    run_case("rect7x5_rand", m, 2.1, rng.uniform(-1, 2, 48), gbar=rng.standard_normal(48), dense=True)
    m = FEMesh.rectangle(6, 9, x_range=(-1.0, 0.5), y_range=(0.2, 3.0), bc_value=-1.2)
    run_case("rect6x9_rand", m, 0.45, rng.uniform(0, 1, 70), gbar=rng.standard_normal(70), dense=True)
    # --- 2D with only part of the boundary constrained (user-edited dict, reversed insertion order)
    m = FEMesh.rectangle(5, 4)
    keys = [k for k in m.dirichlet_nodes if float(m.nodes[k, 0]) == 0.0 or float(m.nodes[k, 1]) == 0.0]
    m.dirichlet_nodes = {k: 0.1 * (i + 1) for i, k in enumerate(reversed(keys))}
    run_case("rect5x4_partial_bc", m, 1.5, rng.uniform(0, 1, 30), gbar=rng.standard_normal(30), dense=True)
    # --- 2D with a degenerate (zero-area) element appended (solver.py:120-121 skip)
    m = FEMesh.rectangle(3, 3)
    m.elements = torch.cat([m.elements, torch.tensor([[5, 5, 6], [0, 1, 2]])], dim=0)
    run_case("rect3_degenerate", m, 1.0, rng.uniform(0, 1, 16), gbar=rng.standard_normal(16), dense=True)
    # --- 2D forward, 32x32
    run_case("rect32_ones", FEMesh.rectangle(32, 32), 1.0, np.ones(33 * 33), backward=False)
    np.savez_compressed(HERE / "ref_small.npz", **out)
    print("wrote ref_small.npz with", len(out), "arrays")


def big():
    out.clear()
    for n in (64, 128):
        m = FEMesh.rectangle(n, n)
        with torch.no_grad():
            u = DifferentiableFESolver(m)(torch.ones(m.n_nodes, dtype=torch.float64))
        put(f"rect{n}_ones", u=u.numpy(), n=n)
        print(n, float(u.max()), float(u.sum()), flush=True)
    np.savez_compressed(HERE / "ref_big.npz", **out)


if __name__ == "__main__":
    if a.big:
        big()
    else:
        small()
