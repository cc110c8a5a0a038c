"""Operator reuse for time stepping (SURVEY §8f N4): dfe_band_factor on M_L + dt K, dfe_band_solve per step."""
import numpy as np
import pytest
import torch

from difffe_physics_lab_b200 import FEMesh, _native

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    _native.build()


def test_heat_eigenmode_decay_closed_form():
    """Backward Euler with the lumped mass on the uniform mesh: the first eigenmode decays by 1 / (1 + dt lambda_h) per
    step, lambda_h = kappa * 8 / h^2 * sin^2(pi h / 2) (5-point operator) — to rounding."""
    from difffe_physics_lab_b200.timestepping import HeatStepper

    nx, kappa, dt, n = 32, 1.3, 1e-3, 20
    mesh = FEMesh.rectangle(nx, nx)
    hs = HeatStepper(mesh, kappa, dt)
    x, y = mesh.nodes[:, 0].cuda(), mesh.nodes[:, 1].cuda()
    u0 = (torch.sin(np.pi * x) * torch.sin(np.pi * y)).reshape(1, -1)
    u = hs.step(u0, n)
    h = 1.0 / nx
    decay = (1.0 + dt * kappa * 8.0 / h ** 2 * np.sin(np.pi * h / 2) ** 2) ** (-n)
    assert float((u - decay * u0).abs().max()) <= 1e-11 * decay


def test_band_solve_matches_sparse_direct():
    """dfe_band_solve (tensor-core block TRSM) on M_L + dt K with a per-element kappa, a source
    term and non-zero Dirichlet data, many right-hand sides, against scipy's sparse LU of the same matrix."""
    import scipy.sparse as sp
    import scipy.sparse.linalg as spla
    from difffe_physics_lab_b200.timestepping import HeatStepper

    rng = np.random.default_rng(5)
    mesh = FEMesh.rectangle(24, 17, x_range=(0.0, 1.4), y_range=(-0.3, 0.5), bc_value=0.2)
    kap = np.exp(rng.uniform(np.log(0.05), 0.0, mesh.n_elements))
    f = torch.tensor(rng.uniform(-1, 1, mesh.n_nodes))
    dt = 5e-3
    hs = HeatStepper(mesh, kap, dt, f=f)
    B = 37
    u0 = torch.tensor(rng.uniform(-1, 1, (B, mesh.n_nodes)), device="cuda")
    u0[:, torch.tensor(list(mesh.dirichlet_nodes), device="cuda")] = 0.2
    u = hs.step(u0, 2).cpu().numpy()
    rp, col = hs.nm.csr(0)
    A = sp.csr_matrix((hs.A.cpu().numpy(), col, rp), shape=(mesh.n_nodes,) * 2)
    free = hs.free.cpu().numpy()
    lu = spla.splu(A[free][:, free].tocsc())
    g, mass, load = hs.g.cpu().numpy(), hs.mass.cpu().numpy(), hs.load.cpu().numpy()
    ref = u0.cpu().numpy()
    for _ in range(2):
        rhs = mass * ref + dt * load - (A @ g)
        nxt = np.tile(g, (B, 1))
        nxt[:, free] = lu.solve(rhs[:, free].T).T
        ref = nxt
    assert np.abs(u - ref).max() <= 1e-11 * np.abs(ref).max()
    # the lumped mass is the reference's load vector of f = 1: positive, sums to the area of the mesh
    assert mass.min() > 0 and abs(mass.sum() - 1.4 * 0.8) < 1e-12
