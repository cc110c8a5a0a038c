"""DifferentiableHeatSolver: backward-Euler rollouts in one kernel launch and their discrete adjoint in time."""
import numpy as np
import pytest
import torch

from difffe_physics_lab_b200 import DifferentiableHeatSolver, FEMesh, _native

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    _native.build()


def _dense_rollout(mesh, kappa, dt, f, u0, n_steps, every):
    """float64 CPU reference: K(kappa) = sum_e kappa_e K0_e and the lumped mass assembled with differentiable torch ops,
    torch.linalg.solve per step; returns the states after steps every, 2 every, ..., n_steps."""
    nodes, el = mesh.nodes.to(torch.float64), mesh.elements
    n, ne = mesh.n_nodes, mesh.n_elements
    x, y = nodes[el][..., 0], nodes[el][..., 1]
    area = 0.5 * ((x[:, 1] - x[:, 0]) * (y[:, 2] - y[:, 0]) - (x[:, 2] - x[:, 0]) * (y[:, 1] - y[:, 0])).abs()
    b = torch.stack([y[:, 1] - y[:, 2], y[:, 2] - y[:, 0], y[:, 0] - y[:, 1]], 1)
    c = torch.stack([x[:, 2] - x[:, 1], x[:, 0] - x[:, 2], x[:, 1] - x[:, 0]], 1)
    K0 = (b[:, :, None] * b[:, None, :] + c[:, :, None] * c[:, None, :]) / (4 * area)[:, None, None]
    kap = kappa.reshape(-1).expand(ne)
    rows, cols = el[:, :, None].expand(-1, 3, 3).reshape(-1), el[:, None, :].expand(-1, 3, 3).reshape(-1)
    K = torch.zeros(n * n, dtype=torch.float64).index_add(0, rows * n + cols, (kap[:, None, None] * K0).reshape(-1)).reshape(n, n)
    M = torch.zeros(n, dtype=torch.float64).index_add(0, el.reshape(-1), (area / 3).repeat_interleave(3))
    F = torch.zeros(n, dtype=torch.float64)
    if f is not None:
        F = F.index_add(0, el.reshape(-1), (area / 3 * f[el].sum(1) / 3).repeat_interleave(3))
    A = torch.diag(M) + dt * K
    free = torch.tensor(mesh.free_nodes())
    D = torch.tensor(list(mesh.dirichlet_nodes.keys()))
    g = torch.zeros(n, dtype=torch.float64)
    g[D] = torch.tensor(list(mesh.dirichlet_nodes.values()), dtype=torch.float64)
    Aff, AfD = A[free][:, free], A[free][:, D]
    u, out = u0, []
    for s in range(n_steps):
        rhs = M[free] * u[:, free] + dt * F[free] - AfD @ g[D]
        nxt = g.repeat(u.shape[0], 1)
        nxt[:, free] = torch.linalg.solve(Aff, rhs.T).T
        u = nxt
        if (s + 1) % every == 0:
            out.append(u)
    return torch.stack(out, 1)


def _grads(mesh, kappa, dt, f, u0, n_steps, every, W, checkpoint=None):
    """(U, dL/du0, dL/dkappa, dL/df) of L = sum(W * U) on the GPU."""
    k = kappa.detach().clone().cuda().requires_grad_(True)
    fs = None if f is None else f.detach().clone().cuda().requires_grad_(True)
    u = u0.detach().clone().cuda().requires_grad_(True)
    U = DifferentiableHeatSolver(mesh, k, dt, fs, checkpoint=checkpoint)(u, n_steps, every=every)
    (W.cuda() * U).sum().backward()
    return U.detach(), u.grad, k.grad, None if fs is None else fs.grad


def test_forward_matches_heat_stepper_and_every_slices():
    from difffe_physics_lab_b200.timestepping import HeatStepper

    rng = np.random.default_rng(5)
    mesh = FEMesh.rectangle(24, 17, x_range=(0.0, 1.4), y_range=(-0.3, 0.5), bc_value=0.2)
    kap = torch.tensor(np.exp(rng.uniform(np.log(0.05), 0.0, mesh.n_elements)))
    f = torch.tensor(rng.uniform(-1, 1, mesh.n_nodes))
    dt, B = 5e-3, 37
    hs = HeatStepper(mesh, kap, dt, f=f)
    u0 = torch.tensor(rng.uniform(-1, 1, (B, mesh.n_nodes)), device="cuda")
    u0[:, torch.tensor(list(mesh.dirichlet_nodes), device="cuda")] = 0.2
    solver = DifferentiableHeatSolver(mesh, kap.cuda(), dt, f.cuda())
    U = solver(u0, 10, every=1)
    assert U.shape == (B, 10, mesh.n_nodes)
    for s in (1, 2, 5):
        ref = hs.step(u0, s)
        assert float((U[:, s - 1] - ref).abs().max()) <= 1e-13 * float(ref.abs().max())
    for k in (2, 5, 10):
        assert torch.equal(solver(u0, 10, every=k), U[:, k - 1::k])
    assert torch.equal(solver(u0, 10), U[:, -1])
    assert torch.equal(solver(u0[3], 10), U[3, -1])
    assert torch.equal(solver(u0.cpu(), 10), U[:, -1].cpu())          # device policy: CPU in, CPU out


def test_closed_form_eigenmode():
    """u0 = phi = sin(pi x) sin(pi y) is an eigenvector of M_L^{-1} K on the uniform mesh: u_N = (1 + dt kappa mu)^-N phi."""
    nx, kappa, dt, N = 32, 1.3, 1e-3, 20
    mesh = FEMesh.rectangle(nx, nx)
    x, y = mesh.nodes[:, 0].cuda(), mesh.nodes[:, 1].cuda()
    phi = torch.sin(np.pi * x) * torch.sin(np.pi * y)
    k = torch.tensor(kappa, dtype=torch.float64, device="cuda", requires_grad=True)
    u0 = phi.clone().requires_grad_(True)
    (phi * DifferentiableHeatSolver(mesh, k, dt)(u0, N)).sum().backward()
    h = 1.0 / nx
    mu = 8.0 / h ** 2 * np.sin(np.pi * h / 2) ** 2
    r = 1.0 + dt * kappa * mu
    s2 = float((phi * phi).sum())
    gk = -N * dt * mu * r ** (-N - 1) * s2
    assert abs(float(k.grad) - gk) <= 1e-10 * abs(gk)
    free = torch.tensor(mesh.free_nodes(), device="cuda")
    ref = r ** (-N) * phi[free]
    assert float((u0.grad[free] - ref).abs().max()) <= 1e-10 * float(ref.abs().max())
    bc = torch.tensor(list(mesh.dirichlet_nodes), device="cuda")
    assert float(u0.grad[bc].abs().max()) == 0.0


@pytest.mark.parametrize("per_element", [False, True])
def test_against_dense_reference(per_element):
    rng = np.random.default_rng(11)
    mesh = FEMesh.rectangle(8, 6, x_range=(0.0, 1.2), y_range=(0.0, 0.9), bc_value=0.35)
    dt, N, every, B = 2e-2, 12, 3, 4
    kap = torch.tensor(np.exp(rng.uniform(-1.0, 0.5, mesh.n_elements)) if per_element else 0.8, dtype=torch.float64)
    f = torch.tensor(rng.uniform(-1, 1, mesh.n_nodes))
    u0 = torch.tensor(rng.uniform(-1, 1, (B, mesh.n_nodes)))
    W = torch.tensor(rng.standard_normal((B, N // every, mesh.n_nodes)))
    U, gu, gk, gf = _grads(mesh, kap, dt, f, u0, N, every, W)
    kr, fr, ur = kap.clone().requires_grad_(True), f.clone().requires_grad_(True), u0.clone().requires_grad_(True)
    Ur = _dense_rollout(mesh, kr, dt, fr, ur, N, every)
    (W * Ur).sum().backward()
    Ur = Ur.detach()
    assert float((U.cpu() - Ur).abs().max()) <= 1e-12 * float(Ur.abs().max())
    assert float((gk.cpu() - kr.grad).abs().sum()) <= 1e-10 * float(kr.grad.abs().sum())
    assert float((gu.cpu() - ur.grad).abs().max()) <= 1e-10 * float(ur.grad.abs().max())
    assert float((gf.cpu() - fr.grad).abs().max()) <= 1e-10 * float(fr.grad.abs().max())


def test_finite_differences():
    rng = np.random.default_rng(3)
    mesh = FEMesh.rectangle(8, 6, bc_value=-0.4)
    dt, N, B = 3e-2, 10, 3
    f = torch.tensor(rng.uniform(-1, 1, mesh.n_nodes), device="cuda")
    u0 = torch.tensor(rng.uniform(-1, 1, (B, mesh.n_nodes)), device="cuda")
    W = torch.tensor(rng.standard_normal((B, 5, mesh.n_nodes)), device="cuda")
    kap_e = torch.tensor(np.exp(rng.uniform(-1.0, 0.5, mesh.n_elements)), device="cuda")

    def loss(k, ff, uu):
        with torch.no_grad():
            return float((W * DifferentiableHeatSolver(mesh, k, dt, ff)(uu, N, every=2)).sum())

    def check(analytic, fd):
        assert abs(analytic - fd) <= 1e-6 * max(abs(fd), 1e-12), (analytic, fd)

    # scalar kappa
    k = torch.tensor(0.9, dtype=torch.float64, device="cuda", requires_grad=True)
    (W * DifferentiableHeatSolver(mesh, k, dt, f)(u0, N, every=2)).sum().backward()
    eps = 1e-6
    check(float(k.grad), (loss(k.detach() + eps, f, u0) - loss(k.detach() - eps, f, u0)) / (2 * eps))
    # random directions in per-element kappa, u0 and f
    ke, fs, us = kap_e.clone().requires_grad_(True), f.clone().requires_grad_(True), u0.clone().requires_grad_(True)
    (W * DifferentiableHeatSolver(mesh, ke, dt, fs)(us, N, every=2)).sum().backward()
    for t in range(2):
        dk = torch.tensor(rng.standard_normal(mesh.n_elements), device="cuda") * kap_e * 1e-6
        check(float((ke.grad * dk).sum()), (loss(kap_e + dk, f, u0) - loss(kap_e - dk, f, u0)) / 2)
        du = torch.tensor(rng.standard_normal(u0.shape), device="cuda") * 1e-6
        check(float((us.grad * du).sum()), (loss(kap_e, f, u0 + du) - loss(kap_e, f, u0 - du)) / 2)
        df = torch.tensor(rng.standard_normal(f.shape), device="cuda") * 1e-6
        check(float((fs.grad * df).sum()), (loss(kap_e, f + df, u0) - loss(kap_e, f - df, u0)) / 2)


def test_checkpointing_is_bit_identical():
    rng = np.random.default_rng(7)
    mesh = FEMesh.rectangle(12, 9, bc_value=0.1)
    dt, N, B = 1e-2, 20, 5
    kap = torch.tensor(np.exp(rng.uniform(-1.0, 0.5, mesh.n_elements)))
    f = torch.tensor(rng.uniform(-1, 1, mesh.n_nodes))
    u0 = torch.tensor(rng.uniform(-1, 1, (B, mesh.n_nodes)))
    for every in (1, 4):
        W = torch.tensor(rng.standard_normal((B, N // every, mesh.n_nodes)))
        ref = _grads(mesh, kap, dt, f, u0, N, every, W, checkpoint=None)
        for c in (1, 3, 7, 20, 50):
            got = _grads(mesh, kap, dt, f, u0, N, every, W, checkpoint=c)
            for a, b in zip(ref, got):
                assert torch.equal(a, b), (every, c)


def test_determinism_and_batch_consistency():
    rng = np.random.default_rng(9)
    mesh = FEMesh.rectangle(8, 6, bc_value=0.25)
    dt, N = 2e-2, 4
    kap = torch.tensor(np.exp(rng.uniform(-1.0, 0.5, mesh.n_elements)))
    f = torch.tensor(rng.uniform(-1, 1, mesh.n_nodes))
    # two identical calls
    B = 21
    u0 = torch.tensor(rng.uniform(-1, 1, (B, mesh.n_nodes)))
    W = torch.tensor(rng.standard_normal((B, N, mesh.n_nodes)))
    a, b = _grads(mesh, kap, dt, f, u0, N, 1, W), _grads(mesh, kap, dt, f, u0, N, 1, W)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    # a batch against single-state calls: states bit for bit, summed gradients to 1e-13
    gk_sum, gf_sum = torch.zeros_like(a[2]), torch.zeros_like(a[3])
    for i in range(B):
        s = _grads(mesh, kap, dt, f, u0[i:i + 1], N, 1, W[i:i + 1])
        assert torch.equal(s[0], a[0][i:i + 1])
        assert float((s[1] - a[1][i:i + 1]).abs().max()) <= 1e-13 * float(a[1].abs().max())
        gk_sum += s[2]
        gf_sum += s[3]
    assert float((gk_sum - a[2]).abs().sum()) <= 1e-13 * float(a[2].abs().sum())
    assert float((gf_sum - a[3]).abs().max()) <= 1e-13 * float(a[3].abs().max())


def test_cta_size_thresholds():
    """The rollout kernels choose warps per CTA from B; per-sample arithmetic must not depend on it."""
    rng = np.random.default_rng(13)
    mesh = FEMesh.rectangle(8, 6, bc_value=0.25)
    dt, N = 2e-2, 3
    kap = torch.tensor(0.7, dtype=torch.float64)
    L = _native.lib()
    h = mesh._native(torch.cuda.current_device()).handle
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    Bs = []
    for w in (4, 8):        # first B whose grid of 16 w states per CTA covers every SM
        t = 16 * w * (sm - 1) + 1
        assert L.dfe_heat_warps(h, t - 1) < w <= L.dfe_heat_warps(h, t)
        Bs += [t - 1, t]
    assert L.dfe_heat_warps(h, 1) == 2
    for B in Bs:
        u0 = torch.tensor(rng.uniform(-1, 1, (B, mesh.n_nodes)), device="cuda")
        U = DifferentiableHeatSolver(mesh, kap, dt)(u0, N, every=1)
        for i in (0, 1, B // 2, B - 1):
            assert torch.equal(DifferentiableHeatSolver(mesh, kap, dt)(u0[i:i + 1], N, every=1), U[i:i + 1])
        try:                # every CTA size gives the same bits
            for w in (2, 4, 8):
                DifferentiableHeatSolver._cta_warps = w
                assert torch.equal(DifferentiableHeatSolver(mesh, kap, dt)(u0, N, every=1), U)
        finally:
            DifferentiableHeatSolver._cta_warps = 0


def test_errors():
    mesh = FEMesh.rectangle(8, 6)
    u0 = torch.zeros(mesh.n_nodes, device="cuda")
    with pytest.raises(_native.BreakdownError):
        DifferentiableHeatSolver(mesh, -1.0, 1e-2)(u0, 3)
    with pytest.raises(NotImplementedError):
        DifferentiableHeatSolver(mesh.to_p2(), 1.0, 1e-2)
    with pytest.raises(NotImplementedError):
        DifferentiableHeatSolver(FEMesh.rectangle(40, 8), 1.0, 1e-2)
    with pytest.raises(NotImplementedError):
        DifferentiableHeatSolver(FEMesh.line(20), 1.0, 1e-2)
    with pytest.raises(ValueError):
        DifferentiableHeatSolver(mesh, 1.0, 1e-2)(u0, 10, every=3)
