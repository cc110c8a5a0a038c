"""Heat rollouts with one conductivity per sample: DifferentiableHeatSolver with kappa (B, 1) or (B, n_el), the
dfe_heat_ps_* kernels (dfe_heat.cu), against the shared-kappa operator bit for bit, a dense float64 rollout, the shared route
row by row, finite differences, and itself across batch splits and checkpointing."""
import re

import numpy as np
import pytest
import torch

from difffe_physics_lab_b200 import DifferentiableHeatSolver, FEMesh, _native
from difffe_physics_lab_b200.timestepping import _HeatOperator
from tests.test_gpu_band_edges import CASES, _grid, _seed

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    _native.build()


# one block row with 31 padding rows, one full block row, padding in the last block, half bandwidth 32, one-warp-sized
# meshes with partial Dirichlet sets, jittered coordinates, and the 32 x 32 benchmark mesh
MESHES = ["r32x32", "r2x2", "r33x2", "r12x4", "r33x3", "r6x6_left", "r8x10_lb", "r12x9_perturbed"]
_cache = {}


def _mesh(name):
    if name not in _cache:
        _cache[name] = _grid(32, 32, seed=1) if name == "r32x32" else _grid(*CASES[name][0], seed=_seed(name))
    return _cache[name]


def _kappa(rng, m, B, per_element):
    """per-element fields log-uniform over [0.3, 3]; per-sample values log-uniform over [0.1, 10]"""
    if per_element:
        return torch.tensor(np.exp(rng.uniform(np.log(0.3), np.log(3.0), (B, m.n_elements))))
    return torch.tensor(np.exp(rng.uniform(np.log(0.1), np.log(10.0), (B, 1))))


def _inputs(rng, m, B, N, every):
    f = torch.tensor(rng.uniform(-1, 1, m.n_nodes))
    u0 = torch.tensor(rng.uniform(-1, 1, (B, m.n_nodes)))
    W = torch.tensor(rng.standard_normal((B, N // every, m.n_nodes)))
    return f, u0, W


def _run(m, kap, dt, f, u0, N, every, W, checkpoint=None):
    """(U, dL/du0, dL/dkappa, dL/df) of L = sum(W * U) on the GPU"""
    k = kap.detach().clone().cuda().requires_grad_(True)
    fs = None if f is None else f.detach().clone().cuda().requires_grad_(True)
    u = u0.detach().clone().cuda().requires_grad_(True)
    U = DifferentiableHeatSolver(m, k, dt, fs, checkpoint=checkpoint)(u, N, every=every)
    (W.cuda() * U).sum().backward()
    return U.detach(), u.grad, k.grad, None if fs is None else fs.grad


def _dense_ps(m, kappa, dt, f, u0, N, every):
    """float64 CPU reference with one K_b = sum_e kappa_{b,e} K0_e per sample (differentiable torch ops, batched
    torch.linalg.solve per step); the states after steps every, 2 every, ..., N as (B, N / every, n)"""
    nodes, el = m.nodes.to(torch.float64), m.elements
    n, ne, B = m.n_nodes, m.n_elements, u0.shape[0]
    x, y = nodes[el][..., 0], nodes[el][..., 1]
    area = 0.5 * ((x[:, 1] - x[:, 0]) * (y[:, 2] - y[:, 0]) - (x[:, 2] - x[:, 0]) * (y[:, 1] - y[:, 0])).abs()
    bb = torch.stack([y[:, 1] - y[:, 2], y[:, 2] - y[:, 0], y[:, 0] - y[:, 1]], 1)
    cc = torch.stack([x[:, 2] - x[:, 1], x[:, 0] - x[:, 2], x[:, 1] - x[:, 0]], 1)
    K0 = (bb[:, :, None] * bb[:, None, :] + cc[:, :, None] * cc[:, None, :]) / (4 * area)[:, None, None]
    kap = kappa.expand(B, ne)
    idx = (el[:, :, None] * n + el[:, None, :]).reshape(-1)
    K = torch.zeros(B, n * n, dtype=torch.float64).index_add(1, idx, (kap[:, :, None, None] * K0).reshape(B, -1))
    K = K.reshape(B, n, n)
    M = torch.zeros(n, dtype=torch.float64).index_add(0, el.reshape(-1), (area / 3).repeat_interleave(3))
    F = torch.zeros(n, dtype=torch.float64)
    if f is not None:
        F = F.index_add(0, el.reshape(-1), (area / 3 * f[el].sum(1) / 3).repeat_interleave(3))
    A = torch.diag(M) + dt * K
    free = torch.tensor(m.free_nodes())
    D = torch.tensor(list(m.dirichlet_nodes.keys()))
    g = torch.zeros(n, dtype=torch.float64)
    g[D] = torch.tensor(list(m.dirichlet_nodes.values()), dtype=torch.float64)
    Aff, AfD = A[:, free][:, :, free], A[:, free][:, :, D]
    u, out = u0, []
    for s in range(N):
        rhs = M[free] * u[:, free] + dt * F[free] - AfD @ g[D]
        nxt = g.repeat(B, 1)
        nxt[:, free] = torch.linalg.solve(Aff, rhs)
        u = nxt
        if (s + 1) % every == 0:
            out.append(u)
    return torch.stack(out, 1)


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {mm.group(1) for e in prof.events() for mm in [re.search(r"(k_\w+)", e.name)] if mm}


def _abi(m, kap, dt, f, u0, N, gbar):
    """dfe_heat_ps_setup / _fwd / _adj / _grad / _grad_sum called directly: (A, factors, c_free, status, traj, lam_1, gk)"""
    L = _native.lib()
    dev = torch.device("cuda", torch.cuda.current_device())
    nm = m._native(dev.index)
    h, B = nm.handle, kap.shape[0]
    st = torch.cuda.current_stream().cuda_stream
    op = _HeatOperator(m, kap[0], dt, f, dev)                     # mass and load do not depend on kappa
    mode = _native.KAPPA_PER_SAMPLE if kap.shape[1] == 1 else _native.KAPPA_PER_SAMPLE_ELEMENT
    kd = kap.cuda().contiguous()
    npad, nf = op.npad, op.free.numel()
    fac = torch.empty(L.dfe_heat_ps_factor_bytes(h, B) // 8, dtype=torch.float64, device=dev)
    ws = torch.empty(L.dfe_heat_ps_workspace_bytes(h, B), dtype=torch.uint8, device=dev)
    cf = torch.empty((B, npad), dtype=torch.float64, device=dev)
    status = torch.full((B,), -1, dtype=torch.int32, device=dev)
    _native.check(L.dfe_heat_ps_setup(h, B, kd.data_ptr(), mode, dt, op.mass.data_ptr(),
                                      None if f is None else op.load.data_ptr(), fac.data_ptr(), cf.data_ptr(),
                                      status.data_ptr(), ws.data_ptr(), ws.numel(), st))
    A = ws[:B * nm.info.nnz_full * 8].view(torch.float64).reshape(B, -1).clone()
    mf = torch.zeros(npad, dtype=torch.float64, device=dev)
    mf[:nf] = op.mass_free
    X = torch.zeros((B, npad), dtype=torch.float64, device=dev)
    traj = torch.empty((B, N, m.n_nodes), dtype=torch.float64, device=dev)
    u = u0.cuda().contiguous()
    _native.check(L.dfe_heat_ps_fwd(h, B, N, u.data_ptr(), u.stride(0), fac.data_ptr(), mf.data_ptr(), cf.data_ptr(),
                                    X.data_ptr(), traj.data_ptr(), traj.stride(0), traj.stride(1), st))
    gb = gbar.cuda().contiguous()
    Xa = torch.zeros_like(X)
    lsum = torch.zeros_like(X)
    lam = torch.empty((N, B, npad), dtype=torch.float64, device=dev)
    _native.check(L.dfe_heat_ps_adj(h, B, 0, N, gb.data_ptr(), gb.stride(0), gb.stride(1), 1, fac.data_ptr(),
                                    mf.data_ptr(), Xa.data_ptr(), lam.data_ptr(), lsum.data_ptr(), st))
    gacc = torch.zeros((B, m.n_elements), dtype=torch.float64, device=dev)
    _native.check(L.dfe_heat_ps_grad(h, B, N, fac.data_ptr(), traj.data_ptr(), traj.stride(0), traj.stride(1),
                                     lam.data_ptr(), gacc.data_ptr(), st))
    gk = torch.empty(tuple(kap.shape) if mode == _native.KAPPA_PER_SAMPLE_ELEMENT else (B,), dtype=torch.float64,
                     device=dev)
    _native.check(L.dfe_heat_ps_grad_sum(h, B, dt, mode, gacc.data_ptr(), gk.data_ptr(), st))
    torch.cuda.synchronize()
    return A, fac, cf, status, traj, Xa, gk, op


def _rel(a, b):
    return float((a - b).abs().max()) / max(float(b.abs().max()), 1e-300)


# ======================================================================================================== A. operator
@pytest.mark.parametrize("name", MESHES)
@pytest.mark.parametrize("per_element", [False, True])
def test_operator_bits(name, per_element):
    rng = np.random.default_rng(_seed(name) + per_element)
    m = _mesh(name)
    B, dt = 5, 7e-3
    kap = _kappa(rng, m, B, per_element)
    f = torch.tensor(rng.uniform(-1, 1, m.n_nodes), device="cuda")
    u0 = torch.tensor(rng.uniform(-1, 1, (B, m.n_nodes)))
    A, fac, cf, status, _, _, _, op0 = _abi(m, kap, dt, f, u0, 2, torch.zeros(B, 2, m.n_nodes))
    assert int(status.abs().max()) == 0
    ne, npad, nf = m.n_elements, op0.npad, op0.free.numel()
    per = npad * 33
    dev = torch.device("cuda", torch.cuda.current_device())
    for b in range(B):
        op = _HeatOperator(m, kap[b].cuda(), dt, f, dev)
        assert torch.equal(A[b], op.A), b
        assert torch.equal(fac[10 * ne + b * per:10 * ne + (b + 1) * per], op.factor.view(torch.float64)[:per]), b
        c = op.rhs_const
        assert float((cf[b, :nf] - c).abs().max()) <= 1e-15 * max(float(c.abs().max()), 1e-300), b
        assert float(cf[b, nf:].abs().max() if npad > nf else 0.0) == 0.0


# ================================================================================================ B. dense reference
@pytest.mark.parametrize("name", MESHES)
@pytest.mark.parametrize("per_element", [False, True])
@pytest.mark.parametrize("every", [1, 3])
def test_against_dense_reference(name, per_element, every):
    rng = np.random.default_rng(_seed(name) + 10 * every + per_element)
    m = _mesh(name)
    B, N, dt = (2 if name == "r32x32" else 3), 12, 2e-2
    kap = _kappa(rng, m, B, per_element)
    f, u0, W = _inputs(rng, m, B, N, every)
    U, gu, gk, gf = _run(m, kap, dt, f, u0, N, every, W)
    kr, fr, ur = kap.clone().requires_grad_(True), f.clone().requires_grad_(True), u0.clone().requires_grad_(True)
    Ur = _dense_ps(m, kr, dt, fr, ur, N, every)
    (W * Ur).sum().backward()
    assert _rel(U.cpu(), Ur.detach()) <= 1e-12
    assert gk.shape == kap.shape
    for b in range(B):
        assert float((gk[b].cpu() - kr.grad[b]).abs().sum()) <= 1e-10 * float(kr.grad[b].abs().sum()), b
    assert _rel(gu.cpu(), ur.grad) <= 1e-10
    assert _rel(gf.cpu(), fr.grad) <= 1e-10


# ============================================================================================= C. against shared route
@pytest.mark.parametrize("name", MESHES)
@pytest.mark.parametrize("per_element", [False, True])
def test_rows_match_shared_route(name, per_element):
    rng = np.random.default_rng(_seed(name) + 100 + per_element)
    m = _mesh(name)
    B, N, every, dt = 6, 8, 2, 1e-2
    kap = _kappa(rng, m, B, per_element)
    f, u0, W = _inputs(rng, m, B, N, every)
    U, gu, gk, gf = _run(m, kap, dt, f, u0, N, every, W)
    gf_sum = torch.zeros_like(gf)
    for b in range(B):
        Ub, gub, gkb, gfb = _run(m, kap[b].reshape(-1), dt, f, u0[b:b + 1], N, every, W[b:b + 1])
        assert _rel(U[b:b + 1], Ub) <= 1e-13, b
        assert _rel(gu[b:b + 1], gub) <= 1e-12, b
        assert float((gk[b] - gkb).abs().sum()) <= 1e-12 * float(gkb.abs().sum()), b
        gf_sum += gfb
    assert _rel(gf, gf_sum) <= 1e-12


def test_rows_match_shared_route_at_4096():
    rng = np.random.default_rng(4096)
    m = _mesh("r32x32")
    B, N, dt = 4096, 5, 1e-2
    kap = _kappa(rng, m, B, True)
    f, u0, W = _inputs(rng, m, B, N, 1)
    U, gu, gk, _ = _run(m, kap, dt, f, u0, N, 1, W)
    for b in (0, B // 2, B - 1):
        Ub, gub, gkb, _ = _run(m, kap[b], dt, f, u0[b:b + 1], N, 1, W[b:b + 1])
        assert _rel(U[b:b + 1], Ub) <= 1e-13, b
        assert _rel(gu[b:b + 1], gub) <= 1e-12, b
        assert float((gk[b] - gkb).abs().sum()) <= 1e-12 * float(gkb.abs().sum()), b


# =============================================================================================== D. bit for bit
@pytest.mark.parametrize("name", ["r32x32", "r6x6_left", "r12x9_perturbed"])
@pytest.mark.parametrize("per_element", [False, True])
def test_batch_splits_are_bit_identical(name, per_element):
    """Through the ABI: a batch of 1 has the shape of a shared kappa ((1, 1) / (1, n_el)) at the Python level."""
    rng = np.random.default_rng(_seed(name) + 200 + per_element)
    m = _mesh(name)
    B, N, dt = 40, 6, 1e-2
    kap = _kappa(rng, m, B, per_element)
    f, u0, W = _inputs(rng, m, B, N, 1)
    fc = f.cuda()
    ref = _abi(m, kap, dt, fc, u0, N, W)
    ne, per = m.n_elements, ref[7].npad * 33
    for size in (1, 2, 37):
        for s in range(0, B, size):
            e = min(s + size, B)
            got = _abi(m, kap[s:e], dt, fc, u0[s:e], N, W[s:e])
            for t in (0, 2, 3, 4, 5, 6):                        # A, c_free, status, trajectory, lambda_1, dL/dkappa
                assert torch.equal(got[t], ref[t][s:e]), (size, s, t)
            assert torch.equal(got[1][10 * ne:], ref[1][10 * ne + s * per:10 * ne + e * per]), (size, s)
    # through the solver: two identical calls agree, and a split into two halves gives the same rows
    a, b = _run(m, kap, dt, f, u0, N, 2, W[:, 1::2]), _run(m, kap, dt, f, u0, N, 2, W[:, 1::2])
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    for s in (0, B // 2):
        h = _run(m, kap[s:s + B // 2], dt, f, u0[s:s + B // 2], N, 2, W[s:s + B // 2, 1::2])
        for x, y in zip(a[:3], h[:3]):                          # dL/df is summed over the batch
            assert torch.equal(x[s:s + B // 2], y), s


@pytest.mark.parametrize("per_element", [False, True])
def test_checkpointing_is_bit_identical(per_element):
    rng = np.random.default_rng(300 + per_element)
    m = _mesh("r12x9_perturbed")
    B, N, dt = 5, 20, 1e-2
    kap = _kappa(rng, m, B, per_element)
    for every in (1, 4):
        f, u0, W = _inputs(rng, m, B, N, every)
        ref = _run(m, kap, dt, f, u0, N, every, W)
        for c in (1, 3, 7, N, 2 * N):
            got = _run(m, kap, dt, f, u0, N, every, W, checkpoint=c)
            for x, y in zip(ref, got):
                assert torch.equal(x, y), (every, c)


# ============================================================================================ E. finite differences
def test_finite_differences():
    rng = np.random.default_rng(3)
    m = FEMesh.rectangle(8, 6, bc_value=-0.4)
    dt, N, B = 3e-2, 10, 3
    f = torch.tensor(rng.uniform(-1, 1, m.n_nodes), device="cuda")
    u0 = torch.tensor(rng.uniform(-1, 1, (B, m.n_nodes)), device="cuda")
    W = torch.tensor(rng.standard_normal((B, 5, m.n_nodes)), device="cuda")
    kap_e = torch.tensor(np.exp(rng.uniform(-1.0, 0.5, (B, m.n_elements))), device="cuda")
    kap_s = torch.tensor(np.exp(rng.uniform(-1.0, 0.5, (B, 1))), device="cuda")

    def loss(k, ff, uu):
        with torch.no_grad():
            return float((W * DifferentiableHeatSolver(m, k, dt, ff)(uu, N, every=2)).sum())

    def check(analytic, fd):
        assert abs(analytic - fd) <= 1e-6 * max(abs(fd), 1e-12), (analytic, fd)

    for kap in (kap_e, kap_s):
        ke, fs, us = kap.clone().requires_grad_(True), f.clone().requires_grad_(True), u0.clone().requires_grad_(True)
        (W * DifferentiableHeatSolver(m, ke, dt, fs)(us, N, every=2)).sum().backward()
        for _ in range(2):
            dk = torch.tensor(rng.standard_normal(tuple(kap.shape)), device="cuda") * kap * 1e-6
            check(float((ke.grad * dk).sum()), (loss(kap + dk, f, u0) - loss(kap - dk, f, u0)) / 2)
            du = torch.tensor(rng.standard_normal(u0.shape), device="cuda") * 1e-6
            check(float((us.grad * du).sum()), (loss(kap, f, u0 + du) - loss(kap, f, u0 - du)) / 2)
            df = torch.tensor(rng.standard_normal(f.shape), device="cuda") * 1e-6
            check(float((fs.grad * df).sum()), (loss(kap, f + df, u0) - loss(kap, f - df, u0)) / 2)


# ======================================================================================================= F. errors
def test_errors():
    m = _mesh("r8x10_lb")
    ne, B = m.n_elements, 8
    u0 = torch.zeros((B, m.n_nodes), device="cuda")
    kap = torch.ones((B, ne), dtype=torch.float64, device="cuda")
    kap[3] = -10.0
    kap[5] = -5.0
    with pytest.raises(_native.BreakdownError, match="sample 3"):
        DifferentiableHeatSolver(m, kap, 1e-2)(u0, 3)
    ok = torch.ones((B, ne), dtype=torch.float64)
    with pytest.raises(ValueError):
        DifferentiableHeatSolver(m, ok, 1e-2)(u0[:B - 1], 3)                 # mismatched B
    with pytest.raises(ValueError):
        DifferentiableHeatSolver(m, torch.ones((B, ne + 1), dtype=torch.float64), 1e-2)(u0, 3)
    with pytest.raises(ValueError):
        DifferentiableHeatSolver(m, ok, 1e-2)(u0[0], 3)                      # un-batched u0
    with pytest.raises(ValueError):
        DifferentiableHeatSolver(m, torch.ones((B, 1), dtype=torch.float64), 1e-2)(u0[0], 3)
    with pytest.raises(NotImplementedError):                                 # half bandwidth 33
        DifferentiableHeatSolver(FEMesh.rectangle(34, 20), torch.ones((B, 1), dtype=torch.float64), 1e-2)


def test_shared_2d_forms_keep_the_shared_route():
    rng = np.random.default_rng(17)
    m = _mesh("r12x4")
    B, N, dt = 4, 5, 1e-2
    f, u0, W = _inputs(rng, m, B, N, 1)
    ke = torch.tensor(np.exp(rng.uniform(-1, 1, m.n_elements)))
    ks = torch.tensor(1.7, dtype=torch.float64)
    for flat, wide in ((ke, ke.reshape(1, -1)), (ks, ks.reshape(1, 1))):
        a, b = _run(m, flat, dt, f, u0, N, 1, W), _run(m, wide, dt, f, u0, N, 1, W)
        for x, y in zip(a, b):
            assert torch.equal(x, y.reshape(x.shape))
        assert b[2].shape == wide.shape
    fn = lambda: DifferentiableHeatSolver(m, ke.reshape(1, -1).cuda(), dt, f.cuda())(u0.cuda(), N)
    k = _kernels(fn)
    assert "k_heat_roll" in k and not any(x.startswith("k_hps") for x in k)


# ==================================================================================================== G. isolation
@pytest.mark.parametrize("per_element", [False, True])
def test_nan_sample_is_isolated(per_element):
    rng = np.random.default_rng(23 + per_element)
    m = _mesh("r12x9_perturbed")
    B, N, dt, j = 9, 4, 1e-2, 4
    kap = _kappa(rng, m, B, per_element)
    f, u0, gbar = _inputs(rng, m, B, N, 1)
    ref = _abi(m, kap, dt, f.cuda(), u0, N, gbar)
    bad = kap.clone()
    bad[j, kap.shape[1] // 2] = float("nan")                     # an interior element: it reaches K_free
    got = _abi(m, bad, dt, f.cuda(), u0, N, gbar)
    assert int(ref[3].abs().max()) == 0
    st = got[3].cpu()
    assert int(st[j]) != 0 and int(st.abs().sum()) == int(st[j].abs())
    ne, per = m.n_elements, ref[7].npad * 33
    keep = [b for b in range(B) if b != j]
    for b in keep:
        assert torch.equal(got[1][10 * ne + b * per:10 * ne + (b + 1) * per], ref[1][10 * ne + b * per:10 * ne + (b + 1) * per])
    for t in (0, 2, 4, 5, 6):                                       # c_free, trajectory, lambda_1, dL/dkappa
        assert torch.equal(got[t][keep], ref[t][keep]), t


# ======================================================================================================== H. routes
def test_routes():
    rng = np.random.default_rng(29)
    m = _mesh("r12x4")
    B, N, dt = 5, 3, 1e-2
    f, u0, W = _inputs(rng, m, B, N, 1)
    kap = _kappa(rng, m, B, True).cuda()

    def ps():
        k = kap.clone().requires_grad_(True)
        (W.cuda() * DifferentiableHeatSolver(m, k, dt, f.cuda())(u0.cuda(), N, every=1)).sum().backward()

    def shared():
        k = kap[0].clone().requires_grad_(True)
        (W.cuda() * DifferentiableHeatSolver(m, k, dt, f.cuda())(u0.cuda(), N, every=1)).sum().backward()

    new = {"k_hps_roll", "k_hps_grad", "k_hps_gsum", "k_hps_shift", "k_hps_cfree", "k_bps_assemble", "k_bps_factor"}
    k = _kernels(ps)
    assert new <= k and "k_heat_roll" not in k and "k_heat_grad" not in k
    k = _kernels(shared)
    assert "k_heat_roll" in k and "k_heat_grad" in k and not (new & k)
