"""Heat rollouts with a source per sample (f (B, n)) or per step (source (N, n) / (B, N, n)): DifferentiableHeatSolver on
both kappa routes against a dense float64 rollout and torch autograd, the bit-level anchors of the source arithmetic, the
adjoint identity, invariance under checkpointing, launch splitting, batch splits and CTA size, 64-bit offsets, errors,
NaN isolation and the kernels that run."""
import zlib

import numpy as np
import pytest
import torch

from difffe_physics_lab_b200 import DifferentiableHeatSolver, _native
from tests.test_gpu_heat_per_sample import MESHES, _kernels, _mesh

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    _native.build()


# kappa routes: shared scalar, shared per-element field, one scalar per sample, one field per sample
ROUTES = ["scalar", "element", "ps_scalar", "ps_element"]
# f (B, n); source (N, n); source (B, N, n); constructor f (n,) together with source (B, N, n)
FORMS = ["f_B", "src_N", "src_BN", "f_and_src"]


def _kappa(rng, m, B, route):
    ne = m.n_elements
    shape = {"scalar": (1,), "element": (ne,), "ps_scalar": (B, 1), "ps_element": (B, ne)}[route]
    return torch.tensor(np.exp(rng.uniform(np.log(0.3), np.log(3.0), shape)))


def _sources(rng, m, B, N, form):
    """(f, source) of a form, float64 on the CPU"""
    n = m.n_nodes
    f = src = None
    if form == "f_B":
        f = torch.tensor(rng.uniform(-1, 1, (B, n)))
    if form == "f_and_src":
        f = torch.tensor(rng.uniform(-1, 1, n))
    if form == "src_N":
        src = torch.tensor(rng.uniform(-1, 1, (N, n)))
    if form in ("src_BN", "f_and_src"):
        src = torch.tensor(rng.uniform(-1, 1, (B, N, n)))
    return f, src


def _run(m, kap, dt, f, src, u0, N, every, W, checkpoint=None):
    """(U, dL/du0, dL/dkappa, dL/df, dL/dsource) of L = sum(W * U) on the GPU"""
    leaf = lambda t: None if t is None else t.detach().clone().cuda().requires_grad_(True)
    k, fs, ss, u = leaf(kap), leaf(f), leaf(src), leaf(u0)
    U = DifferentiableHeatSolver(m, k, dt, fs, checkpoint=checkpoint)(u, N, every=every, source=ss)
    (W.cuda() * U).sum().backward()
    return U.detach(), u.grad, k.grad, None if fs is None else fs.grad, None if ss is None else ss.grad


def _dense(m, kappa, dt, f, src, u0, N, every):
    """float64 CPU rollout, differentiable: K_b = sum_e kappa_{b,e} K0_e, the load F(q) per element area/3 * mean(q), step n
    with F(f) + F(source[n]); one LU factorisation per sample.  The states after steps every, ..., N as (B, N / every, n)"""
    nodes, el = m.nodes.to(torch.float64), m.elements
    n, ne, B = m.n_nodes, m.n_elements, u0.shape[0]
    x, y = nodes[el][..., 0], nodes[el][..., 1]
    area = 0.5 * ((x[:, 1] - x[:, 0]) * (y[:, 2] - y[:, 0]) - (x[:, 2] - x[:, 0]) * (y[:, 1] - y[:, 0])).abs()
    bb = torch.stack([y[:, 1] - y[:, 2], y[:, 2] - y[:, 0], y[:, 0] - y[:, 1]], 1)
    cc = torch.stack([x[:, 2] - x[:, 1], x[:, 0] - x[:, 2], x[:, 1] - x[:, 0]], 1)
    K0 = (bb[:, :, None] * bb[:, None, :] + cc[:, :, None] * cc[:, None, :]) / (4 * area)[:, None, None]
    kap = kappa.reshape(1, -1) if kappa.dim() == 1 else kappa
    kap = kap.expand(B, ne)
    idx = (el[:, :, None] * n + el[:, None, :]).reshape(-1)
    K = torch.zeros(B, n * n, dtype=torch.float64).index_add(1, idx, (kap[:, :, None, None] * K0).reshape(B, -1))
    K = K.reshape(B, n, n)
    M = torch.zeros(n, dtype=torch.float64).index_add(0, el.reshape(-1), (area / 3).repeat_interleave(3))

    def load(q):                                            # q (..., n) -> F(q) (..., n)
        t = (area / 3 * q[..., el].sum(-1) / 3).repeat_interleave(3, dim=-1)
        return torch.zeros(q.shape, dtype=torch.float64).index_add(q.dim() - 1, el.reshape(-1), t)

    A = torch.diag(M) + dt * K
    free = torch.tensor(m.free_nodes())
    D = torch.tensor(list(m.dirichlet_nodes.keys()))
    g = torch.zeros(n, dtype=torch.float64)
    g[D] = torch.tensor(list(m.dirichlet_nodes.values()), dtype=torch.float64)
    Aff, AfD = A[:, free][:, :, free], A[:, free][:, :, D]
    LU, piv = torch.linalg.lu_factor(Aff)
    lift = AfD @ g[D]
    Ff = torch.zeros(n, dtype=torch.float64) if f is None else load(f)
    u, out = u0, []
    for s in range(N):
        F = Ff if src is None else Ff + load(src[s] if src.dim() == 2 else src[:, s])
        rhs = M[free] * u[:, free] + dt * F[..., free] - lift
        nxt = g.repeat(B, 1)
        nxt[:, free] = torch.linalg.lu_solve(LU, piv, rhs[..., None])[..., 0]
        u = nxt
        if (s + 1) % every == 0:
            out.append(u)
    return torch.stack(out, 1)


def _rel(a, b):
    a, b = a.cpu(), b.cpu()
    return float((a - b).abs().max()) / max(float(b.abs().max()), 1e-300)


def _eq(a, b):
    return all((x is None and y is None) or torch.equal(x, y) for x, y in zip(a, b))


# ================================================================================================ 1. dense reference
@pytest.mark.parametrize("name", MESHES)
@pytest.mark.parametrize("route", ROUTES)
@pytest.mark.parametrize("form", FORMS)
def test_against_dense_reference(name, route, form):
    rng = np.random.default_rng(zlib.crc32(f"{name}/{route}/{form}".encode()))
    m = _mesh(name)
    B, N, every, dt = (2 if name == "r32x32" else 3), 6, 2, 2e-2
    kap = _kappa(rng, m, B, route)
    f, src = _sources(rng, m, B, N, form)
    u0 = torch.tensor(rng.uniform(-1, 1, (B, m.n_nodes)))
    W = torch.tensor(rng.standard_normal((B, N // every, m.n_nodes)))
    U, gu, gk, gf, gs = _run(m, kap, dt, f, src, u0, N, every, W)
    leaf = lambda t: None if t is None else t.clone().requires_grad_(True)
    kr, fr, sr, ur = leaf(kap), leaf(f), leaf(src), leaf(u0)
    Ur = _dense(m, kr, dt, fr, sr, ur, N, every)
    (W * Ur).sum().backward()
    assert _rel(U, Ur.detach()) <= 1e-12
    assert _rel(gu, ur.grad) <= 1e-10
    assert gk.shape == kap.shape and _rel(gk, kr.grad) <= 1e-10
    if f is not None:
        assert gf.shape == f.shape and _rel(gf, fr.grad) <= 1e-10
    if src is not None:
        assert gs.shape == src.shape and _rel(gs, sr.grad) <= 1e-10
        D = list(m.dirichlet_nodes.keys())                  # source values on Dirichlet nodes enter the free rows
        assert float(sr.grad[..., D].abs().max()) > 0
        assert float((gs[..., D].cpu() - sr.grad[..., D]).abs().max()) <= 1e-10 * float(sr.grad.abs().max())


# ===================================================================================================== 2. bit anchors
@pytest.mark.parametrize("route", ROUTES)
@pytest.mark.parametrize("name", ["r12x9_perturbed", "r33x3"])
def test_bit_anchors(route, name):
    rng = np.random.default_rng(7 + ROUTES.index(route))
    m = _mesh(name)
    B, N, dt = 4, 5, 1e-2
    kap = _kappa(rng, m, B, route)
    u0 = torch.tensor(rng.uniform(-1, 1, (B, m.n_nodes)))
    W = torch.tensor(rng.standard_normal((B, N, m.n_nodes)))
    f = torch.tensor(rng.uniform(-1, 1, m.n_nodes))
    # (a) a per-sample f whose rows all equal a shared f: the shared-f trajectory, bit for bit
    a = _run(m, kap, dt, f, None, u0, N, 1, W)
    b = _run(m, kap, dt, f.expand(B, -1).clone(), None, u0, N, 1, W)
    assert torch.equal(a[0], b[0])
    assert _rel(b[3].sum(0), a[3]) <= 1e-13
    # (b) source[n] == f for every n, no constructor f: the constructor-f trajectory, bit for bit
    c = _run(m, kap, dt, None, f.expand(N, -1).clone(), u0, N, 1, W)
    assert torch.equal(a[0], c[0])
    assert _rel(c[4].sum(0), a[3]) <= 1e-13
    # a (B, N, n) source with equal rows: the (N, n) source's states, bit for bit; its batch-summed gradient
    src = torch.tensor(rng.uniform(-1, 1, (N, m.n_nodes)))
    d = _run(m, kap, dt, f, src, u0, N, 1, W)
    e = _run(m, kap, dt, f, src.expand(B, -1, -1).clone(), u0, N, 1, W)
    assert torch.equal(d[0], e[0])
    assert _rel(e[4].sum(0), d[4]) <= 1e-13


# ================================================================================================ 3. adjoint identity
@pytest.mark.parametrize("route", ["element", "ps_element"])
def test_adjoint_identity_and_finite_differences(route):
    rng = np.random.default_rng(31 + ROUTES.index(route))
    m = _mesh("r12x4")
    B, N, dt = 3, 7, 2e-2
    kap = _kappa(rng, m, B, route)
    u0 = torch.tensor(rng.uniform(-1, 1, (B, m.n_nodes)))
    W = torch.tensor(rng.standard_normal((B, N, m.n_nodes)))
    f = torch.tensor(rng.uniform(-1, 1, (B, m.n_nodes)))

    def loss(f_, s_):
        with torch.no_grad():
            U = DifferentiableHeatSolver(m, kap.cuda(), dt, f_.cuda())(u0.cuda(), N, every=1, source=s_.cuda())
        return float((W.cuda() * U).sum())

    for shape in ((N, m.n_nodes), (B, N, m.n_nodes)):
        q = torch.tensor(rng.uniform(-1, 1, shape))
        _, _, _, gf, gq = _run(m, kap, dt, f, q, u0, N, 1, W)
        dq = torch.tensor(rng.standard_normal(shape))
        lhs, rhs = loss(f, q + dq) - loss(f, q), float((gq.cpu() * dq).sum())
        assert abs(lhs - rhs) <= 1e-10 * abs(rhs)
        h = 1e-3                                            # L is affine in f and q: central differences are exact
        for _ in range(3):
            i = tuple(int(rng.integers(0, s)) for s in shape)
            e = torch.zeros(shape, dtype=torch.float64)
            e[i] = h
            fd = (loss(f, q + e) - loss(f, q - e)) / (2 * h)
            assert abs(fd - float(gq[i])) <= 1e-7 * max(abs(float(gq[i])), float(gq.abs().max()) * 1e-3)
            j = (int(rng.integers(0, B)), int(rng.integers(0, m.n_nodes)))
            e = torch.zeros((B, m.n_nodes), dtype=torch.float64)
            e[j] = h
            fd = (loss(f + e, q) - loss(f - e, q)) / (2 * h)
            assert abs(fd - float(gf[j])) <= 1e-7 * max(abs(float(gf[j])), float(gf.abs().max()) * 1e-3)


# ======================================================================================================= 4. invariance
@pytest.mark.parametrize("route", ROUTES)
@pytest.mark.parametrize("form", FORMS)
def test_checkpointing_and_launch_splitting_are_bit_identical(route, form, monkeypatch):
    rng = np.random.default_rng(41 + ROUTES.index(route) + 10 * FORMS.index(form))
    m = _mesh("r8x10_lb")
    B, N, dt = 5, 12, 1e-2
    kap = _kappa(rng, m, B, route)
    f, src = _sources(rng, m, B, N, form)
    u0 = torch.tensor(rng.uniform(-1, 1, (B, m.n_nodes)))
    W = torch.tensor(rng.standard_normal((B, N // 2, m.n_nodes)))
    ref = _run(m, kap, dt, f, src, u0, N, 2, W)
    for c in (1, 3, N):
        assert _eq(_run(m, kap, dt, f, src, u0, N, 2, W, checkpoint=c), ref), c
    for steps in (1, 5):
        monkeypatch.setattr(DifferentiableHeatSolver, "_src_steps", steps)
        assert _eq(_run(m, kap, dt, f, src, u0, N, 2, W), ref), steps
        assert _eq(_run(m, kap, dt, f, src, u0, N, 2, W, checkpoint=3), ref), steps


@pytest.mark.parametrize("route", ROUTES)
def test_batch_splits_are_bit_identical(route):
    rng = np.random.default_rng(53 + ROUTES.index(route))
    m = _mesh("r12x9_perturbed")
    B, N, dt = 7, 4, 1e-2
    kap = _kappa(rng, m, B, route)
    f = torch.tensor(rng.uniform(-1, 1, (B, m.n_nodes)))
    src = torch.tensor(rng.uniform(-1, 1, (B, N, m.n_nodes)))
    u0 = torch.tensor(rng.uniform(-1, 1, (B, m.n_nodes)))
    W = torch.tensor(rng.standard_normal((B, N, m.n_nodes)))
    full = _run(m, kap, dt, f, src, u0, N, 1, W)
    per = route.startswith("ps")
    for lo, hi in ((0, 2), (2, 7), (4, 6)):            # (a single sample with 2-D kappa is the shared route by design)
        k = kap[lo:hi] if per else kap
        part = _run(m, k, dt, f[lo:hi], src[lo:hi], u0[lo:hi], N, 1, W[lo:hi])
        for t in (0, 1, 3, 4):
            assert torch.equal(part[t], full[t][lo:hi]), (lo, hi, t)
        if per:
            assert torch.equal(part[2], full[2][lo:hi])


@pytest.mark.parametrize("form", FORMS)
def test_cta_warps_are_bit_identical(form, monkeypatch):
    rng = np.random.default_rng(59 + FORMS.index(form))
    m = _mesh("r33x2")
    B, N, dt = 37, 5, 1e-2
    kap = _kappa(rng, m, B, "element")
    f, src = _sources(rng, m, B, N, form)
    u0 = torch.tensor(rng.uniform(-1, 1, (B, m.n_nodes)))
    W = torch.tensor(rng.standard_normal((B, N, m.n_nodes)))
    outs = []
    for w in (2, 4, 8):
        monkeypatch.setattr(DifferentiableHeatSolver, "_cta_warps", w)
        outs.append(_run(m, kap, dt, f, src, u0, N, 1, W))
    assert _eq(outs[0], outs[1]) and _eq(outs[0], outs[2])


# ============================================================================================================ 5. scale
def _sampled_rows(m, kap, dt, src, u0, N, every, W, U, gs, rows):
    """the dense reference of a few samples (rows are independent) against the GPU's rows"""
    sr = src[rows].clone().requires_grad_(True)
    Ur = _dense(m, kap, dt, None, sr, u0[rows], N, every)
    (W[rows] * Ur).sum().backward()
    assert _rel(U[rows], Ur.detach()) <= 1e-12
    assert _rel(gs[rows], sr.grad) <= 1e-10


@pytest.mark.parametrize("route", ["scalar", "ps_element"])
def test_batch_4096(route):
    rng = np.random.default_rng(61)
    m = _mesh("r32x32")
    B, N, dt = 4096, 4, 1e-2
    kap = _kappa(rng, m, B, route)
    src = torch.tensor(rng.uniform(-1, 1, (B, N, m.n_nodes)))
    u0 = torch.tensor(rng.uniform(-1, 1, (B, m.n_nodes)))
    W = torch.tensor(rng.standard_normal((B, N, m.n_nodes)))
    U, _, _, _, gs = _run(m, kap, dt, None, src, u0, N, 1, W)
    rows = [0, 1, 2047, 4095]
    _sampled_rows(m, kap[rows] if route.startswith("ps") else kap, dt, src, u0, N, 1, W, U.cpu(), gs.cpu(), rows)


def test_64_bit_offsets():
    """B * N * n_nodes > 2^31: every offset into the source, its constants, the trajectory and dL/dsource is 64-bit"""
    m = _mesh("r32x32")
    B, N, every, dt, c = 8192, 256, 64, 1e-2, 16
    assert B * N * m.n_nodes > 2 ** 31
    g = torch.Generator(device="cuda").manual_seed(5)
    src = torch.rand((B, N, m.n_nodes), dtype=torch.float64, device="cuda", generator=g).requires_grad_(True)
    u0 = torch.rand((B, m.n_nodes), dtype=torch.float64, device="cuda", generator=g)
    W = torch.randn((B, N // every, m.n_nodes), dtype=torch.float64, device="cuda", generator=g)
    kap = torch.tensor([0.7], dtype=torch.float64)
    U = DifferentiableHeatSolver(m, kap.cuda(), dt, checkpoint=c)(u0, N, every=every, source=src)
    (W * U).sum().backward()
    rows = [0, 4097, B - 1]
    Ur_src = src.detach()[rows].cpu()
    sr = Ur_src.clone().requires_grad_(True)
    Ur = _dense(m, kap, dt, None, sr, u0[rows].cpu(), N, every)
    (W[rows].cpu() * Ur).sum().backward()
    assert _rel(U.detach()[rows], Ur.detach()) <= 1e-12
    assert _rel(src.grad[rows], sr.grad) <= 1e-10


# ================================================================================================ 6. errors, isolation
def test_malformed_shapes_raise():
    m = _mesh("r12x4")
    n, B, N = m.n_nodes, 3, 4
    u0 = torch.zeros((B, n), dtype=torch.float64, device="cuda")
    z = lambda *s: torch.zeros(s, dtype=torch.float64, device="cuda")
    for f in (z(B + 1, n), z(B, n + 1), z(n + 1), z(1, B, n)):
        with pytest.raises(ValueError):
            DifferentiableHeatSolver(m, 1.0, 1e-2, f)(u0, N)
    with pytest.raises(ValueError):                          # a per-sample f needs a batched u0
        DifferentiableHeatSolver(m, 1.0, 1e-2, z(1, n))(u0[0], N)
    for s in (z(N + 1, n), z(N, n + 1), z(N * n), z(B + 1, N, n), z(B, N - 1, n), z(B, N, n - 1), z(1, B, N, n)):
        with pytest.raises(ValueError):
            DifferentiableHeatSolver(m, 1.0, 1e-2)(u0, N, source=s)
    with pytest.raises(ValueError):                          # a per-sample source needs a batched u0
        DifferentiableHeatSolver(m, 1.0, 1e-2)(u0[0], N, source=z(1, N, n))
    with pytest.raises(ValueError):
        DifferentiableHeatSolver(m, torch.ones((B, 1), dtype=torch.float64), 1e-2)(u0, N, source=z(B - 1, N, n))


@pytest.mark.parametrize("route", ["element", "ps_element"])
def test_nan_sample_is_isolated(route):
    rng = np.random.default_rng(67)
    m = _mesh("r12x9_perturbed")
    B, N, dt, j = 9, 6, 1e-2, 4
    kap = _kappa(rng, m, B, route)
    f = torch.tensor(rng.uniform(-1, 1, (B, m.n_nodes)))
    src = torch.tensor(rng.uniform(-1, 1, (B, N, m.n_nodes)))
    u0 = torch.tensor(rng.uniform(-1, 1, (B, m.n_nodes)))
    W = torch.tensor(rng.standard_normal((B, N, m.n_nodes)))
    ref = _run(m, kap, dt, f, src, u0, N, 1, W, checkpoint=2)
    bad = src.clone()
    bad[j, 2, m.free_nodes()[5]] = float("nan")
    got = _run(m, kap, dt, f, bad, u0, N, 1, W, checkpoint=2)
    keep = [b for b in range(B) if b != j]
    assert bool(torch.isnan(got[0][j]).any())
    for t in (0, 1, 3, 4):
        assert torch.equal(got[t][keep], ref[t][keep]), t
    if route.startswith("ps"):
        assert torch.equal(got[2][keep], ref[2][keep])


# ============================================================================================================ 7. routes
@pytest.mark.parametrize("route", ["element", "ps_element"])
def test_routes(route):
    rng = np.random.default_rng(71)
    m = _mesh("r12x4")
    B, N, dt = 5, 3, 1e-2
    kap = _kappa(rng, m, B, route).cuda()
    f = torch.tensor(rng.uniform(-1, 1, m.n_nodes), device="cuda")
    fB = torch.tensor(rng.uniform(-1, 1, (B, m.n_nodes)), device="cuda")
    src = torch.tensor(rng.uniform(-1, 1, (N, m.n_nodes)), device="cuda")
    u0 = torch.tensor(rng.uniform(-1, 1, (B, m.n_nodes)), device="cuda")

    def call(f_, s_):
        k = kap.clone().requires_grad_(True)
        ff = f_.clone().requires_grad_(True)
        ss = None if s_ is None else s_.clone().requires_grad_(True)
        DifferentiableHeatSolver(m, k, dt, ff)(u0, N, every=1, source=ss).sum().backward()

    base = _kernels(lambda: call(f, None))
    new = {"k_hsrc", "k_hsrc_tables"}
    assert not base & new
    assert _kernels(lambda: call(f, src)) == base | new
    assert new <= _kernels(lambda: call(fB, None))
