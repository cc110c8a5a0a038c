"""The one-CTA-per-sample batched Jacobi-PCG kernel at every unroll width and mesh shape it accepts, against float64 references.

`k_batch<BWD, RPT>` (dfe_batch.cu, behind dfe_batch_fwd / dfe_batch_bwd) keeps K_free in SELL-32 form in shared memory.
Each warp owns RPT slices of 32 rows, and `dispatch` picks RPT from ceil(n_slices / 8): 1, 2, 3, 4, 6, 6, 8, 8.  Every
RPT is a separately unrolled kernel.  The cases below reach each of these buckets.  They also reach slices wider than the
unrolled SELL loop (WMAX = 8: nodes with 8 neighbours on a mesh with flipped quad diagonals), the 1-D branches of the
load and of the gradients, a permuted node numbering, partial Dirichlet sides with varying data, and a zero-area
triangle.  The tests compare the kernel with the float64 oracle.  They check that a sample's bits do not depend on where
it sits in the batch, that results scale exactly with powers of two (the kernel scales each right-hand side so that its
largest entry lies in [1, 2)), and that status arrays, strided rows and the support predicate behave as documented.
"""
import re

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla
import torch

from difffe_physics_lab_b200 import _native
from diffhe.mesh import FEMesh
from diffhe.solver import DifferentiableFESolver
from oracle import oracle as O
from tests.test_gpu_band_edges import _grid
from tests.test_gpu_parity import TOL2D, abi_assemble, oracle_run, relerr, run

pytestmark = pytest.mark.gpu

BNW = 8      # warps per CTA of k_batch (BT / 32)
WMAX = 8     # SELL slice widths up to WMAX take the unrolled loop
TOL = 1e-13  # DifferentiableFESolver's default pcg_tol


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    _native.build()


def _permuted(nx, ny, seed):
    """rectangle(nx, ny) with randomly renumbered nodes; the Dirichlet dict keeps the rectangle's order, so the lifting
    runs in an order that is not ascending in node id."""
    rng = np.random.default_rng(seed)
    m = FEMesh.rectangle(nx, ny, x_range=(-0.5, 0.8), y_range=(0.0, 1.1))
    perm = rng.permutation(m.n_nodes)                        # old id -> new id
    nodes = np.empty_like(m.nodes.numpy())
    nodes[perm] = m.nodes.numpy()
    x, y = m.nodes.numpy().T
    bc = {int(perm[p]): 0.1 + 0.3 * x[p] * y[p] for p in m.dirichlet_nodes}
    return FEMesh(nodes=torch.from_numpy(nodes), elements=torch.from_numpy(perm[m.elements.numpy()]), dirichlet_nodes=bc)


def _line(n_el, seed):
    """A 1-D mesh that is not a chain for the fused path: non-uniform spacing, an interior Dirichlet node, natural right end."""
    rng = np.random.default_rng(seed)
    x = np.concatenate(([0.0], np.cumsum(rng.uniform(0.5, 1.5, n_el))))
    x = -0.3 + 2.0 * x / x[-1]
    el = np.stack((np.arange(n_el), np.arange(1, n_el + 1)), 1)
    return FEMesh(nodes=torch.from_numpy(x[:, None]), elements=torch.from_numpy(el), dirichlet_nodes={0: 0.3, n_el // 3: -0.2})


def _degenerate(nx, ny):
    """rectangle(nx, ny) plus one zero-area triangle on three collinear interior nodes (skipped by the assembly)."""
    m = FEMesh.rectangle(nx, ny, bc_value=-0.1)
    p = 5 * (nx + 1) + 7
    el = np.concatenate((m.elements.numpy(), [[p, p + 1, p + 2]]))
    return FEMesh(nodes=m.nodes, elements=torch.from_numpy(el), dirichlet_nodes=m.dirichlet_nodes)


# name: mesh factory, then what the handle must give: (n_free, n_slices, max SELL slice width)
CASES = {
    "r34x8": (lambda: FEMesh.rectangle(34, 8, bc_value=0.2), (231, 8, 7)),
    "r34x9": (lambda: FEMesh.rectangle(34, 9, x_range=(-1.0, 2.0), bc_value=-0.4), (264, 9, 7)),
    "r34x20": (lambda: FEMesh.rectangle(34, 20, y_range=(0.0, 0.3)), (627, 20, 7)),
    "r40x25": (lambda: FEMesh.rectangle(40, 25, bc_value=1.5), (936, 30, 7)),
    "r40x31": (lambda: FEMesh.rectangle(40, 31, x_range=(0.0, 3.0), y_range=(-1.0, 1.0)), (1170, 37, 7)),
    "r40x37": (lambda: FEMesh.rectangle(40, 37, bc_value=0.05), (1404, 44, 7)),
    "r42x42": (lambda: FEMesh.rectangle(42, 42, bc_value=-0.3), (1681, 53, 7)),
    "r45x44": (lambda: FEMesh.rectangle(45, 44), (1892, 60, 7)),
    "flip38x40": (lambda: _grid(38, 40, "lrbt", 0.0, 0.5, seed=11), (1443, 46, 9)),   # 8-neighbour nodes
    "perm9x8": (lambda: _permuted(9, 8, 0), (56, 2, 7)),
    "lb38x16": (lambda: _grid(38, 16, "lb", 0.0, 0.0), (608, 19, 7)),                  # Dirichlet data on two sides
    "line800": (lambda: _line(800, 3), (799, 25, 3)),
    "degen36x20": (lambda: _degenerate(36, 20), (665, 21, 8)),
}
NAMES = list(CASES)


def _mesh(name):
    return CASES[name][0]()


def _structure(nm):
    """(n_free, n_slices, SELL slice widths, half bandwidth) of K_free from the handle's pattern."""
    rpf, colf = nm.csr(1)
    nf = len(rpf) - 1
    nsl = -(-nf // 32)
    rl = np.diff(rpf)
    widths = [int(rl[32 * s:32 * s + 32].max()) for s in range(nsl)]
    band = int(np.abs(np.repeat(np.arange(nf), rl) - colf).max())
    return nf, nsl, widths, band


def _rpt(nsl):
    """The unroll width `dispatch` (dfe_batch.cu) launches for n_slices slices."""
    return {1: 1, 2: 2, 3: 3, 4: 4, 5: 6, 6: 6, 7: 8, 8: 8}[-(-nsl // BNW)]


def _launched(fn):
    """Run fn() under torch.profiler; returns its result and the names of the project's kernels it launched, template
    arguments included (k_batch<false,2>)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        m = re.search(r"(?:^|::|void)(k_\w+?)(<[^>]*>)?\(", e.name.replace(" ", ""))
        if m:
            names.add(m.group(1) + (m.group(2) or ""))
    return out, names


def _batch_size():
    """More than two samples per resident CTA (at most two CTAs per SM), plus a remainder."""
    return 2 * (2 * torch.cuda.get_device_properties(0).multi_processor_count) + 7


def _rows(B):
    """A row of the first pass over the CTAs, one of a later pass, and the last sample."""
    return [0, B // 2 + 1, B - 1]


def _inputs(m, B, seed):
    rng = np.random.default_rng(seed)
    f = rng.uniform(-0.5, 1.0, (B, m.n_nodes))
    gbar = rng.standard_normal((B, m.n_nodes))
    kap_e = np.exp(rng.uniform(np.log(1e-2), 0.0, m.n_elements))
    return f, gbar, kap_e


def _solver(m, k, force):
    s = DifferentiableFESolver(m, kappa=k)
    if force:
        s._opts["batch_solver"] = "pcg"
    return s


def _run(m, kap, f, gbar, force):
    """u, dL/dkappa, dL/df and the solver for L = sum(gbar * u), optionally with the batched PCG route forced."""
    k = torch.tensor(kap, dtype=torch.float64, device="cuda", requires_grad=True)
    ft = torch.tensor(f, device="cuda", requires_grad=True)
    s = _solver(m, k, force)
    u = s(ft)
    (u * torch.tensor(gbar, device="cuda")).sum().backward()
    return u.detach().cpu().numpy(), k.grad.cpu().numpy(), ft.grad.cpu().numpy(), s


def _reference(m, kap, f, gbar):
    """u, dL/df and per-element dL/dkappa of every row of a batch that shares one matrix, in float64.

    The assembly and the lifting are the oracle's (O.assemble_csr, O.apply_bc).  One sparse LU of K_free solves all rows,
    refined twice with residuals in long double (as O.solve_csr does).  The gradients are the closed forms of
    O.adjoint_and_grads, vectorised over the batch.  The tests check this against O.forward / O.adjoint_and_grads on the
    rows they compare one by one."""
    nodes, el, bc = m.nodes.numpy(), m.elements.numpy(), m.dirichlet_nodes
    n, B = m.n_nodes, f.shape[0]
    rp, col, vals, _ = O.assemble_csr(nodes, el, kap, np.zeros(n))
    free, rpf, colf, vf, lift = O.apply_bc(rp, col, vals, np.zeros(n), bc)
    nf = len(free)
    lu = spla.splu(sp.csc_matrix(sp.csr_matrix((vf, colf, rpf), shape=(nf, nf))))
    vl = vf.astype(np.longdouble)[:, None]

    def solve(R):
        X = lu.solve(R)
        for _ in range(2):   # every row of K_free holds its diagonal entry: no empty segment in reduceat
            AX = np.add.reduceat(vl * X.astype(np.longdouble)[colf], rpf[:-1], axis=0)
            X = (X.astype(np.longdouble) + lu.solve((R.astype(np.longdouble) - AX).astype(np.float64))).astype(np.float64)
        return X

    # the load is F = P f (P symmetric), so dL/df = P lambda
    if m.dim == 1:
        h, _ = O.element_1d(nodes, el, 1.0)
        P = sp.coo_matrix((np.repeat(h / 2.0, 2), (el.ravel(), el.ravel())), shape=(n, n)).tocsr()
    else:
        area, b, c, _, keep = O.element_2d(nodes, el, 1.0)
        ek = el[keep]
        P = sp.coo_matrix((np.repeat(area[keep] / 9.0, 9), (np.repeat(ek, 3, axis=1).ravel(), np.tile(ek, (1, 3)).ravel())),
                          shape=(n, n)).tocsr()
    g = np.zeros(n)
    g[list(bc)] = list(bc.values())
    U = np.tile(g, (B, 1))
    U[:, free] = solve((P @ f.T)[free] + lift[:, None]).T
    Lam = np.zeros((B, n))
    Lam[:, free] = solve(gbar[:, free].T).T
    GF = (P @ Lam.T).T
    if m.dim == 1:
        i, j = el[:, 0], el[:, 1]
        GK = -(Lam[:, j] - Lam[:, i]) * (U[:, j] - U[:, i]) / h
    else:
        bl, bu = np.einsum("ec,bec->be", b, Lam[:, el]), np.einsum("ec,bec->be", b, U[:, el])
        cl, cu = np.einsum("ec,bec->be", c, Lam[:, el]), np.einsum("ec,bec->be", c, U[:, el])
        with np.errstate(divide="ignore", invalid="ignore"):
            GK = np.where(keep, -(bl * bu + cl * cu) / (4.0 * area), 0.0)
    return U, GF, GK


class _Abi:
    """dfe_assemble / dfe_eliminate once, then dfe_batch_fwd / dfe_batch_bwd straight through the C ABI, as
    _batch_forward / _batch_backward call them.  Rows are passed as (data_ptr, stride(0)) of 2-D views."""

    def __init__(self, m, kap):
        self.L = L = _native.lib()
        self.nm = nm = m._native(torch.cuda.current_device())
        I = self.I = nm.info
        self.st = torch.cuda.current_stream().cuda_stream
        kt = torch.as_tensor(np.atleast_1d(np.asarray(kap, dtype=np.float64)), device="cuda")
        self.mode = _native.KAPPA_SCALAR if kt.numel() == 1 else _native.KAPPA_PER_ELEMENT
        self.nk = 1 if self.mode == _native.KAPPA_SCALAR else I.n_elements
        self.vals = torch.empty(max(I.nnz_full, 1), dtype=torch.float64, device="cuda")
        F0 = torch.empty(I.n_nodes, dtype=torch.float64, device="cuda")
        self.sell = torch.empty(max(I.sell_nnz, 1), dtype=torch.float64, device="cuda")
        self.dinv = torch.empty(max(I.n_free, 1), dtype=torch.float64, device="cuda")
        Ff0 = torch.empty(max(I.n_free, 1), dtype=torch.float64, device="cuda")
        f0 = torch.zeros(I.n_nodes, dtype=torch.float64, device="cuda")
        _native.check(L.dfe_assemble(nm.handle, kt.data_ptr(), self.mode, f0.data_ptr(), self.vals.data_ptr(), F0.data_ptr(), self.st))
        _native.check(L.dfe_eliminate(nm.handle, self.vals.data_ptr(), F0.data_ptr(), None, self.sell.data_ptr(), Ff0.data_ptr(),
                                      self.dinv.data_ptr(), self.st))
        self.maxit = max(10 * I.n_free, 1000)

    def _status(self, B):
        return (torch.full((B,), -7, dtype=torch.int32, device="cuda"), torch.full((B,), -1.0, dtype=torch.float64, device="cuda"),
                torch.full((B,), -7, dtype=torch.int32, device="cuda"))

    def fwd(self, f, u, maxit=None):
        """u[b] for the rows of the view f; returns (iters, relres, status)."""
        B = f.shape[0]
        it, rel, stat = self._status(B)
        _native.check(self.L.dfe_batch_fwd(self.nm.handle, B, f.data_ptr(), f.stride(0), self.vals.data_ptr(), self.sell.data_ptr(),
                                           self.dinv.data_ptr(), u.data_ptr(), u.stride(0), TOL, maxit or self.maxit,
                                           it.data_ptr(), rel.data_ptr(), stat.data_ptr(), self.st))
        torch.cuda.synchronize()
        return it, rel, stat

    def bwd(self, gbar, u, gf, gk, maxit=None):
        """dL/df (into gf, or none) and per-sample dL/dkappa (gk: (B, 1) or (B, n_el)); returns (iters, relres, status)."""
        B = gbar.shape[0]
        it, rel, stat = self._status(B)
        _native.check(self.L.dfe_batch_bwd(self.nm.handle, B, gbar.data_ptr(), gbar.stride(0), u.data_ptr(), u.stride(0),
                                           self.sell.data_ptr(), self.dinv.data_ptr(), self.mode,
                                           None if gf is None else gf.data_ptr(), self.I.n_nodes if gf is None else gf.stride(0),
                                           gk.data_ptr(), TOL, maxit or self.maxit, it.data_ptr(), rel.data_ptr(), stat.data_ptr(),
                                           self.st))
        torch.cuda.synchronize()
        return it, rel, stat

    def solve(self, f, gbar, with_gf=True):
        """Forward and adjoint of the whole batch on fresh buffers: (u, dL/df or None, dL/dkappa per sample)."""
        B, n = f.shape
        u = torch.empty((B, n), dtype=torch.float64, device="cuda")
        assert int(self.fwd(f, u)[2].abs().max()) == 0
        gf = torch.empty((B, n), dtype=torch.float64, device="cuda") if with_gf else None
        gk = torch.empty((B, self.nk), dtype=torch.float64, device="cuda")
        assert int(self.bwd(gbar, u, gf, gk)[2].abs().max()) == 0
        return u, gf, gk


# ==================================================================================================== the case table
def test_case_table_structure():
    L = _native.lib()
    buckets = set()
    for name in NAMES:
        m = _mesh(name)
        nm = m._native(torch.cuda.current_device())
        nf, nsl, widths, band = _structure(nm)
        assert (nf, nsl, max(widths)) == CASES[name][1], name
        assert nm.info.n_free == nf and nm.info.sell_nnz == 32 * sum(widths), name
        assert L.dfe_batch_supported(nm.handle) == 1, name
        assert band > 32 if m.dim == 2 else band == 1, name
        assert L.dfe_band_supported(nm.handle) == (0 if m.dim == 2 else 1), name   # the 1-D line is forced onto the route
        buckets.add(-(-nsl // BNW))
    assert buckets == set(range(1, 9))
    m = _mesh("flip38x40")
    assert sum(w > WMAX for w in _structure(m._native(torch.cuda.current_device()))[2]) >= 5
    m = _mesh("perm9x8")
    d = list(m.dirichlet_nodes)
    assert d != sorted(d)
    m = _mesh("lb38x16")
    assert len(set(m.dirichlet_nodes.values())) > 30
    m = _mesh("line800")
    assert m._native(torch.cuda.current_device()).info.chain1d == 0 and m.dirichlet_nodes.get(800) is None
    m = _mesh("degen36x20")
    area = O.element_2d(m.nodes.numpy(), m.elements.numpy(), 1.0)[0]
    assert area[-1] == 0.0 and (area[:-1] > 1e-4).all()


# ============================================================= route, instantiation and the float64 oracle, end to end
@pytest.mark.parametrize("name", NAMES)
def test_vs_oracle(name):
    """Scalar and shared per-element kappa through DifferentiableFESolver at B = 4 #SMs + 7: the kernels that ran, u and
    dL/df of rows from different passes against the oracle, and the batch-summed dL/dkappa against the sum of the
    float64 gradients of every row."""
    m = _mesh(name)
    nm = m._native(torch.cuda.current_device())
    force = m.dim == 1
    B = _batch_size()
    f, gbar, kap_e = _inputs(m, B, 100 + NAMES.index(name))
    kap_s = 0.8
    (scalar, elem), names = _launched(lambda: (_run(m, kap_s, f, gbar, force), _run(m, kap_e, f, gbar, force)))
    R = _rpt(_structure(nm)[1])
    assert {k for k in names if k.startswith("k_batch")} == {f"k_batch<false,{R}>", f"k_batch<true,{R}>"}, names
    assert not any(k.startswith(("k_band", "k_pcg")) for k in names), names

    worst = {}
    for kap, (u, gk, gf, s) in ((kap_s, scalar), (kap_e, elem)):
        assert s.last_pcg[0][0] > 0 and s._opts["last_pcg_adjoint"][0][0] > 0
        U, GF, GK = _reference(m, kap, f, gbar)
        for b in _rows(B):
            uo, gko, gfo = oracle_run(m, kap, f[b], gbar[b])
            # the batched reference is the oracle's arithmetic
            assert relerr(U[b], uo) <= 1e-12 and relerr(GF[b], gfo) <= 1e-12
            assert np.abs(GK[b] - gko).max() <= 1e-12 * np.abs(gko).sum()
            eu, ef = relerr(u[b], uo), relerr(gf[b], gfo)
            assert eu <= TOL2D and ef <= TOL2D, (b, eu, ef)
            worst["u"], worst["gf"] = max(worst.get("u", 0), eu), max(worst.get("gf", 0), ef)
        if np.ndim(kap) == 0:
            eg = abs(float(gk) - GK.sum()) / np.abs(GK).sum()
        else:
            mag = np.abs(GK).sum(0)
            err = np.abs(gk - GK.sum(0))
            assert np.all(err <= TOL2D * mag)
            eg = float((err / np.where(mag > 0, mag, 1.0)).max())
        assert eg <= TOL2D
        worst["gk_scalar" if np.ndim(kap) == 0 else "gk_elem"] = eg
    print(f"\n[{name}] k_batch<*,{R}> worst relative errors: " + ", ".join(f"{k} {v:.2e}" for k, v in worst.items()))


# =============================================================================== bits do not depend on the position
@pytest.mark.parametrize("name", NAMES)
def test_bits_independent_of_position(name):
    """Rows from the first pass, a later pass and the last sample, re-solved alone (B = 1), give the same bits for u,
    dL/df and the per-sample dL/dkappa (scalar and per element); the adjoint without dL/df gives the same dL/dkappa."""
    m = _mesh(name)
    B = _batch_size()
    f, gbar, kap_e = _inputs(m, B, 200 + NAMES.index(name))
    ft, gt = torch.tensor(f, device="cuda"), torch.tensor(gbar, device="cuda")
    for kap in (1.3, kap_e):
        abi = _Abi(m, kap)
        u, gf, gk = abi.solve(ft, gt)
        _, no_gf, gk2 = abi.solve(ft, gt, with_gf=False)
        assert no_gf is None and torch.equal(gk2, gk)
        for b in _rows(B):
            u1, gf1, gk1 = abi.solve(ft[b:b + 1], gt[b:b + 1])
            assert torch.equal(u1[0], u[b]) and torch.equal(gf1[0], gf[b]) and torch.equal(gk1[0], gk[b]), b
        # the per-sample gradient itself, against the oracle (the module only returns the batch sum)
        b = B - 1
        uo, gko, _ = oracle_run(m, kap, f[b], gbar[b])
        ref = gko.sum() if np.ndim(kap) == 0 else gko
        assert np.abs(gk[b].cpu().numpy() - ref).max() <= TOL2D * np.abs(gko).sum()


# ============================================================================= power-of-two scaling of the input data
def _scaled_run(m, f, gbar):
    u, gk, gf, s = run(m, 1.3, f, gbar)
    assert s.last_pcg[0][0] > 0                                 # the batched PCG route (the default for this mesh)
    return u, gk, gf


def test_power_of_two_scale_invariance():
    """f and gbar times 2^k: u and dL/df are 2^k, dL/dkappa 2^2k times the unscaled result, bit for bit, as long as
    every intermediate stays normal (|k| <= 400 here)."""
    rng = np.random.default_rng(31)
    m = FEMesh.rectangle(40, 35)
    L = _native.lib()
    assert L.dfe_band_supported(m._native(torch.cuda.current_device()).handle) == 0
    f, gbar = rng.uniform(0.5, 1.0, (3, m.n_nodes)), rng.uniform(0.5, 1.0, (3, m.n_nodes))
    u0, gk0, gf0 = _scaled_run(m, f, gbar)
    for k in (-400, -64, 1, 64, 400):
        s = 2.0 ** k
        u, gk, gf = _scaled_run(m, f * s, gbar * s)
        assert np.array_equal(u, u0 * s) and np.array_equal(gf, gf0 * s), k
        assert np.array_equal(gk, gk0 * s * s), k


@pytest.mark.parametrize("side", ["f", "gbar"])
@pytest.mark.parametrize("scale", [2.0 ** -1000, 1e-160, 2.0 ** 1000], ids=["2^-1000", "1e-160", "2^1000"])
def test_extreme_magnitudes(scale, side):
    """Right-hand sides whose squares underflow (|F| < ~1e-162: ||F||^2 == 0) or overflow, in the forward (f scaled) or
    in the adjoint (gbar scaled).  Products such as area / 9 * lambda may become subnormal, so these are checked at TOL2D
    against the unscaled result times the scale and against the oracle, not bit for bit."""
    rng = np.random.default_rng(32)
    m = FEMesh.rectangle(40, 35)
    nodes, el, bc = m.nodes.numpy(), m.elements.numpy(), m.dirichlet_nodes
    f, gbar = rng.uniform(0.5, 1.0, (3, m.n_nodes)), rng.uniform(0.5, 1.0, (3, m.n_nodes))
    u0, gk0, gf0 = _scaled_run(m, f, gbar)

    def check(u, gk, gf, fs, gs, su, sg):
        assert relerr(u, u0 * su) <= TOL2D and relerr(gf, gf0 * sg) <= TOL2D
        assert abs(float(gk) - float(gk0) * su * sg) <= TOL2D * abs(float(gk0) * su * sg)
        assert np.abs(u[:, m.free_nodes()]).min() > 0.0 and np.abs(gf[:, m.free_nodes()]).min() > 0.0
        tot, mag = 0.0, 0.0
        for b in range(3):
            uo = O.forward(nodes, el, bc, 1.3, fs[b])
            gko, gfo, _ = O.adjoint_and_grads(nodes, el, bc, 1.3, uo, gs[b])
            assert relerr(u[b], uo) <= TOL2D and relerr(gf[b], gfo) <= TOL2D, b
            tot, mag = tot + gko.sum(), mag + np.abs(gko).sum()
        assert mag > 0.0 and abs(float(gk) - tot) <= TOL2D * mag

    if side == "f":
        u, gk, gf = _scaled_run(m, f * scale, gbar)
        assert np.array_equal(gf, gf0)                           # lambda depends on gbar alone
        check(u, gk, gf, f * scale, gbar, scale, 1.0)
    else:
        u, gk, gf = _scaled_run(m, f, gbar * scale)
        assert np.array_equal(u, u0)
        check(u, gk, gf, f, gbar * scale, 1.0, scale)


# ========================================================================================= status arrays through the ABI
def test_status_arrays():
    """Per-sample status / iters / relres of dfe_batch_fwd / dfe_batch_bwd when some samples fail, and the exceptions the
    module raises from them."""
    m = FEMesh.rectangle(40, 25)                                 # zero Dirichlet data
    rng = np.random.default_rng(41)
    B, n = 9, m.n_nodes
    kap = 0.7
    abi = _Abi(m, kap)
    f = torch.tensor(rng.uniform(-0.5, 1.0, (B, n)), device="cuda")
    gbar = torch.tensor(rng.standard_normal((B, n)), device="cuda")
    u = torch.empty_like(f)
    it, rel, stat = abi.fwd(f, u)
    assert bool((stat == 0).all()) and bool((it > 0).all()) and bool((rel <= TOL).all()) and bool((rel >= 0).all())
    gf, gk = torch.empty_like(f), torch.empty((B, 1), dtype=torch.float64, device="cuda")
    it_a, rel_a, stat_a = abi.bwd(gbar, u, gf, gk)
    assert bool((stat_a == 0).all()) and bool((it_a > 0).all()) and bool((rel_a <= TOL).all())
    # true residual of the converged solutions, in float64 from the K_free and F_free that dfe_eliminate assembles
    free = abi.nm.free_nodes()
    rpf, colf = abi.nm.csr(1)
    for b in (0, 5, B - 1):
        _, _, _, vf, Ff, _ = abi_assemble(m, kap, f[b].cpu().numpy())
        A = sp.csr_matrix((vf, colf, rpf), shape=(len(free),) * 2)
        assert np.linalg.norm(A @ u[b].cpu().numpy()[free] - Ff) <= 1e-11 * np.linalg.norm(Ff), b
        uo, _, gfo = oracle_run(m, kap, f[b].cpu().numpy(), gbar[b].cpu().numpy())
        assert relerr(u[b].cpu().numpy(), uo) <= TOL2D and relerr(gf[b].cpu().numpy(), gfo) <= TOL2D, b
    # one NaN sample: status 5 for it alone, every other row the bits of the clean run
    fn = f.clone()
    fn[4, free[100]] = float("nan")
    un = torch.empty_like(f)
    _, _, st = abi.fwd(fn, un)
    assert st.tolist() == [5 if b == 4 else 0 for b in range(B)]
    keep = [b for b in range(B) if b != 4]
    assert torch.equal(un[keep], u[keep])
    gn = gbar.clone()
    gn[6, free[7]] = float("nan")
    gfn, gkn = torch.empty_like(f), torch.empty_like(gk)
    _, _, st = abi.bwd(gn, u, gfn, gkn)
    assert st.tolist() == [5 if b == 6 else 0 for b in range(B)]
    keep = [b for b in range(B) if b != 6]
    assert torch.equal(gfn[keep], gf[keep]) and torch.equal(gkn[keep], gk[keep])
    # a zero right-hand side: converged after 0 iterations, u == 0, and zero gradients for gbar == 0
    fz = f.clone()
    fz[2] = 0.0
    uz = torch.empty_like(f)
    it, rel, st = abi.fwd(fz, uz)
    assert int(st[2]) == 0 and int(it[2]) == 0 and float(rel[2]) == 0.0 and bool((uz[2] == 0).all())
    assert torch.equal(uz[3:], u[3:])
    gz = gbar.clone()
    gz[2] = 0.0
    gfz, gkz = torch.empty_like(f), torch.empty_like(gk)
    it, rel, st = abi.bwd(gz, uz, gfz, gkz)
    assert int(st[2]) == 0 and int(it[2]) == 0 and bool((gfz[2] == 0).all()) and float(gkz[2, 0]) == 0.0
    # too few iterations: status 4 and iters == maxit for every sample
    it, _, st = abi.fwd(f, torch.empty_like(f), maxit=5)
    assert bool((st == 4).all()) and bool((it == 5).all())
    it, _, st = abi.bwd(gbar, u, None, torch.empty_like(gk), maxit=5)
    assert bool((st == 4).all()) and bool((it == 5).all())

    # the module turns them into the per-sample path's exceptions, naming the failing sample
    def module(fv, gv, maxit=None):
        k = torch.tensor(kap, dtype=torch.float64, device="cuda", requires_grad=True)
        s = DifferentiableFESolver(m, kappa=k, pcg_maxit=maxit)
        (s(fv) * gv).sum().backward()

    with pytest.raises(_native.BreakdownError, match=r"dfe_batch_fwd: breakdown in sample 4 "):
        module(fn, gbar)
    with pytest.raises(_native.BreakdownError, match=r"dfe_batch_bwd: breakdown in sample 6 "):
        module(f, gn)
    one = torch.zeros_like(f)
    one[7] = f[7]
    with pytest.raises(_native.NotConvergedError, match=r"dfe_batch_fwd: sample 7 not converged after 5 iterations"):
        module(one, gbar, maxit=5)
    one = torch.zeros_like(gbar)
    one[3] = gbar[3]
    with pytest.raises(_native.NotConvergedError, match=r"dfe_batch_bwd: sample 3 not converged after 5 iterations"):
        module(torch.zeros_like(f), one, maxit=5)


# ========================================================================================= strided rows through the ABI
@pytest.mark.parametrize("name", ["r34x9", "line800", "flip38x40"])
def test_abi_strided_rows(name):
    """dfe_batch_fwd / dfe_batch_bwd on column slices of NaN-padded (B, ld) buffers with odd ld (rows alternate between the
    two 16-byte phases; offset 1 puts row 0 at 8 mod 16), against the contiguous call, bit for bit; the padding of u and
    dL/df stays untouched."""
    m = _mesh(name)
    n, B = m.n_nodes, 11
    ld = n + 1 if n % 2 == 0 else n + 2
    f, gbar, kap_e = _inputs(m, B, 300 + NAMES.index(name))
    ft, gt = torch.tensor(f, device="cuda"), torch.tensor(gbar, device="cuda")
    nan_bits = torch.tensor(float("nan"), dtype=torch.float64).view(torch.int64).item()

    def padded(off, data=None):
        buf = torch.full((B, ld), float("nan"), dtype=torch.float64, device="cuda")
        if data is not None:
            buf[:, off:off + n] = data
        return buf, buf[:, off:off + n]

    def untouched(buf, off):
        keep = torch.ones(ld, dtype=torch.bool)
        keep[off:off + n] = False
        return bool((buf[:, keep.cuda()].view(torch.int64) == nan_bits).all())

    for kap in (0.9, kap_e):
        abi = _Abi(m, kap)
        u_ref, gf_ref, gk_ref = abi.solve(ft, gt)
        for a, b in ((0, 1), (1, 0)):                           # offsets of the inputs / outputs inside their buffers
            fb, fv = padded(a, ft)
            ub, uv = padded(b)
            assert uv.data_ptr() % 16 == 8 * b
            _, _, st = abi.fwd(fv, uv)
            assert int(st.abs().max()) == 0
            assert torch.equal(uv, u_ref) and untouched(ub, b)
            gb, gv = padded(b, gt)
            ub2, uv2 = padded(a, u_ref)
            gfb, gfv = padded(a)
            gk = torch.empty_like(gk_ref)
            _, _, st = abi.bwd(gv, uv2, gfv, gk)
            assert int(st.abs().max()) == 0
            assert torch.equal(gfv, gf_ref) and torch.equal(gk, gk_ref) and untouched(gfb, a)
            gk2 = torch.empty_like(gk_ref)
            abi.bwd(gv, uv2, None, gk2)                          # without dL/df
            assert torch.equal(gk2, gk_ref)


# ===================================================================================================== support predicate
LIMIT = 200 * 1024


def _smem(nm):
    """batch_smem(m, true) (dfe_batch.cu): SELL values and columns, the search direction, the reduction slots and lambda on
    every node, in bytes."""
    I = nm.info
    nsl = -(-I.n_free // 32)
    return (I.sell_nnz + 32 * nsl + 6 * BNW + I.n_nodes) * 8 + I.sell_nnz * 4 + 16


def _fits(m, nm):
    """batch_fits (dfe_batch.cu) restated: a device handle of a P1 mesh with a free node, at most 8 warps x 8 slices, and
    the adjoint's shared memory within 200 KB."""
    I = nm.info
    if I.device < 0 or I.n_free < 1 or m.elements.shape[1] != m.dim + 1:
        return False
    return -(-I.n_free // 32) <= BNW * 8 and _smem(nm) <= LIMIT


def test_support_predicate():
    """dfe_batch_supported against the restated predicate on both sides of each of its limits."""
    L = _native.lib()
    dev = torch.cuda.current_device()
    # name: mesh, n_slices, supported
    meshes = {
        "line2049": (FEMesh.line(2049), 64, True),              # 2048 free nodes: 64 slices
        "line2050": (FEMesh.line(2050), 65, False),             # 2049 free nodes: 65 slices
        "r65x33": (FEMesh.rectangle(65, 33), 64, True),
        "r66x33": (FEMesh.rectangle(66, 33), 65, False),
        "r47x45": (FEMesh.rectangle(47, 45), 64, True),         # 624 bytes below the shared-memory limit
        "flip40x44": (_grid(40, 44, "lrbt", 0.0, 0.5, seed=1), 53, False),   # 9-wide slices: over it with 53 slices
        "r45x44": (FEMesh.rectangle(45, 44), 60, True),
        "r60x60": (FEMesh.rectangle(60, 60), 109, False),
        "r1x1": (FEMesh.rectangle(1, 1), 0, False),             # no free node
        "r4x4_p2": (FEMesh.rectangle(4, 4).to_p2(), 2, False),  # P2 elements
    }
    for name, (m, nsl, want) in meshes.items():
        nm = m._native(dev)
        assert -(-nm.info.n_free // 32) == nsl, name
        assert _fits(m, nm) == want, name
        assert L.dfe_batch_supported(nm.handle) == int(want), name
        assert L.dfe_batch_supported(m._native(-1).handle) == 0, name   # a host-only handle
    # the slice limit alone separates line2049 from line2050 (both far below the shared-memory limit) ...
    assert all(_smem(meshes[k][0]._native(dev)) <= LIMIT - 64 * 1024 for k in ("line2049", "line2050"))
    # ... and the shared-memory limit alone r47x45 from flip40x44 (both within the slice limit)
    assert LIMIT - 1024 < _smem(meshes["r47x45"][0]._native(dev)) <= LIMIT
    assert LIMIT < _smem(meshes["flip40x44"][0]._native(dev)) <= LIMIT + 2 * 1024
