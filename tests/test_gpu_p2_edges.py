"""The quadratic-element (P2) route at every mesh shape, kappa layout and solver partition it accepts, against the
quadrature oracle (oracle/oracle_p2.py) and against exact quadratic solutions.

A P2 mesh (``FEMesh.to_p2()``) takes the general route: `k_assemble` (the P2 branch of `assemble_row`, closed-form element
matrices of dfe_p2.cuh), `k_eliminate`, `k_fill_sell`, the cooperative Jacobi-PCG `k_pcg`, `k_scatter`, `k_gather`,
`k_grad_elem` and `k_grad_f`.  Its rows are wider and more varied than P1 rows: a vertex of valence v has 1 + 3v entries
(19 on a rectangle, 16 or 22 next to it on an unstructured mesh), an edge midpoint 9, the centre of a 45-spoke wheel 136.
Rows of more than ROWMAX = 16 entries are assembled by read-modify-write in global memory.  The case table reaches one
`k_pcg` CTA with a partial last slice, a full grid with CTAs left without a slice, warps that make two trips with an odd
last pair, a slice far wider than the others, clockwise triangles, element areas over nine decades, a zero-area triangle,
and 1-D lines of 1, 2 and 700 elements.

The oracle integrates the element matrices by quadrature; they are computed once per mesh and assembled here per kappa,
so the solve and the adjoint share one factorisation.
"""
import functools
import warnings

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as spla
import torch
from scipy.spatial import Delaunay

from difffe_physics_lab_b200 import _native, assemble_sparse
from diffhe.mesh import FEMesh
from oracle import oracle_p2 as P
from tests.test_gpu_batch_pcg import _launched
from tests.test_gpu_coop_pcg import PW, _plan, _slices, _wheel
from tests.test_gpu_parity import TOL2D, abi_assemble, relerr, run

pytestmark = pytest.mark.gpu

AREA_EPS = 1e-15   # dfe_assemble_row.cuh: triangles below this area contribute nothing
ROWMAX = 16        # dfe_assemble_row.cuh: longer rows of K are accumulated in global memory


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    _native.build()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _dev():
    return torch.cuda.current_device()


# ================================================================================================= the case table
def _p2_square(pred, start):
    """The smallest even n >= start whose rectangle(n, n).to_p2() ((2n - 1)^2 free nodes, the count of a P1
    rectangle(2n)) gives a k_pcg split with pred(grid, per_cta, CTAs without a slice)."""
    sms = _sms()
    for n in range(start + start % 2, 4 * start, 2):
        if pred(*_plan(-(-(2 * n - 1) ** 2 // 32), sms)):
            return n
    raise AssertionError("no rectangle size fits")


def _n_empty():
    """A full grid in which some CTAs get no slice: rectangle(170, 170) on 148 SMs."""
    return _p2_square(lambda g, per, empty: g == _sms() and empty >= 1, 170)


def _n_two_trips():
    """A full grid whose warps make two trips, the second with an odd last pair: rectangle(250, 250) on 148 SMs."""
    return _p2_square(lambda g, per, empty: g == _sms() and 2 * PW < per < 3 * PW, 250)


def _delaunay():
    """Delaunay triangulation of a jittered 45 x 45 lattice in the unit square plus 4 x 24 points on its boundary (the
    Dirichlet nodes).  Each triangle's vertex order is rotated or reflected at random before to_p2(), so about half the
    triangles are clockwise; interior vertices have 4 to 8 neighbours."""
    rng = np.random.default_rng(11)
    k = 24
    t = np.arange(k) / k
    z, o = np.zeros(k), np.ones(k)
    edge = np.concatenate((np.stack((t, z), 1), np.stack((o, t), 1), np.stack((1 - t, o), 1), np.stack((z, 1 - t), 1)))
    g = (np.arange(45) + 0.5) / 45
    lat = np.stack(np.meshgrid(g, g), -1).reshape(-1, 2) + rng.uniform(-0.3 / 45, 0.3 / 45, (45 * 45, 2))
    xy = np.concatenate((edge, lat))
    el = Delaunay(xy).simplices.astype(np.int64)
    perms = np.array([[0, 1, 2], [1, 2, 0], [2, 0, 1], [0, 2, 1], [2, 1, 0], [1, 0, 2]])
    el = np.take_along_axis(el, perms[rng.integers(0, 6, len(el))], axis=1)
    bc = {i: 0.1 + 0.2 * xy[i, 0] - 0.1 * xy[i, 1] for i in range(4 * k)}
    return FEMesh(nodes=torch.from_numpy(xy), elements=torch.from_numpy(el), dirichlet_nodes=bc).to_p2()


def _graded():
    """rectangle(24, 24) on the unit square with its vertices moved by p -> p |p|^3: elements shrink towards the origin
    (nearly isotropically: the map stretches radial lengths 4 times more than angular ones), areas from 4.5e-12 to 2.5e-2."""
    m = FEMesh.rectangle(24, 24, bc_value=0.3)
    x = m.nodes.numpy()
    xg = x * np.linalg.norm(x, axis=1, keepdims=True) ** 3
    return FEMesh(nodes=torch.from_numpy(xg), elements=m.elements, dirichlet_nodes=m.dirichlet_nodes).to_p2()


DEG_NX, DEG_NY, DEG_A = 9, 7, 3 * 10 + 3   # the zero-area triangle [a, a + 1, a + 2]: three interior vertices of row 3


def _degenerate_p1():
    return FEMesh.rectangle(DEG_NX, DEG_NY, x_range=(0.0, 1.2), bc_value=0.15)


def _degenerate(free_mid=False):
    """rectangle(9, 7) plus a last triangle on three collinear interior vertices a, b, c.  Its edges (a, b) and (b, c)
    are mesh edges; its third edge (c, a) is new, and that edge's midpoint (local node 5) belongs to no other triangle.
    That midpoint is made Dirichlet, unless free_mid: then K_free has a zero row there."""
    base = _degenerate_p1()
    tri = torch.tensor([[DEG_A, DEG_A + 1, DEG_A + 2]], dtype=base.elements.dtype)
    m = FEMesh(nodes=base.nodes, elements=torch.cat((base.elements, tri)), dirichlet_nodes=base.dirichlet_nodes).to_p2()
    if free_mid:
        return m
    bc = dict(m.dirichlet_nodes)
    bc[int(m.elements[-1, 5])] = 0.37
    return FEMesh(nodes=m.nodes, elements=m.elements, dirichlet_nodes=bc)


def _line_p2(n):
    """A 1-D P2 line of n elements with random spacing on [0.3, 2.1], a natural right end, and Dirichlet data at the
    left end (n = 1), at the middle vertex only (n = 2: both ends natural) or at the left end and vertex n // 3."""
    rng = np.random.default_rng(n)
    x = np.concatenate(([0.0], np.cumsum(rng.uniform(0.2, 1.8, n))))
    x = 0.3 + 1.8 * x / x[-1]
    bc = {0: 0.4} if n == 1 else ({1: -0.2} if n == 2 else {0: 0.4, n // 3: -0.2})
    el = np.stack((np.arange(n), np.arange(n) + 1), 1)
    return FEMesh(nodes=torch.from_numpy(x[:, None]), elements=torch.from_numpy(el), dirichlet_nodes=bc).to_p2()


CASES = {
    "rect_one_cta": lambda: FEMesh.rectangle(10, 8, x_range=(-0.5, 1.0), y_range=(0.0, 0.8), bc_value=0.2).to_p2(),
    "rect_empty_cta": lambda: FEMesh.rectangle(_n_empty(), _n_empty(), bc_value=0.1).to_p2(),
    "rect_two_trips": lambda: FEMesh.rectangle(_n_two_trips(), _n_two_trips()).to_p2(),
    "wheel": lambda: _wheel(12).to_p2(),
    "delaunay": _delaunay,
    "graded": _graded,
    "degenerate": _degenerate,
    "line_p2_1": lambda: _line_p2(1),
    "line_p2_2": lambda: _line_p2(2),
    "line_p2_700": lambda: _line_p2(700),
}
CASES_2D = ["rect_one_cta", "rect_empty_cta", "rect_two_trips", "wheel", "delaunay", "graded", "degenerate"]
ORACLE_CASES = [c for c in CASES if c != "rect_two_trips"]
LAYOUTS = ("scalar", "elem", "sample", "sample_elem")


@functools.lru_cache(maxsize=None)
def _mesh(name):
    return CASES[name]()


def _areas(m):
    x = m.nodes.numpy()
    p = x[m.elements.numpy()[:, :3]]
    return 0.5 * np.abs((p[:, 1, 0] - p[:, 0, 0]) * (p[:, 2, 1] - p[:, 0, 1]) - (p[:, 2, 0] - p[:, 0, 0]) * (p[:, 1, 1] - p[:, 0, 1]))


def test_case_table_structure():
    """What each mesh gives the kernels, from the handle's pattern of K_free: the k_pcg block split (its values on 148
    SMs), the widths of vertex and midpoint rows, orientations, areas and the Dirichlet set."""
    sms = _sms()
    want148 = {"rect_one_cta": (285, 9, 1, 9, 0), "rect_empty_cta": (339 ** 2, 3592, 148, 25, 4),
               "rect_two_trips": (499 ** 2, 7782, 148, 53, 1)}
    for name in CASES:
        m = _mesh(name)
        nm = m._native(_dev())
        nf, widths = _slices(m)
        nsl = len(widths)
        grid, per, empty = _plan(nsl, sms)
        rpf, _ = nm.csr(1)
        free = nm.free_nodes()
        el = m.elements.numpy()
        nv = int(el[:, :m.dim + 1].max()) + 1                  # to_p2() keeps the vertices first
        rl = np.diff(rpf)
        vrows, mrows = rl[free < nv], rl[free >= nv]
        assert nm.info.n_free == nf == len(free) and nm.info.sell_nnz == 32 * sum(widths), name
        assert nm.info.chain1d == 0 and el.shape[1] == (3 if m.dim == 1 else 6), name
        if sms == 148 and name in want148:
            assert (nf, nsl, grid, per, empty) == want148[name], (name, nf, nsl, grid, per, empty)
        if name == "rect_one_cta":
            assert grid == 1 and nf % 32 != 0                             # one CTA, partial last slice
            assert vrows.max() == 19 and 9 in set(mrows.tolist()) and mrows.max() == 9
        if name == "rect_empty_cta":
            assert grid == sms and empty >= 1 and _n_empty() % 2 == 0
        if name == "rect_two_trips":
            assert grid == sms and 2 * PW < per < 3 * PW and _n_two_trips() % 2 == 0
        if name == "wheel":
            assert free[0] == 0 and rl[0] == 1 + 3 * 45 == 136 > ROWMAX    # the centre: global read-modify-write
            assert widths[0] == 136 and sorted(widths)[-2] <= 24           # one slice far wider than the rest
        if name == "delaunay":
            assert {16, 19} <= set(vrows.tolist()) and vrows.min() < ROWMAX < vrows.max() and mrows.max() == 9
            x = m.nodes.numpy()[el[:, :3]]
            det = (x[:, 1, 0] - x[:, 0, 0]) * (x[:, 2, 1] - x[:, 0, 1]) - (x[:, 2, 0] - x[:, 0, 0]) * (x[:, 1, 1] - x[:, 0, 1])
            assert (det > 0).sum() > len(el) // 3 and (det < 0).sum() > len(el) // 3
            assert len(np.unique(el[:, :3])) == nv                        # qhull kept every point
        if name == "graded":
            a = _areas(m)
            assert a.min() > 1000 * AREA_EPS and a.max() / a.min() > 1e6 and (a < 1e-6).sum() > 10
        if name == "degenerate":
            a = _areas(m)
            assert a[-1] == 0.0 and a[:-1].min() > 1e-3
            mid = int(el[-1, 5])
            assert (el == mid).sum() == 1 and mid in m.dirichlet_nodes
        if name.startswith("line_p2"):
            n_el = int(name.rsplit("_", 1)[1])
            assert m.n_elements == n_el and n_el not in m.dirichlet_nodes  # a natural right end
            if n_el > 1:
                assert any(0 < v < n_el for v in m.dirichlet_nodes)        # an interior Dirichlet vertex


# ================================================================================================ inputs and oracle
def _kappa_field(name, rng, B):
    """B per-element kappa fields.  2-D: independent values over two decades.  Lines: four decades, varying smoothly
    along the line (up or down) with a +-0.1 decade jitter; independent values over four decades would make Jacobi-PCG
    need 10-15 times n_free iterations on line_p2_700 and leave errors of ~1e-9 (measured with the same algorithm in
    float64 on the CPU), so the comparison would test the conditioning, not the kernels."""
    m = _mesh(name)
    if m.dim == 2:
        return 10.0 ** rng.uniform(-2.0, 0.0, (B, m.n_elements))
    x = m.nodes.numpy()[:, 0]
    t = (x[m.elements.numpy()[:, 2]] - x.min()) / (x.max() - x.min())
    return np.stack([10.0 ** (-2.0 + 4.0 * (t if b % 2 == 0 else 1 - t) + rng.uniform(-0.1, 0.1, m.n_elements))
                     for b in range(B)])


def _inputs(name, layout, seed=0):
    """(f, gbar, kappa) of a layout: scalar and (n_el,) kappa with one sample, (B, 1) and (B, n_el) with B samples."""
    m = _mesh(name)
    rng = np.random.default_rng(1000 * seed + 10 * sorted(CASES).index(name) + LAYOUTS.index(layout))
    B = 2 if name == "rect_empty_cta" else 3
    shape = (B, m.n_nodes) if layout.startswith("sample") else (m.n_nodes,)
    f, gbar = rng.uniform(-0.5, 1.0, shape), rng.standard_normal(shape)
    kap = {"scalar": lambda: np.asarray(1.3),
           "elem": lambda: _kappa_field(name, rng, 1)[0],
           "sample": lambda: np.exp(rng.uniform(-1.0, 1.0, (B, 1))),
           "sample_elem": lambda: _kappa_field(name, rng, B)}[layout]()
    return f, gbar, kap


@functools.lru_cache(maxsize=None)
def _elem_mats(name):
    """(K0, M) of every element by quadrature, and the COO indices that assemble them."""
    m = _mesh(name)
    el = m.elements.numpy()
    K0, M = P.element_matrices(m.nodes.numpy(), el)
    npe = el.shape[1]
    return K0, M, np.repeat(el, npe, axis=1).ravel(), np.tile(el, (1, npe)).ravel()


def _oracle_mats(name, kap_e):
    """K (kappa_e per element) and the mass matrix, both over all nodes."""
    m = _mesh(name)
    K0, M, rows, cols = _elem_mats(name)
    n = m.n_nodes
    K = sp.csr_matrix(((kap_e[:, None, None] * K0).ravel(), (rows, cols)), shape=(n, n))
    return K, sp.csr_matrix((M.ravel(), (rows, cols)), shape=(n, n))


def _oracle(name, kap_e, f, gbar):
    """u, dL/dkappa_e, dL/df for L = gbar . u, and the scale max_e |lam_e|^T |K0_e| |u_e| of dL/dkappa_e; the solve and
    the adjoint share one sparse LU with two steps of iterative refinement, as in oracle_p2.forward."""
    m = _mesh(name)
    el = m.elements.numpy()
    K0 = _elem_mats(name)[0]
    K, Mg = _oracle_mats(name, kap_e)
    n = m.n_nodes
    d = np.fromiter(m.dirichlet_nodes.keys(), dtype=np.int64, count=len(m.dirichlet_nodes))
    g = np.fromiter(m.dirichlet_nodes.values(), dtype=np.float64, count=len(m.dirichlet_nodes))
    free = np.setdiff1d(np.arange(n), d)
    Kff = K[free][:, free].tocsc()
    lu = spla.splu(Kff)

    def solve(rhs):
        x = lu.solve(rhs)
        for _ in range(2):
            x = x + lu.solve(rhs - Kff @ x)
        return x

    u = np.zeros(n)
    u[d] = g
    u[free] = solve((Mg @ f)[free] - K[free][:, d] @ g)
    lam = np.zeros(n)
    lam[free] = solve(np.asarray(gbar)[free])
    ue, le = u[el], lam[el]
    gk = -np.einsum("ei,eij,ej->e", le, K0, ue)
    scale = float(np.einsum("ei,eij,ej->e", np.abs(le), np.abs(K0), np.abs(ue)).max())
    return u, gk, Mg @ lam, scale


def _kap_rows(kap, B, n_el):
    """kappa_e of every sample, (B, n_el), for any of the four layouts."""
    k = np.asarray(kap, dtype=np.float64)
    return np.broadcast_to(k.reshape(B if k.ndim == 2 else 1, -1), (B, n_el))


# ========================================================================================================= assembly
@pytest.mark.parametrize("kind", ["scalar", "elem"])
@pytest.mark.parametrize("name", list(CASES))
def test_assembly_vs_quadrature(name, kind):
    """K and F = M f through the C ABI and through assemble_sparse (the same bits), against the oracle's quadrature:
    K entrywise within 1e-13 of the largest |K| of its row, F within 1e-13 of (|M| |f|) of its row, so that the rows of
    elements ten decades smaller than the largest are held to the same relative accuracy."""
    m = _mesh(name)
    f, _, kap = _inputs(name, kind)
    nm, vals, F, *_ = abi_assemble(m, kap, f)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        Ks, Fs = assemble_sparse(m, torch.as_tensor(kap), torch.as_tensor(f, device="cuda"))
        assert np.array_equal(Ks.values().cpu().numpy(), vals) and np.array_equal(Fs.cpu().numpy(), F)
        assert np.array_equal(Ks.crow_indices().cpu().numpy(), nm.csr(0)[0])
        assert np.array_equal(Ks.col_indices().cpu().numpy(), nm.csr(0)[1])
    rp, col = nm.csr(0)
    n = m.n_nodes
    Ko, Mg = _oracle_mats(name, _kap_rows(kap, 1, m.n_elements)[0])
    dK = abs(sp.csr_matrix((vals, col, rp), shape=(n, n)) - Ko).max(axis=1).toarray().ravel()
    sK = abs(Ko).max(axis=1).toarray().ravel()
    Fo = Mg @ f
    dF, sF = np.abs(F - Fo), abs(Mg) @ np.abs(f)
    # (rows that only the zero-area triangle touches have sK = sF = 0: there the kernels must give exact zeros)
    assert (dK <= 1e-13 * sK).all() and (dF <= 1e-13 * sF).all()
    ek, eF = (d[s > 0] / s[s > 0] for d, s in ((dK, sK), (dF, sF)))
    print(f"\n[{name}/{kind}] K {ek.max():.1e}  F {eF.max():.1e} (row-relative)")
    if name == "rect_one_cta":                   # the per-kappa assembly here is oracle_p2's own
        Kp, Fp, _, _ = P.assemble(m.nodes.numpy(), m.elements.numpy(), kap, f)
        assert abs(Kp - Ko).max() == 0 and np.array_equal(Fp, Fo)


# ================================================================================================ solve and gradients
SOLVE_CASES = [(c, lay) for c in ORACLE_CASES for lay in LAYOUTS if c != "rect_empty_cta" or lay == "sample_elem"]


@pytest.mark.parametrize("name,layout", SOLVE_CASES)
def test_solve_vs_oracle(name, layout):
    """u, dL/df and dL/dkappa through DifferentiableFESolver against the oracle in every kappa layout: a scalar, one
    field (n_el,), one scalar per sample (B, 1) and one field per sample (B, n_el).  Per-element gradients are held
    element by element to TOL2D * max_e |lam_e|^T |K0_e| |u_e| (lam: the oracle's adjoint), a bound that does not grow
    with the number of elements; summed ones to TOL2D * sum_e |dL/dkappa_e|."""
    m = _mesh(name)
    f, gbar, kap = _inputs(name, layout)
    u, gk, gf, s = run(m, kap, f, gbar)
    assert s._opts["last_solver2d"] == "jacobi" and all(it > 0 for it, _ in s.last_pcg)
    B = f.shape[0] if f.ndim == 2 else 1
    u, gf, f2, g2 = u.reshape(B, -1), gf.reshape(B, -1), f.reshape(B, -1), gbar.reshape(B, -1)
    krows = _kap_rows(kap, B, m.n_elements)
    worst = [0.0, 0.0, 0.0]
    for b in range(B):
        uo, gko, gfo, scale = _oracle(name, krows[b], f2[b], g2[b])
        eu, ef = relerr(u[b], uo), relerr(gf[b], gfo)
        if layout in ("scalar", "sample"):
            eg = abs(float(np.asarray(gk).reshape(B)[b]) - gko.sum()) / np.abs(gko).sum()
        else:
            eg = float(np.abs(gk.reshape(B, -1)[b] - gko).max() / scale)
        assert eu <= TOL2D and ef <= TOL2D and eg <= TOL2D, (b, eu, ef, eg)
        worst = [max(w, e) for w, e in zip(worst, (eu, ef, eg))]
    print(f"\n[{name}/{layout}] u {worst[0]:.1e} gf {worst[1]:.1e} gk {worst[2]:.1e}")


# ======================================================================================= exact quadratic reproduction
def _ustar(xy):
    x, y = xy[:, 0], xy[:, 1]
    return 1 + 0.3 * x - 0.2 * y + 0.5 * x ** 2 - 0.4 * x * y + 0.7 * y ** 2


@pytest.mark.parametrize("name", CASES_2D)
def test_quadratic_reproduction(name):
    """u* = 1 + 0.3x - 0.2y + 0.5x^2 - 0.4xy + 0.7y^2 with f = -kappa Lap u* = -2.4 kappa and u* on every Dirichlet
    vertex and midpoint: P2 on an affine triangulation reproduces u* exactly, so |u - u*| is the solver's error alone.
    On rect_two_trips, also the true residual of the system assembled through the C ABI.  Measured on a B200 (1000 W
    power limit): |u - u*| / max|u*| = 2.3e-12 on rect_two_trips (2203 iterations, true residual 1.3e-13 ||F_free||),
    3.0e-12 on rect_empty_cta, at most 1.5e-12 on the others."""
    m0 = _mesh(name)
    xy = m0.nodes.numpy()
    us = _ustar(xy)
    m = FEMesh(nodes=m0.nodes, elements=m0.elements, dirichlet_nodes={p: float(us[p]) for p in m0.dirichlet_nodes})
    kap = 1.3
    f = np.full(m.n_nodes, -2.4 * kap)
    u, _, _, s = run(m, kap, f, np.ones(m.n_nodes))
    err = float(np.abs(u - us).max() / np.abs(us).max())
    msg = f"\n[{name}] |u - u*| / max|u*| = {err:.1e} after {s.last_pcg[0][0]} iterations"
    assert err <= 1e-9, err
    if name == "rect_two_trips":
        nm, _, _, vf, Ff, _ = abi_assemble(m, kap, f)
        rpf, colf = nm.csr(1)
        Kf = sp.csr_matrix((vf, colf, rpf), shape=(len(Ff), len(Ff)))
        res = float(np.linalg.norm(Ff - Kf @ u[nm.free_nodes()]) / np.linalg.norm(Ff))
        msg += f", true residual {res:.1e}"
        assert res <= 1e-9, res
    print(msg)


# ======================================================================================= identities at the largest size
def test_adjoint_and_euler_identities_at_the_largest_size():
    """rect_two_trips, zero Dirichlet data, a positive kappa field, f and gbar: <gbar, u> = <dL/df, f> (the adjoint
    solve agrees with the forward one) and sum_e kappa_e dL/dkappa_e = -L (K is homogeneous of degree 1 in kappa), both
    to 1e-8 relative: each side carries the PCG error of its solve.  Measured on a B200: 0 and 8.1e-13."""
    m0 = _mesh("rect_two_trips")
    m = FEMesh(nodes=m0.nodes, elements=m0.elements, dirichlet_nodes={p: 0.0 for p in m0.dirichlet_nodes})
    rng = np.random.default_rng(41)
    f, gbar = rng.uniform(0.5, 1.0, m.n_nodes), rng.uniform(0.5, 1.0, m.n_nodes)
    kap = 10.0 ** rng.uniform(-2.0, 0.0, m.n_elements)
    u, gk, gf, s = run(m, kap, f, gbar)
    L = float(gbar @ u)
    e_adj = abs(float(gf @ f) - L) / abs(L)
    e_eul = abs(float(kap @ gk) + L) / abs(L)
    print(f"\n[rect_two_trips] adjoint {e_adj:.1e}  Euler {e_eul:.1e}  iterations {s.last_pcg[0][0]} / "
          f"{s._opts['last_pcg_adjoint'][0][0]}")
    assert e_adj <= 1e-8 and e_eul <= 1e-8, (e_adj, e_eul)


# ========================================================================================== invariance and bits
def _reorder(m, seed):
    """The mesh with each element's node order rotated or reflected at random, vertices and midpoints together
    ([v0, v1, v2, m01, m12, m20] under a vertex permutation pi is [v_pi0, v_pi1, v_pi2, m_pi0pi1, m_pi1pi2, m_pi2pi0])."""
    rng = np.random.default_rng(seed)
    perms = np.array([[0, 1, 2], [1, 2, 0], [2, 0, 1], [0, 2, 1], [2, 1, 0], [1, 0, 2]])
    mid = {frozenset((0, 1)): 3, frozenset((1, 2)): 4, frozenset((0, 2)): 5}
    full = np.array([list(p) + [mid[frozenset((p[k], p[(k + 1) % 3]))] for k in range(3)] for p in perms])
    el = m.elements.numpy()
    choice = rng.integers(0, 6, len(el))
    assert (choice >= 3).any() and (choice < 3).any()
    new = np.take_along_axis(el, full[choice], axis=1)
    return FEMesh(nodes=m.nodes, elements=torch.from_numpy(new), dirichlet_nodes=m.dirichlet_nodes)


INVARIANCE_CASES = ["rect_one_cta", "wheel", "delaunay", "graded", "degenerate"]


@pytest.mark.parametrize("name", INVARIANCE_CASES)
def test_element_node_order_invariance(name):
    """Rotating or reflecting each element's node order changes nothing but rounding: u and dL/dkappa within 1e-12 of
    their max norms (a reflected triangle has a negative signed area; the kernels take its absolute value).  Both solves
    run to a 1e-15 recursive residual: at the default 1e-13 the stopping error alone moves dL/dkappa on delaunay by
    ~1e-11 (float64 Jacobi-PCG on the CPU, against the oracle)."""
    m = _mesh(name)
    f, gbar, kap = _inputs(name, "elem", seed=3)
    u, gk, gf, _ = run(m, kap, f, gbar, pcg_tol=1e-15)
    u2, gk2, gf2, _ = run(_reorder(m, 5), kap, f, gbar, pcg_tol=1e-15)
    eu, eg, ef = relerr(u2, u), relerr(gk2, gk), relerr(gf2, gf)
    print(f"\n[{name}] reordered: u {eu:.1e} gk {eg:.1e} gf {ef:.1e}")
    assert eu <= 1e-12 and eg <= 1e-12 and ef <= 1e-12, (eu, eg, ef)


@pytest.mark.parametrize("name", ["rect_one_cta", "wheel", "delaunay", "line_p2_700"])
def test_batch_rows_and_repeats_are_bit_identical(name):
    """Row b of a batched solve with shared kappa (scalar and per element) is the single-sample solve of row b bit for
    bit (u and dL/df), and two identical calls return identical bits (u, dL/dkappa, dL/df)."""
    m = _mesh(name)
    for kind in ("scalar", "elem"):
        f, gbar, kap = _inputs(name, kind, seed=4)
        fb, gb, _ = _inputs(name, "sample", seed=4)
        u, gk, gf, _ = run(m, kap, fb, gb)
        for b in (0, fb.shape[0] - 1):
            u1, _, gf1, _ = run(m, kap, fb[b], gb[b])
            assert np.array_equal(u[b], u1) and np.array_equal(gf[b], gf1), (kind, b)
        u2, gk2, gf2, _ = run(m, kap, fb, gb)
        assert np.array_equal(u, u2) and np.array_equal(gk, gk2) and np.array_equal(gf, gf2), kind


def test_degenerate_triangle_is_skipped():
    """The zero-area triangle gets dL/dkappa = 0 exactly, and u on the nodes it shares with rectangle(9, 7).to_p2()
    equals the solution on that mesh (the two systems K_free differ only by structural zeros)."""
    m = _mesh("degenerate")
    base = _degenerate_p1().to_p2()
    f, gbar, kap = _inputs("degenerate", "elem", seed=6)
    u, gk, gf, _ = run(m, kap, f, gbar)
    assert gk[-1] == 0.0 and np.abs(gk[:-1]).min() > 0
    to_deg = np.empty(base.n_nodes, dtype=np.int64)
    to_deg[base.elements.numpy()] = m.elements.numpy()[:-1]
    ub, gkb, gfb, _ = run(base, kap[:-1], f[to_deg], gbar[to_deg])
    eu, eg = relerr(u[to_deg], ub), relerr(gk[:-1], gkb)
    print(f"\n[degenerate] against the mesh without the triangle: u {eu:.1e} gk {eg:.1e}")
    assert eu <= 1e-13 and eg <= 1e-13, (eu, eg)


# ========================================================================================================= routing
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("name", ["rect_one_cta", "graded", "line_p2_700"])
def test_route(name, layout):
    """A P2 forward + backward runs the general route's kernels (k_sum only to sum a scalar kappa's gradient) and none
    of the structured assembly, multigrid, one-CTA batch or banded kernels, in every kappa layout.  The pair runs twice
    under the profiler: in a long session the trace can miss the first launches of the window (k_assemble and
    k_eliminate of a one-sample solve were missing once after the whole GPU suite)."""
    m = _mesh(name)
    f, gbar, kap = _inputs(name, layout)
    _, names = _launched(lambda: [run(m, kap, f, gbar) for _ in range(2)])
    base = {k.split("<")[0] for k in names}
    want = {"k_assemble", "k_eliminate", "k_fill_sell", "k_pcg", "k_scatter", "k_gather", "k_grad_elem", "k_grad_f"}
    assert want <= base, (want - base, names)
    assert ("k_sum" in base) == (layout in ("scalar", "sample")), names
    banned = ("k_assemble_tile", "k_assemble_grid", "k_mgpcg", "k_batch", "k_band", "k_bps")
    assert not any(k.startswith(banned) for k in names), names


# ====================================================================================================== error path
def test_zero_row_raises_breakdown():
    """With the degenerate triangle's lone midpoint left free, K_free has a zero row there (1 / diag = inf): the solve
    raises BreakdownError instead of returning NaN."""
    m = _degenerate(free_mid=True)
    mid = int(m.elements[-1, 5])
    f, gbar, _ = _inputs("degenerate", "scalar")
    nm, _, _, vf, _, dinv = abi_assemble(m, 1.3, f)
    r = int(np.searchsorted(nm.free_nodes(), mid))
    rpf, _ = nm.csr(1)
    assert nm.free_nodes()[r] == mid and not vf[rpf[r]:rpf[r + 1]].any() and np.isinf(dinv[r])
    with pytest.raises(_native.BreakdownError):
        run(m, 1.3, f, gbar)
