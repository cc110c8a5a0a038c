"""CPU oracle for the differentiable-FEM hot path.  TEST INFRASTRUCTURE ONLY.

This module is a numpy/scipy float64 restatement of the reference algorithm in
``diffhe/solver.py`` (reference repo, cited as ``solver.py:LINE`` below).  It is
imported only by ``tests/``, ``__graft_entry__.smoke()`` and the CPU-baseline leg
of ``bench.py``.  Nothing under ``difffe_physics_lab_b200/`` may import it: the
product path is CUDA-only and fails loudly without its extension.

Parity status: PINNED.  ``tests/test_oracle_golden.py`` checks every function
here against (a) golden vectors produced by running the *unmodified* reference
in the build container (``tests/golden/make_golden.py``), including bit-exact
dense ``K``/``F``, and (b) the reference tests' own known answers
(``tests/test_fem.py:85-179`` upstream).

What is restated, and where it comes from
-----------------------------------------
* ``assemble_1d``/``assemble_2d``   solver.py:82-96 / solver.py:112-145 — the
  exact IEEE operation order of the element loop, accumulated in ascending
  element order (``np.add.at`` is unbuffered and sequential), so dense ``K`` and
  ``F`` are bit-identical to the reference's.
* ``structural_csr``                the set of (p,q) the reference *writes*
  (solver.py:89-92, :137-140): rows ascending, columns ascending.
* ``apply_bc``                      solver.py:162-171 (lifting in dict order,
  free-rank renumbering from mesh.py:127-129).
* ``solve_*``                       solver.py:174 (``torch.linalg.solve``): the
  oracle solves the *same float64 system* in higher precision (Decimal Thomas
  in 1D, sparse LU + extended-precision refinement in 2D), so it is the arbiter
  for the 1e-12 / 1e-9 parity bounds where the dense reference cannot run.
* ``adjoint_and_grads``             autograd of solver.py:88-96, :139-145, :169
  + ``LinalgSolveExBackward0`` written in closed form (SURVEY §8a rows A7/A8).
* ``forward_exact``/``grads_1d_exact``  1-D chains: the same solve and gradients kept in 50 digits until the
  final rounding (dL/dkappa_e differences neighbouring values: at n_el ~ 1e5 the float64 version costs ~1e-12).
* per-element kappa                 the reference loop with ``kappa`` replaced
  by ``kappa[e]`` at solver.py:88 / :139 (extension; the reference itself raises).
"""
from __future__ import annotations

from decimal import Decimal, getcontext
from typing import Dict, Optional, Sequence, Tuple

import numpy as np

AREA_EPS = 1e-15  # solver.py:120


# --------------------------------------------------------------------------- mesh
def line_mesh(n_elements: int, x_left=0.0, x_right=1.0, bc_left=0.0, bc_right=0.0):
    """mesh.py:58-77.  Nodes come from torch.linspace (NOT i/n): use torch."""
    import torch

    x = torch.linspace(x_left, x_right, n_elements + 1, dtype=torch.float64).numpy().copy()
    nodes = x.reshape(-1, 1)
    idx = np.arange(n_elements, dtype=np.int64)
    elements = np.stack([idx, idx + 1], axis=1)
    bc: Dict[int, float] = {}
    if bc_left is not None:
        bc[0] = bc_left
    if bc_right is not None:
        bc[n_elements] = bc_right
    return nodes, elements, bc


def rectangle_mesh(nx: int, ny: int, x_range=(0.0, 1.0), y_range=(0.0, 1.0), bc_value=0.0):
    """mesh.py:79-121 vectorised (node id row*(nx+1)+col; tris [a,b,d],[b,c,d])."""
    xs = np.linspace(x_range[0], x_range[1], nx + 1)
    ys = np.linspace(y_range[0], y_range[1], ny + 1)
    xx, yy = np.meshgrid(xs, ys)
    coords = np.stack([xx.ravel(), yy.ravel()], axis=1)
    i, j = np.meshgrid(np.arange(ny), np.arange(nx), indexing="ij")
    a = (i * (nx + 1) + j).ravel()
    b = a + 1
    c = a + nx + 2
    d = a + nx + 1
    tris = np.empty((2 * nx * ny, 3), dtype=np.int64)
    tris[0::2] = np.stack([a, b, d], axis=1)
    tris[1::2] = np.stack([b, c, d], axis=1)
    x, y = coords[:, 0], coords[:, 1]
    on = (
        np.isclose(x, x_range[0])
        | np.isclose(x, x_range[1])
        | np.isclose(y, y_range[0])
        | np.isclose(y, y_range[1])
    )
    bc = {int(k): bc_value for k in np.nonzero(on)[0]}
    return coords, tris, bc


def free_nodes(n_nodes: int, bc: Dict[int, float]) -> np.ndarray:
    """mesh.py:127-129 (ascending)."""
    mask = np.ones(n_nodes, dtype=bool)
    if bc:
        mask[np.fromiter(bc.keys(), dtype=np.int64)] = False
    return np.nonzero(mask)[0]


# ----------------------------------------------------------------- element kernels
def _kappa_e(kappa, n_el):
    kappa = np.asarray(kappa, dtype=np.float64)
    if kappa.ndim == 0 or kappa.size == 1:
        return np.full(n_el, float(kappa.reshape(-1)[0]))
    assert kappa.shape == (n_el,)
    return kappa


def element_1d(nodes, elements, kappa):
    """solver.py:84-88: h = xj - xi ; k_e = kappa / h."""
    x = nodes[:, 0]
    i, j = elements[:, 0], elements[:, 1]
    h = x[j] - x[i]
    k = _kappa_e(kappa, len(elements)) / h
    return h, k


def element_2d(nodes, elements, kappa):
    """solver.py:119-140.  Returns area, b(3), c(3), k_local(n_el,3,3), keep mask."""
    x, y = nodes[:, 0], nodes[:, 1]
    i, j, k = elements[:, 0], elements[:, 1], elements[:, 2]
    xi, yi, xj, yj, xk, yk = x[i], y[i], x[j], y[j], x[k], y[k]
    area = 0.5 * np.abs((xj - xi) * (yk - yi) - (xk - xi) * (yj - yi))
    keep = ~(area < AREA_EPS)
    b = np.stack([yj - yk, yk - yi, yi - yj], axis=1)
    c = np.stack([xk - xj, xi - xk, xj - xi], axis=1)
    kap = _kappa_e(kappa, len(elements))
    with np.errstate(divide="ignore", invalid="ignore"):
        bb = b[:, :, None] * b[:, None, :] + c[:, :, None] * c[:, None, :]
        kloc = (kap[:, None, None] * bb) / (4.0 * area)[:, None, None]
    return area, b, c, kloc, keep


# ------------------------------------------------------------------ dense assembly
def assemble_dense(nodes, elements, kappa, f):
    """Dense K (n,n), F (n,) exactly as solver.py:79-96 / :109-145 build them."""
    n = nodes.shape[0]
    f = np.asarray(f, dtype=np.float64)
    K = np.zeros((n, n))
    F = np.zeros(n)
    if nodes.shape[1] == 1:
        h, k = element_1d(nodes, elements, kappa)
        i, j = elements[:, 0], elements[:, 1]
        rows = np.stack([i, i, j, j], axis=1).ravel()
        cols = np.stack([i, j, i, j], axis=1).ravel()  # (i,i),(i,j),(j,i),(j,j)
        vals = np.stack([k, -k, -k, k], axis=1).ravel()
        np.add.at(K, (rows, cols), vals)
        hh = h / 2.0
        np.add.at(F, np.stack([i, j], axis=1).ravel(), np.stack([hh * f[i], hh * f[j]], axis=1).ravel())
    else:
        area, b, c, kloc, keep = element_2d(nodes, elements, kappa)
        el = elements[keep]
        rows = np.repeat(el, 3, axis=1).ravel()          # p repeated for q=0..2
        cols = np.tile(el, (1, 3)).ravel()
        np.add.at(K, (rows, cols), kloc[keep].reshape(-1))
        fc = ((f[el[:, 0]] + f[el[:, 1]]) + f[el[:, 2]]) / 3.0
        load = (area[keep] / 3.0) * fc
        np.add.at(F, el.ravel(), np.repeat(load, 3))
    return K, F


# -------------------------------------------------------------------- CSR assembly
def structural_csr(n_nodes: int, elements: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """Pattern {(p,q): some element contains p and q}; rows/cols ascending.

    Degenerate (skipped) elements are NOT removed from the pattern: the pattern
    is a function of connectivity alone, values there are exact zeros.
    """
    npe = elements.shape[1]
    rows = np.repeat(elements, npe, axis=1).ravel()
    cols = np.tile(elements, (1, npe)).ravel()
    key = np.unique(rows.astype(np.int64) * n_nodes + cols)
    r = key // n_nodes
    c = key % n_nodes
    rowptr = np.zeros(n_nodes + 1, dtype=np.int64)
    np.add.at(rowptr, r + 1, 1)
    rowptr = np.cumsum(rowptr)
    return rowptr, c.astype(np.int64)


def assemble_csr(nodes, elements, kappa, f):
    """CSR values on the structural pattern, accumulated in ascending element
    order (bit-identical to the dense reference at pattern positions)."""
    n = nodes.shape[0]
    f = np.asarray(f, dtype=np.float64)
    rowptr, col = structural_csr(n, elements)
    key = np.repeat(np.arange(n), np.diff(rowptr)) * n + col
    vals = np.zeros(len(col))
    F = np.zeros(n)

    def pos(rows, cols):
        return np.searchsorted(key, rows.astype(np.int64) * n + cols)

    if nodes.shape[1] == 1:
        h, k = element_1d(nodes, elements, kappa)
        i, j = elements[:, 0], elements[:, 1]
        rows = np.stack([i, i, j, j], axis=1).ravel()
        cols = np.stack([i, j, i, j], axis=1).ravel()
        v = np.stack([k, -k, -k, k], axis=1).ravel()
        np.add.at(vals, pos(rows, cols), v)
        hh = h / 2.0
        np.add.at(F, np.stack([i, j], axis=1).ravel(), np.stack([hh * f[i], hh * f[j]], axis=1).ravel())
    else:
        area, b, c, kloc, keep = element_2d(nodes, elements, kappa)
        el = elements[keep]
        rows = np.repeat(el, 3, axis=1).ravel()
        cols = np.tile(el, (1, 3)).ravel()
        np.add.at(vals, pos(rows, cols), kloc[keep].reshape(-1))
        fc = ((f[el[:, 0]] + f[el[:, 1]]) + f[el[:, 2]]) / 3.0
        load = (area[keep] / 3.0) * fc
        np.add.at(F, el.ravel(), np.repeat(load, 3))
    return rowptr, col, vals, F


def apply_bc(rowptr, col, vals, F, bc: Dict[int, float]):
    """solver.py:162-171 on CSR.  Returns (free, rowptr_f, col_f, vals_f, F_free).

    Lifting: for each Dirichlet (d,g) in dict order, F_free[fi] -= K[f,d]*g; only
    structurally coupled rows change (K[f,d] is an exact 0 elsewhere).
    ``col_f`` is renumbered by rank in ``free_nodes()``.
    """
    n = len(rowptr) - 1
    free = free_nodes(n, bc)
    rank = -np.ones(n, dtype=np.int64)
    rank[free] = np.arange(len(free))
    Fw = F.copy()
    row_of = np.repeat(np.arange(n), np.diff(rowptr))
    if bc:
        order = {d: t for t, d in enumerate(bc.keys())}
        isd = np.zeros(n, dtype=bool)
        isd[list(bc.keys())] = True
        sel = np.nonzero(isd[col] & ~isd[row_of])[0]
        t = np.array([order[int(d)] for d in col[sel]], dtype=np.int64)
        g = np.array([bc[int(d)] for d in col[sel]], dtype=np.float64)
        o = np.argsort(t, kind="stable")
        # sequential in dict order: F[row] = F[row] - K*g
        np.add.at(Fw, row_of[sel][o], -(vals[sel][o] * g[o]))
    keepnz = (rank[row_of] >= 0) & (rank[col] >= 0)
    col_f = rank[col[keepnz]]
    vals_f = vals[keepnz]
    cnt = np.zeros(len(free) + 1, dtype=np.int64)
    np.add.at(cnt, rank[row_of[keepnz]] + 1, 1)
    rowptr_f = np.cumsum(cnt)
    return free, rowptr_f, col_f, vals_f, Fw[free]


# --------------------------------------------------------------------------- solves
def _thomas_decimal(a, d, c, b, prec=50):
    """Tridiagonal solve in ``prec``-digit decimal arithmetic (arbiter)."""
    return np.array([float(v) for v in _thomas_decimal_exact(a, d, c, b, prec)])


def _thomas_decimal_exact(a, d, c, b, prec=50):
    """``_thomas_decimal`` without the final rounding: the ``prec``-digit solution as a list of Decimals."""
    getcontext().prec = prec
    n = len(d)
    if n == 0:
        return []
    a = [Decimal(float(v)) for v in a]
    d = [Decimal(float(v)) for v in d]
    c = [Decimal(float(v)) for v in c]
    b = [Decimal(float(v)) for v in b]
    cp = [Decimal(0)] * n
    bp = [Decimal(0)] * n
    cp[0] = c[0] / d[0]
    bp[0] = b[0] / d[0]
    for i in range(1, n):
        m = d[i] - a[i] * cp[i - 1]
        cp[i] = c[i] / m
        bp[i] = (b[i] - a[i] * bp[i - 1]) / m
    x = [Decimal(0)] * n
    x[-1] = bp[-1]
    for i in range(n - 2, -1, -1):
        x[i] = bp[i] - cp[i] * x[i + 1]
    return x


def _is_tridiagonal(rowptr, col):
    row_of = np.repeat(np.arange(len(rowptr) - 1), np.diff(rowptr))
    return bool(np.all(np.abs(row_of - col) <= 1))


def solve_csr(rowptr, col, vals, rhs, exact=True):
    """Solve the float64 system accurately (<=1e-15 rel) — replaces solver.py:174.

    Tridiagonal systems: Decimal Thomas when ``exact`` (else scipy banded).
    Everything else: sparse LU + refinement with an extended-precision residual.
    """
    import scipy.sparse as sp
    import scipy.sparse.linalg as spla

    n = len(rowptr) - 1
    if n == 0:
        return np.zeros(0)
    if _is_tridiagonal(rowptr, col):
        A = sp.csr_matrix((vals, col, rowptr), shape=(n, n))
        d = A.diagonal()
        lo = np.concatenate([[0.0], A.diagonal(-1)])
        up = np.concatenate([A.diagonal(1), [0.0]])
        if exact:
            return _thomas_decimal(lo, d, up, rhs)
        from scipy.linalg import solve_banded

        ab = np.zeros((3, n))
        ab[0, 1:] = up[:-1]
        ab[1] = d
        ab[2, :-1] = lo[1:]
        return solve_banded((1, 1), ab, rhs)
    A = sp.csc_matrix(sp.csr_matrix((vals, col, rowptr), shape=(n, n)))
    lu = spla.splu(A)
    x = lu.solve(rhs)
    if exact:
        row_of = np.repeat(np.arange(n), np.diff(rowptr))
        vl = vals.astype(np.longdouble)
        for _ in range(3):
            ax = np.zeros(n, dtype=np.longdouble)
            np.add.at(ax, row_of, vl * x.astype(np.longdouble)[col])
            r = (rhs.astype(np.longdouble) - ax).astype(np.float64)
            x = (x.astype(np.longdouble) + lu.solve(r).astype(np.longdouble)).astype(np.float64)
    return x


def forward(nodes, elements, bc, kappa, f, exact=True):
    """u = DifferentiableFESolver(mesh, kappa)(f)  (solver.py:49-67,153-183)."""
    n = nodes.shape[0]
    rowptr, col, vals, F = assemble_csr(nodes, elements, kappa, f)
    free, rp, cf, vf, Ff = apply_bc(rowptr, col, vals, F, bc)
    u_free = solve_csr(rp, cf, vf, Ff, exact=exact)
    u = np.zeros(n)
    for d, g in bc.items():
        u[d] = g
    u[free] = u_free
    return u


def adjoint_and_grads(nodes, elements, bc, kappa, u, gbar, exact=True):
    """Closed-form backward (SURVEY §8a rows A7/A8).

    Returns (g_kappa_per_element, g_f, lam_full).  Scalar kappa: sum g_kappa.
      lam_free = K_free^{-T} gbar_free  (K symmetric)
      dL/dkappa_e = -lam_e^T K_e^0 u_e   with lam = 0, u = g on Dirichlet nodes
      1D: dL/df_i = lam_i (h_{i-1}+h_i)/2 ;  2D: dL/df_q = sum_{e∋q} area_e/9 * sum_{p∈e} lam_p
    """
    n = nodes.shape[0]
    n_el = len(elements)
    rowptr, col, vals, _ = assemble_csr(nodes, elements, kappa, np.zeros(n))
    free, rp, cf, vf, _ = apply_bc(rowptr, col, vals, np.zeros(n), {k: 0.0 for k in bc})
    lam = np.zeros(n)
    lam[free] = solve_csr(rp, cf, vf, np.asarray(gbar, dtype=np.float64)[free], exact=exact)
    if nodes.shape[1] == 1:
        h, _ = element_1d(nodes, elements, 1.0)
        i, j = elements[:, 0], elements[:, 1]
        gk = -(lam[j] - lam[i]) * (u[j] - u[i]) / h
        gf = np.zeros(n)
        np.add.at(gf, i, (h / 2.0) * lam[i])
        np.add.at(gf, j, (h / 2.0) * lam[j])
    else:
        area, b, c, _, keep = element_2d(nodes, elements, 1.0)
        el = elements
        bl = (b * lam[el]).sum(1)
        bu = (b * u[el]).sum(1)
        cl = (c * lam[el]).sum(1)
        cu = (c * u[el]).sum(1)
        with np.errstate(divide="ignore", invalid="ignore"):
            gk = np.where(keep, -(bl * bu + cl * cu) / (4.0 * area), 0.0)
        gf = np.zeros(n)
        contrib = np.where(keep, (area / 9.0) * lam[el].sum(1), 0.0)
        np.add.at(gf, el.ravel(), np.repeat(contrib, 3))
    assert gk.shape == (n_el,)
    return gk, gf, lam


# ------------------------------------------------ 1-D gradients without float64 rounding
def _tridiag_free(nodes, elements, bc, kappa, f):
    """The float64 system K_free u_free = F_free of a 1-D chain as (free, lower, diagonal, upper, rhs)."""
    import scipy.sparse as sp

    rowptr, col, vals, F = assemble_csr(nodes, elements, kappa, f)
    free, rp, cf, vf, Ff = apply_bc(rowptr, col, vals, F, bc)
    assert _is_tridiagonal(rp, cf), "a 1-D chain has a tridiagonal K_free"
    A = sp.csr_matrix((vf, cf, rp), shape=(len(free), len(free)))
    lo = np.concatenate([[0.0], A.diagonal(-1)])
    up = np.concatenate([A.diagonal(1), [0.0]])
    return free, lo, A.diagonal(), up, Ff


def forward_exact(nodes, elements, bc, kappa, f, prec=50):
    """``forward`` on a 1-D chain, unrounded: the ``prec``-digit solution of the float64 system as a list of Decimals
    (Dirichlet nodes hold their data exactly)."""
    free, lo, d, up, rhs = _tridiag_free(nodes, elements, bc, kappa, f)
    u = [Decimal(0)] * nodes.shape[0]
    for k, g in bc.items():
        u[k] = Decimal(float(g))
    for i, v in zip(free, _thomas_decimal_exact(lo, d, up, rhs, prec)):
        u[i] = v
    return u


def grads_1d_exact(nodes, elements, bc, kappa, u, gbar, prec=50):
    """``adjoint_and_grads`` on a 1-D chain with every step after the float64 system in ``prec``-digit arithmetic.

    ``u`` is a float64 vector (converted exactly: e.g. a kernel's stored solution) or the Decimal list of
    ``forward_exact``.  Returns (gk, gf, lam): gk_e = -(lam_j - lam_i)(u_j - u_i)/h_e and
    gf_i = sum_{e ∋ i} (h_e/2) lam_i, each formed from the unrounded lam and rounded once; lam is the ``prec``-digit adjoint
    (list of Decimals, 0 on Dirichlet nodes).  The float64 ``adjoint_and_grads`` rounds lam and u first and differences the
    rounded values: at n_el = 1e5 that alone moves gk by ~1e-12 relative (DESIGN.md §3.1b).
    """
    n = nodes.shape[0]
    free, lo, d, up, rhs = _tridiag_free(nodes, elements, {k: 0.0 for k in bc}, kappa, np.zeros(n))
    rhs = np.asarray(gbar, dtype=np.float64)[free]
    getcontext().prec = prec
    lam = [Decimal(0)] * n
    for i, v in zip(free, _thomas_decimal_exact(lo, d, up, rhs, prec)):
        lam[i] = v
    ud = u if (len(u) and isinstance(u[0], Decimal)) else [Decimal(float(v)) for v in np.asarray(u, dtype=np.float64)]
    h, _ = element_1d(nodes, elements, 1.0)
    gk = np.empty(len(elements))
    gf = [Decimal(0)] * n
    for e, (i, j) in enumerate(elements.tolist()):
        he = Decimal(float(h[e]))
        gk[e] = float(-(lam[j] - lam[i]) * (ud[j] - ud[i]) / he)
        gf[i] += he / 2 * lam[i]
        gf[j] += he / 2 * lam[j]
    return gk, np.array([float(v) for v in gf]), lam


# ------------------------------------------------- reference Jacobi-PCG (2D timing)
def jacobi_pcg(rowptr, col, vals, rhs, tol=1e-13, maxit=100000):
    """Plain float64 Jacobi-PCG to recursive ||r||/||b|| < tol (CPU baseline and
    iteration-count reference for the CUDA solver)."""
    import scipy.sparse as sp

    n = len(rowptr) - 1
    A = sp.csr_matrix((vals, col, rowptr), shape=(n, n))
    dinv = 1.0 / A.diagonal()
    x = np.zeros(n)
    r = rhs.copy()
    bn = np.sqrt(rhs @ rhs)
    if bn == 0.0:
        return x, 0, 0.0
    z = dinv * r
    p = z.copy()
    rz = r @ z
    it = 0
    while it < maxit:
        q = A @ p
        alpha = rz / (p @ q)
        x += alpha * p
        r -= alpha * q
        it += 1
        rn = np.sqrt(r @ r)
        if rn <= tol * bn:
            break
        z = dinv * r
        rz_new = r @ z
        p = z + (rz_new / rz) * p
        rz = rz_new
    return x, it, float(np.sqrt(r @ r) / bn)
