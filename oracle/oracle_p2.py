"""CPU oracle for the P2 (quadratic Lagrange) extension of the hot path.  TEST INFRASTRUCTURE ONLY.

Parity status: UNPINNED BY CONSTRUCTION.  The reference has no P2 elements — they are an unchecked item of its roadmap
(reference ``README.md:139-143``; SURVEY §8(f) N4: "none exists upstream, so no parity burden").  The conventions below
are therefore this repo's own, chosen to continue the reference's P1 code (``diffhe/solver.py:73-183``) in the obvious
way; the oracle is anchored on closed-form solutions instead of golden vectors (``tests/test_p2_oracle.py``).

Conventions
-----------
* 1-D element ``[left, right, mid]``, 2-D element ``[v0, v1, v2, m01, m12, m20]`` (vertices, then the midpoints of the
  edges (0,1), (1,2), (2,0)); geometry is affine and read from the VERTICES only (like ``solver.py:84-85`` / ``:114-134``).
* ``K_e = kappa_e * int grad(phi_i) . grad(phi_j)`` exactly; degenerate triangles (area < 1e-15) are skipped (``:120-121``).
* load ``F = M f`` with the consistent P2 mass matrix (f is interpolated in the element's own space) — the P1 code's
  nodal / centroid rules (``:95-96``, ``:143-145``) are only first-order accurate and would cap the P2 convergence rate.
* Dirichlet lifting, free-node numbering and scatter as ``solver.py:162-181``.

Everything here is computed with numerical quadrature (Gauss points on the interval, a degree-4 rule on the triangle):
an implementation independent of the closed-form element matrices inside the CUDA kernels it checks.
"""
from __future__ import annotations

from typing import Dict

import numpy as np
import scipy.sparse as sp
import scipy.sparse.linalg as spla

# ----------------------------------------------------------------------------------------------- meshes (test helpers)


def line_p2(n_elements: int, x_left=0.0, x_right=1.0, bc_left=0.0, bc_right=0.0):
    """Vertices 0..n (np.linspace), then the element midpoints n+1..2n; elements [e, e+1, n+1+e]."""
    xv = np.linspace(x_left, x_right, n_elements + 1)
    xm = 0.5 * (xv[:-1] + xv[1:])
    nodes = np.concatenate((xv, xm))[:, None]
    e = np.arange(n_elements, dtype=np.int64)
    elements = np.stack((e, e + 1, n_elements + 1 + e), axis=1)
    bc: Dict[int, float] = {}
    if bc_left is not None:
        bc[0] = bc_left
    if bc_right is not None:
        bc[n_elements] = bc_right
    return nodes, elements, bc


# ----------------------------------------------------------------------------------------------- shape functions

_G3 = (np.array([-np.sqrt(0.6), 0.0, np.sqrt(0.6)]), np.array([5.0, 8.0, 5.0]) / 9.0)   # exact to degree 5 on [-1, 1]


def _shape_1d(xi):
    """P2 shape functions on [0, 1] in the order (left, right, mid) and their xi-derivatives."""
    N = np.array([(1 - xi) * (1 - 2 * xi), xi * (2 * xi - 1), 4 * xi * (1 - xi)])
    dN = np.array([4 * xi - 3, 4 * xi - 1, 4 - 8 * xi])
    return N, dN


# Dunavant degree-4 rule (6 points), barycentric coordinates and weights (sum = 1)
_a1, _w1 = 0.445948490915965, 0.223381589678011
_a2, _w2 = 0.091576213509771, 0.109951743655322
_TRI_PTS = np.array([[1 - 2 * _a1, _a1, _a1], [_a1, 1 - 2 * _a1, _a1], [_a1, _a1, 1 - 2 * _a1],
                     [1 - 2 * _a2, _a2, _a2], [_a2, 1 - 2 * _a2, _a2], [_a2, _a2, 1 - 2 * _a2]])
_TRI_W = np.array([_w1, _w1, _w1, _w2, _w2, _w2])
_EDGES = ((0, 1), (1, 2), (2, 0))


def _shape_2d(lam, glam):
    """P2 shape functions (6,) and gradients (..., 6, 2) at barycentric point lam (3,), glam = grad lambda (..., 3, 2)."""
    N = np.empty(6)
    G = np.empty(glam.shape[:-2] + (6, 2))
    for i in range(3):
        N[i] = lam[i] * (2 * lam[i] - 1)
        G[..., i, :] = (4 * lam[i] - 1) * glam[..., i, :]
    for k, (i, j) in enumerate(_EDGES):
        N[3 + k] = 4 * lam[i] * lam[j]
        G[..., 3 + k, :] = 4 * (lam[i] * glam[..., j, :] + lam[j] * glam[..., i, :])
    return N, G


def element_matrices(nodes, elements):
    """(K0_e, M_e) for every element: stiffness at kappa = 1 and consistent mass, shapes (n_el, npe, npe).  The
    quadrature is applied to all elements at once (one pass per quadrature point), so meshes of 1e5 elements take a
    fraction of a second."""
    nodes = np.asarray(nodes, dtype=np.float64)
    elements = np.asarray(elements, dtype=np.int64)
    ne, npe = elements.shape
    K0 = np.zeros((ne, npe, npe))
    M = np.zeros((ne, npe, npe))
    if nodes.shape[1] == 1:
        assert npe == 3
        gp, gw = 0.5 * (_G3[0] + 1.0), 0.5 * _G3[1]
        h = nodes[elements[:, 1], 0] - nodes[elements[:, 0], 0]
        for xi, w in zip(gp, gw):
            N, dN = _shape_1d(xi)
            K0 += (w * np.outer(dN, dN))[None] / h[:, None, None]
            M += w * h[:, None, None] * np.outer(N, N)[None]
    else:
        assert npe == 6
        P = nodes[elements[:, :3]]                                       # (ne, 3 vertices, 2)
        J = np.stack((P[:, 1] - P[:, 0], P[:, 2] - P[:, 0]), axis=2)      # J[e] = [[x1-x0, x2-x0], [y1-y0, y2-y0]]
        det = J[:, 0, 0] * J[:, 1, 1] - J[:, 0, 1] * J[:, 1, 0]
        area = 0.5 * np.abs(det)
        keep = ~(area < 1e-15)                                          # degenerate triangles contribute nothing
        Jinv = np.linalg.inv(J[keep])                                   # rows: gradients of lambda_1, lambda_2
        glam = np.stack((-(Jinv[:, 0] + Jinv[:, 1]), Jinv[:, 0], Jinv[:, 1]), axis=1)   # (nk, 3, 2)
        a = area[keep][:, None, None]
        Kk = np.zeros((len(glam), 6, 6))
        Mk = np.zeros((len(glam), 6, 6))
        for lam, w in zip(_TRI_PTS, _TRI_W):
            N, G = _shape_2d(lam, glam)
            Kk += w * a * np.einsum("eik,ejk->eij", G, G)
            Mk += w * a * np.outer(N, N)[None]
        K0[keep] = Kk
        M[keep] = Mk
    return K0, M


# ----------------------------------------------------------------------------------------------- the path


def assemble(nodes, elements, kappa, f):
    """Sparse K (csr, all nodes), F = M f, and the assembled mass matrix."""
    elements = np.asarray(elements, dtype=np.int64)
    n = np.asarray(nodes).shape[0]
    ne, npe = elements.shape
    kap = np.broadcast_to(np.asarray(kappa, dtype=np.float64).reshape(-1), (ne,)) if np.ndim(kappa) else np.full(ne, float(kappa))
    K0, M = element_matrices(nodes, elements)
    rows = np.repeat(elements, npe, axis=1).ravel()
    cols = np.tile(elements, (1, npe)).ravel()
    K = sp.csr_matrix(((kap[:, None, None] * K0).ravel(), (rows, cols)), shape=(n, n))
    Mg = sp.csr_matrix((M.ravel(), (rows, cols)), shape=(n, n))
    return K, Mg @ np.asarray(f, dtype=np.float64), Mg, K0


def forward(nodes, elements, bc: Dict[int, float], kappa, f):
    """u on all nodes (solver.py:162-181 with the P2 system)."""
    K, F, _, _ = assemble(nodes, elements, kappa, f)
    n = K.shape[0]
    d = np.fromiter(bc.keys(), dtype=np.int64, count=len(bc))
    g = np.fromiter(bc.values(), dtype=np.float64, count=len(bc))
    free = np.setdiff1d(np.arange(n), d)
    u = np.zeros(n)
    u[d] = g
    rhs = F[free] - K[free][:, d] @ g
    Kff = K[free][:, free].tocsc()
    lu = spla.splu(Kff)
    x = lu.solve(rhs)
    for _ in range(2):                                   # iterative refinement
        x = x + lu.solve(rhs - Kff @ x)
    u[free] = x
    return u


def adjoint_and_grads(nodes, elements, bc: Dict[int, float], kappa, u, gbar):
    """(dL/dkappa_e (n_el,), dL/df (n_nodes,)) for an upstream gradient gbar = dL/du (entries at Dirichlet nodes dropped)."""
    K, _, Mg, K0 = assemble(nodes, elements, kappa, np.zeros(np.asarray(nodes).shape[0]))
    n = K.shape[0]
    elements = np.asarray(elements, dtype=np.int64)
    d = np.fromiter(bc.keys(), dtype=np.int64, count=len(bc))
    free = np.setdiff1d(np.arange(n), d)
    Kff = K[free][:, free].tocsc()
    lu = spla.splu(Kff)
    rhs = np.asarray(gbar, dtype=np.float64)[free]
    x = lu.solve(rhs)
    x = x + lu.solve(rhs - Kff @ x)
    lam = np.zeros(n)
    lam[free] = x
    ue, le = np.asarray(u)[elements], lam[elements]
    gk = -np.einsum("ei,eij,ej->e", le, K0, ue)
    return gk, Mg @ lam
