"""The 50-digit 1-D gradient reference (``oracle.forward_exact`` / ``oracle.grads_1d_exact``).

``adjoint_and_grads`` rounds lam and u to float64 and then forms dL/dkappa_e = -(lam_j - lam_i)(u_j - u_i)/h_e from
the rounded values.  At n_el ~ 1e5 that cancellation costs about 1e-12 relative, as much as the 1-D parity tolerance.
``grads_1d_exact`` forms both differences in 50-digit arithmetic and rounds once, so a kernel's gradient can be checked
at 1e-12 against the exact gradient of the kernel's own stored u (tests/test_gpu_1d_per_element.py).
"""
from decimal import Decimal

import numpy as np
import pytest

from oracle import oracle as O

LINE_CASES = ["c1_line20", "line10_bc12_rand", "line40_rand", "line8_left_only", "line8_right_only", "line2_bc",
              "line3_bc", "line100_ones", "line400_ones"]


def l1rel(a, b):
    return float(np.abs(a - b).sum() / np.abs(b).sum())


def maxrel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


@pytest.mark.parametrize("name", LINE_CASES)
def test_agrees_with_float64_adjoint_on_golden_lines(golden, name):
    c = golden.case(name)
    nodes, el, bc, kap = c["nodes"], c["elements"], c["bc"], float(c["kappa"])
    ue = O.forward_exact(nodes, el, bc, kap, c["f"])
    assert all(isinstance(v, Decimal) for v in ue) and len(ue) == nodes.shape[0]
    u = O.forward(nodes, el, bc, kap, c["f"])
    assert np.array_equal(np.array([float(v) for v in ue]), u)        # forward == forward_exact rounded once
    assert all(ue[k] == Decimal(float(g)) for k, g in bc.items())
    gk, gf, lam = O.adjoint_and_grads(nodes, el, bc, kap, u, c["gbar"])
    for uin in (ue, u):
        gke, gfe, lame = O.grads_1d_exact(nodes, el, bc, kap, uin, c["gbar"])
        assert np.array_equal(np.array([float(v) for v in lame]), lam)
        assert all(lame[k] == 0 for k in bc)
        # float64 error of adjoint_and_grads at n <= 400: a few ulps of lam and u, amplified by the differences
        assert maxrel(gk, gke) <= 1e-13
        assert maxrel(gf, gfe) <= 1e-15
        assert abs(gke.sum() - float(c["gkappa"])) <= 1e-10 * np.abs(gke).sum()   # the reference's own LU noise
        assert maxrel(gfe, c["gf"]) <= 1e-11


@pytest.mark.parametrize("n", [1, 2, 7, 64])
@pytest.mark.parametrize("kap", [1.0, 2.7])
def test_closed_form_quadratic(n, kap):
    """kappa uniform, f = gbar = 1, zero Dirichlet data on line(n): u_i = x_i(1 - x_i)/(2 kappa) is nodally exact,
    lam = u/h (the adjoint right-hand side is gbar itself, not h*gbar), so dL/dkappa_e = -(1 - x_i - x_j)^2/(4 kappa^2)
    and dL/df_i = h lam_i = u_i (interior nodes)."""
    nodes, el, bc = O.line_mesh(n)
    x = np.arange(n + 1) / n                       # exact i/n; the mesh's linspace nodes differ by ulps
    one = np.ones(n + 1)
    ue = O.forward_exact(nodes, el, bc, kap, one)
    gk, gf, lam = O.grads_1d_exact(nodes, el, bc, kap, ue, one)
    u_cf = x * (1 - x) / (2 * kap)
    if n > 1:
        assert maxrel(np.array([float(v) for v in ue]), u_cf) <= 1e-13
        assert maxrel(gf, u_cf) <= 1e-13
        assert maxrel(np.array([float(v) for v in lam]), u_cf * n) <= 1e-13
    gk_cf = -((1 - x[:-1] - x[1:]) ** 2) / (4 * kap * kap)
    assert np.abs(gk - gk_cf).max() <= 1e-12 * np.abs(gk_cf).max()
    assert gf[0] == 0.0 and gf[-1] == 0.0


def test_float64_reference_error_split():
    """The cost of rounding before differencing, on line(30000, bc_left=0.1, bc_right=None), kappa ~ logU[0.1, 10],
    f ~ U(0, 1), gbar ~ N(0, 1), seed 1 (the n_el = 1e5 figures of the same set-up are in DESIGN.md §3.1b).
    Rows: the float64 oracle, the exact flux on the float64-rounded u, and the float64 oracle against the exact flux on
    the same given u — each as (L1 relative, max-entry relative to max |gk|), pinned to two digits."""
    n = 30000
    rng = np.random.default_rng(1)
    nodes, el, bc = O.line_mesh(n, bc_left=0.1, bc_right=None)
    kap = np.exp(rng.uniform(np.log(0.1), np.log(10.0), n))
    f = rng.uniform(0, 1, n + 1)
    gbar = rng.standard_normal(n + 1)
    ue = O.forward_exact(nodes, el, bc, kap, f)
    u64 = np.array([float(v) for v in ue])
    assert np.array_equal(u64, O.forward(nodes, el, bc, kap, f))
    gke, gfe, _ = O.grads_1d_exact(nodes, el, bc, kap, ue, gbar)
    gko, gfo, _ = O.adjoint_and_grads(nodes, el, bc, kap, u64, gbar)
    gku, gfu, _ = O.grads_1d_exact(nodes, el, bc, kap, u64, gbar)
    assert np.array_equal(gfu, gfe)                      # dL/df does not depend on u
    assert maxrel(gfo, gfe) <= 1e-15

    def two(v):
        return float(f"{v:.2g}")

    assert (two(l1rel(gko, gke)), two(maxrel(gko, gke))) == (7.3e-13, 1.3e-12)
    assert (two(l1rel(gku, gke)), two(maxrel(gku, gke))) == (7.1e-13, 1.3e-12)
    assert (two(l1rel(gko, gku)), two(maxrel(gko, gku))) == (1.0e-13, 1.0e-13)
