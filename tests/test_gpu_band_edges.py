"""The banded tensor-core solver and the heat rollout at their structural edges, against float64 references.

`k_band_solve_mma` (dfe_batch.cu) and `k_heat_roll` (dfe_heat.cu) share one block-TRSM step (`band_step`, dfe_band_mma.cuh)
on 32 x 32 blocks, and the stencil-form load / gradient kernels stage rows of f / u in shared memory (`row_to_smem`).  The
meshes below reach what a 'middle of the road' rectangle does not: one block row, no padding and 31 padding rows, the
full half bandwidth of 32 (the only case in which the diagonal of the coupling blocks S_k is non-zero), one-warp CTAs on
an odd node count with a free last node, perturbed coordinates, mixed quad diagonals (the element-form kernels), and a
random SPD matrix with diagonal scaling, whose factor blocks differ from block row to block row.
"""
import re
import zlib

import numpy as np
import pytest
import scipy.linalg as sla
import torch

from difffe_physics_lab_b200 import DifferentiableHeatSolver, _native
from diffhe.mesh import FEMesh
from diffhe.solver import DifferentiableFESolver
from tests.test_gpu_heat_adjoint import _dense_rollout, _grads
from tests.test_gpu_parity import TOL2D, oracle_run, relerr, run

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    _native.build()


# name: (nx, ny, Dirichlet sides, coordinate perturbation / h, share of flipped quad diagonals), then what the element
# table must give: (n_nodes, n_free, npad, half bandwidth of K_free in free numbering)
CASES = {
    "r2x2": ((2, 2, "lrbt", 0.0, 0.0), (9, 1, 32, 0)),                  # one unknown, 31 padding rows
    "r33x2": ((33, 2, "lrbt", 0.0, 0.0), (102, 32, 32, 1)),             # one full block row, no padding
    "r17x3": ((17, 3, "lrbt", 0.0, 0.0), (72, 32, 32, 16)),
    "r12x4": ((12, 4, "lrbt", 0.0, 0.0), (65, 33, 64, 11)),             # 31 padding rows in the last block
    "r33x3": ((33, 3, "lrbt", 0.0, 0.0), (136, 64, 64, 32)),            # half bandwidth 32: diag(S_k) != 0
    "r33x20": ((33, 20, "lrbt", 0.0, 0.0), (714, 608, 608, 32)),
    "r6x6_left": ((6, 6, "l", 0.0, 0.0), (49, 42, 64, 6)),              # one-warp CTAs, odd n_nodes, last node free
    "r8x10_lb": ((8, 10, "lb", 0.0, 0.0), (99, 80, 96, 8)),             # odd n_nodes, multi-warp CTAs
    "r12x9_perturbed": ((12, 9, "lrbt", 0.3, 0.0), (130, 88, 96, 11)),  # non-uniform geometry, stencil kernels
    "r20x14_flipped": ((20, 14, "lrbt", 0.0, 0.5), (315, 247, 256, 20)),  # 8-neighbour nodes: element-form kernels
}
NAMES = list(CASES)


def _seed(name):
    return zlib.crc32(name.encode())


def _grid(nx, ny, sides="lrbt", perturb=0.0, flip=0.0, seed=0):
    """rectangle(nx, ny) on the unit square with Dirichlet data (varying along the boundary) on the given sides, interior
    nodes moved by up to `perturb` * h, and a share `flip` of the quads split along the other diagonal."""
    rng = np.random.default_rng(seed)
    m = FEMesh.rectangle(nx, ny)
    x, y = m.nodes[:, 0].numpy().copy(), m.nodes[:, 1].numpy().copy()
    on = {"l": np.isclose(x, 0.0), "r": np.isclose(x, 1.0), "b": np.isclose(y, 0.0), "t": np.isclose(y, 1.0)}
    dmask = np.zeros(len(x), dtype=bool)
    for s in sides:
        dmask |= on[s]
    bc = {int(p): 0.15 + 0.2 * x[p] - 0.1 * y[p] for p in np.flatnonzero(dmask)}
    if perturb:
        inner = ~(on["l"] | on["r"] | on["b"] | on["t"])
        h = min(1.0 / nx, 1.0 / ny)
        x[inner] += rng.uniform(-perturb, perturb, inner.sum()) * h
        y[inner] += rng.uniform(-perturb, perturb, inner.sum()) * h
    el = m.elements.numpy().copy()
    if flip:
        q = np.flatnonzero(rng.uniform(size=nx * ny) < flip)        # quad q owns triangles 2q ([a,b,d]) and 2q+1 ([b,c,d])
        a, b, c, d = el[2 * q, 0], el[2 * q, 1], el[2 * q + 1, 1], el[2 * q, 2]
        el[2 * q] = np.stack((a, b, c), 1)
        el[2 * q + 1] = np.stack((a, c, d), 1)
    return FEMesh(nodes=torch.from_numpy(np.stack((x, y), 1)), elements=torch.from_numpy(el), dirichlet_nodes=bc)


def _mesh(name):
    return _grid(*CASES[name][0], seed=_seed(name))


def _structure(mesh):
    """(n_free, npad, half bandwidth of K_free) from the element table, free nodes numbered in ascending order."""
    el = mesh.elements.numpy()
    rank = np.full(mesh.n_nodes, -1)
    free = np.asarray(mesh.free_nodes(), dtype=np.int64)
    rank[free] = np.arange(len(free))
    w = 0
    for i in range(el.shape[1]):
        for j in range(el.shape[1]):
            ri, rj = rank[el[:, i]], rank[el[:, j]]
            both = (ri >= 0) & (rj >= 0)
            if both.any():
                w = max(w, int(np.abs(ri[both] - rj[both]).max()))
    return len(free), -(-len(free) // 32) * 32, w


def _cta(rows):
    """Threads per CTA of the stencil-form kernels for `rows` rows (npad: k_band_rhs_fwd3, n_nodes: k_band_grad3)."""
    return ((rows + 1) // 2 + 31) & ~31


def _spi(row_bytes, forced=None):
    """band_spi (dfe_batch.cu): samples per CTA barrier of a stencil-form kernel whose ring row has row_bytes bytes."""
    cap = 216 * 1024
    spi = 4 if 12 * row_bytes <= cap else 2 if 8 * row_bytes <= cap else 1
    return forced if forced in (1, 2, 4) and forced <= spi else spi


def _route(mesh, nm, per_element, need_f, forced_spi=None):
    """The load kernel of dfe_band_fwd and the gradient kernel of dfe_band_bwd for this mesh, restated from the host code
    in dfe_batch.cu (band_stencil_fits, band_reg_fits, band_spi).  A change of those predicates must be made here too."""
    I = nm.info
    n, ne = I.n_nodes, I.n_elements
    nfree, npad, _ = _structure(mesh)
    nnp = (n + 1) & ~1
    rp, col = nm.csr(0)
    rows = np.repeat(np.arange(n), np.diff(rp))
    dirichlet = np.ones(n, dtype=bool)
    dirichlet[mesh.free_nodes()] = False
    n_lift = int((~dirichlet[rows] & dirichlet[col]).sum())
    max_adj = int(np.bincount(mesh.elements.numpy().ravel(), minlength=n).max())
    stencil = (I.dim == 2 and I.max_row_nnz <= 7 and n <= 1280 and npad <= 1024
               and 6 * (2 * n + 34) * 8 <= 200 * 1024)
    reg = (I.dim == 2 and ne <= 8 * 256 and nfree <= 4 * 256 and n <= 5 * 256 and n_lift <= 8192 and max_adj <= 6)
    fwd = f"k_band_rhs_fwd3<{_spi((nnp + 2) * 8, forced_spi)}>" if stencil else "k_band_rhs_fwd"
    if not per_element and stencil:
        row = (nnp + 2 + npad) * 8
        grad = f"k_band_grad3<true,{_spi(row, forced_spi)}>" if need_f else f"k_band_grad3<false,{_spi(2 * row, forced_spi)}>"
    else:
        grad = "k_band_grad2" if reg else "k_band_grad"
    return fwd, grad


def _launched(fn):
    """Run fn() under torch.profiler; returns its result and the load / gradient kernels it launched, named as in _route."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    names = set()
    for e in prof.events():
        m = re.search(r"(k_band_(?:rhs_fwd|grad)\w*?)(?:<([^>]*)>)?(?:\(|$)", e.name.replace(" ", ""))
        if m:
            k, t = m.group(1), m.group(2)
            names.add(k + ("<" + ",".join(t.split(",")[:-1]) + ">" if t else ""))   # drop the ring depth NG
    return out, names


def _stream():
    return torch.cuda.current_stream().cuda_stream


# =============================================================================================== the case table itself
def test_case_table_structure():
    L = _native.lib()
    for name, (_, (n_nodes, n_free, npad, w)) in CASES.items():
        m = _mesh(name)
        nm = m._native(torch.cuda.current_device())
        assert (m.n_nodes, *_structure(m)) == (n_nodes, n_free, npad, w), name
        rpf, colf = nm.csr(1)                             # the handle's K_free pattern has the same half bandwidth
        assert np.abs(np.repeat(np.arange(n_free), np.diff(rpf)) - colf).max() == w, name
        assert L.dfe_band_supported(nm.handle) == 1, name
        assert L.dfe_band_npad(nm.handle) == npad, name
    m = FEMesh.rectangle(34, 3)
    assert _structure(m)[2] == 33
    nm = m._native(torch.cuda.current_device())
    assert L.dfe_band_supported(nm.handle) == 0 and L.dfe_band_npad(nm.handle) == 0
    # the structural edges the table is meant to reach
    m = _mesh("r6x6_left")
    assert _cta(64) == 32 and _cta(m.n_nodes) == 32 and m.n_nodes % 2 == 1 and m.n_nodes - 1 in m.free_nodes()
    m = _mesh("r8x10_lb")
    assert _cta(96) > 32 and _cta(m.n_nodes) > 32 and m.n_nodes % 2 == 1 and m.n_nodes - 1 in m.free_nodes()
    m = _mesh("r20x14_flipped")
    assert m._native(torch.cuda.current_device()).info.max_row_nnz > 7


def test_case_table_reaches_every_band_kernel():
    """Every load and gradient kernel of the banded route is reached by a case of this file (the routes are checked
    against the kernels actually launched in test_end_to_end_vs_oracle and test_spi_variants_same_bits)."""
    reached = set()
    for name in NAMES:
        m = _mesh(name)
        nm = m._native(torch.cuda.current_device())
        for per_element, need_f in ((False, True), (False, False), (True, True)):
            reached.update(_route(m, nm, per_element, need_f))
        if _route(m, nm, False, True)[0] != "k_band_rhs_fwd":
            for spi in (1, 2, 4):
                for need_f in (True, False):
                    reached.update(_route(m, nm, False, need_f, spi))
    want = {"k_band_rhs_fwd3<4>", "k_band_rhs_fwd3<2>", "k_band_rhs_fwd3<1>", "k_band_rhs_fwd",
            "k_band_grad2", "k_band_grad"} | {f"k_band_grad3<{gf},{s}>" for gf in ("true", "false") for s in (1, 2, 4)}
    assert want <= reached, want - reached


# =============================================================================== A. dfe_band_factor + dfe_band_solve alone
def _random_spd(nm, rng):
    """A random symmetric, strictly diagonally dominant matrix on the full pattern of K, scaled as D A D with
    D = exp(U(-3, 3)); returns (values on the pattern, dense matrix, D)."""
    n = nm.info.n_nodes
    rp, col = nm.csr(0)
    rows = np.repeat(np.arange(n), np.diff(rp))
    A = np.zeros((n, n))
    A[rows, col] = rng.uniform(-1.0, 1.0, len(rows))
    A = np.triu(A, 1)
    A = A + A.T
    A[np.arange(n), np.arange(n)] = np.abs(A).sum(1) + rng.uniform(0.5, 1.5, n)
    D = np.exp(rng.uniform(-3.0, 3.0, n))
    A = D[:, None] * A * D[None, :]
    return A[rows, col], A, D


def _matvec_ld(A, X, w):
    """Rows of X times the symmetric band matrix A (half bandwidth w), in long double."""
    n = A.shape[0]
    Al, Xl = A.astype(np.longdouble), X.astype(np.longdouble)
    Y = np.zeros_like(Xl)
    for d in range(-w, w + 1):
        lo, hi = max(0, -d), min(n, n - d)
        Y[:, lo:hi] += np.diagonal(Al, d)[None, :] * Xl[:, lo + d:hi + d]
    return Y


@pytest.mark.parametrize("name", NAMES)
def test_factor_and_block_trsm(name):
    L = _native.lib()
    rng = np.random.default_rng(_seed(name) + 1)
    m = _mesh(name)
    nm = m._native(torch.cuda.current_device())
    nf, npad, w = _structure(m)
    vals, A, D = _random_spd(nm, rng)
    free = nm.free_nodes()
    Aff, Df = A[np.ix_(free, free)], D[free]
    vt = torch.tensor(vals, device="cuda")
    factor = torch.empty(L.dfe_band_factor_bytes(nm.handle), dtype=torch.uint8, device="cuda")
    status = torch.full((1,), -1, dtype=torch.int32, device="cuda")
    _native.check(L.dfe_band_factor(nm.handle, vt.data_ptr(), factor.data_ptr(), status.data_ptr(), _stream()))
    assert int(status) == 0

    def solve(rhs):
        """rhs (B, n_free) -> the solutions; checks the padding columns and three sentinel rows after row B."""
        B = rhs.shape[0]
        buf = torch.zeros((B + 3, npad), dtype=torch.float64, device="cuda")
        buf[:B, :nf] = torch.tensor(rhs)
        buf[B:] = torch.tensor(rng.standard_normal((3, npad)))
        sentinel = buf[B:].clone()
        _native.check(L.dfe_band_solve(nm.handle, B, buf.data_ptr(), factor.data_ptr(), _stream()))
        torch.cuda.synchronize()
        assert torch.equal(buf[B:].view(torch.int64), sentinel.view(torch.int64)), "rows past B were written"
        assert bool((buf[:B, nf:].view(torch.int64) == 0).all()), "padding rows are not +0.0"
        return buf[:B, :nf].cpu().numpy()

    # identity right-hand sides: A_ff^{-1}.  Y = D X D is the inverse of the well-conditioned D^-1 A_ff D^-1, so its
    # asymmetry and residual are rounding-sized whatever the scaling (the factorisation is scaling-invariant).
    X = solve(np.eye(nf))
    Y = Df[:, None] * X * Df[None, :]
    assert np.abs(Y - Y.T).max() <= 1e-12 * np.abs(Y).max()
    E = (_matvec_ld(Aff, X, w) - np.eye(nf, dtype=np.longdouble)) * (Df[:, None] / Df[None, :])
    assert float(np.abs(E).max()) <= 1e-12

    # random right-hand sides: normwise backward error against scipy's banded Cholesky on the same system
    ab = np.zeros((w + 1, nf))
    for k in range(w + 1):
        ab[k, :nf - k] = np.diagonal(Aff, -k)
    cb = sla.cholesky_banded(ab, lower=True)
    normA = np.abs(Aff).sum(1).max()
    cond = np.linalg.cond(Aff, np.inf)
    assert cond > 1e4 or nf == 1

    def berr(x, b):
        r = np.abs(b.astype(np.longdouble) - _matvec_ld(Aff, x, w)).max(1).astype(np.float64)
        return r / (normA * np.abs(x).max(1) + np.abs(b).max(1))

    for B in (1, 15, 16, 17, 127, 128, 129, 1000):
        b = rng.standard_normal((B, nf))
        x = solve(b)
        xr = sla.cho_solve_banded((cb, True), b.T).T
        eg, er = berr(x, b), berr(xr, b)
        assert eg.max() <= max(1e-14, 4 * er.max()), B
        ferr = np.abs(x - xr).max(1) / np.abs(xr).max(1)
        assert np.all(ferr <= 4 * cond * (eg + er) + 1e-15), B


# ============================================================== B. the banded route of DifferentiableFESolver, end to end
def _check_oracle(m, kap, f, gbar, u, gk, gf):
    per_element = np.ndim(kap) > 0
    tot, mag, gsum = 0.0, 0.0, np.zeros(m.n_elements)
    for b in range(f.shape[0]):
        uo, gko, gfo = oracle_run(m, kap, f[b], gbar[b])
        assert relerr(u[b], uo) <= TOL2D, b
        if gf is not None:
            assert np.abs(gf[b] - gfo).max() <= TOL2D * np.abs(gfo).max(), b
        tot, mag, gsum = tot + gko.sum(), mag + np.abs(gko).sum(), gsum + gko
    if per_element:
        assert np.abs(gk - gsum).max() <= TOL2D * np.abs(gsum).max()
    else:
        assert abs(float(gk) - tot) <= TOL2D * mag


def _run_no_df(m, kap, f, gbar):
    """u and dL/dkappa with f.requires_grad = False (the adjoint without dL/df)."""
    k = torch.tensor(kap, dtype=torch.float64, device="cuda", requires_grad=True)
    u = DifferentiableFESolver(m, kappa=k)(torch.tensor(f, device="cuda"))
    (u * torch.tensor(gbar, device="cuda")).sum().backward()
    return u.detach(), k.grad


@pytest.mark.parametrize("name", NAMES)
def test_end_to_end_vs_oracle(name):
    rng = np.random.default_rng(_seed(name) + 2)
    m = _mesh(name)
    nm = m._native(torch.cuda.current_device())
    B = 17                                             # a full 16-sample warp of the solve and one sample of the next
    f = rng.uniform(-1.0, 1.0, (B, m.n_nodes))
    gbar = rng.standard_normal((B, m.n_nodes))
    kap_s, kap_e = 0.7, np.exp(rng.uniform(np.log(1e-2), 0.0, m.n_elements))

    def calls():
        return run(m, kap_s, f, gbar), _run_no_df(m, kap_s, f, gbar), run(m, kap_e, f, gbar)

    (scalar, no_df, elem), names = _launched(calls)
    fwd, grad_s = _route(m, nm, False, True)
    want = {fwd, grad_s, _route(m, nm, False, False)[1], _route(m, nm, True, True)[1]}
    assert names == want, (names, want)

    u, gk, gf, s = scalar
    assert s.last_pcg == [(0, 0.0)]                      # the direct route ran
    _check_oracle(m, kap_s, f, gbar, u, gk, gf)
    assert torch.equal(no_df[0].cpu(), torch.tensor(u)) and torch.equal(no_df[1].cpu(), torch.tensor(gk))
    u_e, gk_e, gf_e, _ = elem
    _check_oracle(m, kap_e, f, gbar, u_e, gk_e, gf_e)

    if name == "r8x10_lb":                                # the one-CTA-per-sample PCG route on the same problem
        k = torch.tensor(kap_s, dtype=torch.float64, device="cuda", requires_grad=True)
        ft = torch.tensor(f, device="cuda", requires_grad=True)
        sp = DifferentiableFESolver(m, kappa=k)
        sp._opts["batch_solver"] = "pcg"
        up = sp(ft)
        (up * torch.tensor(gbar, device="cuda")).sum().backward()
        assert sp.last_pcg[0][0] > 0
        assert relerr(up.detach().cpu().numpy(), u) <= 1e-11
        assert abs(float(k.grad) - float(gk)) <= 1e-10 * abs(float(gk))
        assert relerr(ft.grad.cpu().numpy(), gf) <= 1e-11


STENCIL = [n for n in NAMES if n != "r20x14_flipped"]


@pytest.mark.parametrize("name", STENCIL)
def test_spi_variants_same_bits(monkeypatch, name):
    """The stencil-form kernels with 1, 2 and 4 samples per CTA barrier, with and without dL/df: the same bits."""
    rng = np.random.default_rng(_seed(name) + 3)
    m = _mesh(name)
    nm = m._native(torch.cuda.current_device())
    B = 7
    f = rng.uniform(-1.0, 1.0, (B, m.n_nodes))
    gbar = rng.standard_normal((B, m.n_nodes))

    def calls():
        out = []
        for spi in (1, 2, 4):
            monkeypatch.setenv("DFE_BAND_SPI", str(spi))
            u, gk, gf, _ = run(m, 1.3, f, gbar)
            out.append((u, gk, gf) + tuple(t.cpu().numpy() for t in _run_no_df(m, 1.3, f, gbar)))
        monkeypatch.delenv("DFE_BAND_SPI")
        return out

    outs, names = _launched(calls)
    want = set()
    for spi in (1, 2, 4):
        want.update(_route(m, nm, False, True, spi) + _route(m, nm, False, False, spi)[1:])
    assert names == want, (names, want)
    for o in outs:
        assert np.array_equal(o[3], outs[0][0]) and np.array_equal(o[4], outs[0][1])     # without dL/df
        for a, b in zip(o[:3], outs[0][:3]):
            assert np.array_equal(a, b)
    _check_oracle(m, 1.3, f, gbar, *outs[0][:3])


# ==================================================== C. strided rows with alternating 16-byte phase through the C ABI
@pytest.mark.parametrize("name", ["r6x6_left", "r8x10_lb", "r33x3"])
def test_abi_strided_rows(name):
    """dfe_band_fwd / dfe_band_bwd on column slices of NaN-padded (B, ld) buffers with odd ld (rows alternate between the
    two 16-byte phases), against the contiguous call, bit for bit; the NaN padding of u and dL/df stays untouched."""
    L = _native.lib()
    rng = np.random.default_rng(_seed(name) + 4)
    m = _mesh(name)
    nm = m._native(torch.cuda.current_device())
    I = nm.info
    n, B, st = I.n_nodes, 6, _stream()
    ld = n + 1 if n % 2 == 0 else n + 2
    kap = torch.tensor([0.9], dtype=torch.float64, device="cuda")
    vals = torch.empty(I.nnz_full, dtype=torch.float64, device="cuda")
    F = torch.empty(n, dtype=torch.float64, device="cuda")
    f0 = torch.zeros(n, dtype=torch.float64, device="cuda")
    _native.check(L.dfe_assemble(nm.handle, kap.data_ptr(), _native.KAPPA_SCALAR, f0.data_ptr(), vals.data_ptr(), F.data_ptr(), st))
    factor = torch.empty(L.dfe_band_factor_bytes(nm.handle), dtype=torch.uint8, device="cuda")
    _native.check(L.dfe_band_factor(nm.handle, vals.data_ptr(), factor.data_ptr(), None, st))
    ws = torch.empty(L.dfe_band_workspace_bytes(nm.handle, B), dtype=torch.uint8, device="cuda")
    f = torch.tensor(rng.uniform(-1.0, 1.0, (B, n)), device="cuda")
    gbar = torch.tensor(rng.standard_normal((B, n)), device="cuda")
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

    def fwd(fv, ldf, uv, ldu):
        _native.check(L.dfe_band_fwd(nm.handle, B, fv.data_ptr(), ldf, vals.data_ptr(), factor.data_ptr(), uv.data_ptr(), ldu,
                                     ws.data_ptr(), ws.numel(), st))

    def bwd(gv, ldg, uv, ldu, mode, gfv, ldgf, gk):
        _native.check(L.dfe_band_bwd(nm.handle, B, gv.data_ptr(), ldg, uv.data_ptr(), ldu, factor.data_ptr(), mode,
                                     None if gfv is None else gfv.data_ptr(), ldgf, gk.data_ptr(), ws.data_ptr(), ws.numel(), st))

    u_ref = torch.empty((B, n), dtype=torch.float64, device="cuda")
    fwd(f, n, u_ref, n)
    refs = {}
    for mode, nk in ((_native.KAPPA_SCALAR, 1), (_native.KAPPA_PER_ELEMENT, I.n_elements)):
        gf_ref = torch.empty((B, n), dtype=torch.float64, device="cuda")
        gk_ref = torch.empty((B, nk), dtype=torch.float64, device="cuda")
        bwd(gbar, n, u_ref, n, mode, gf_ref, n, gk_ref)
        refs[mode] = (gf_ref, gk_ref)
    for a, b in ((0, 1), (1, 0)):                          # offsets of the inputs / outputs inside their buffers
        fb, fv = padded(a, f)
        ub, uv = padded(b)
        fwd(fv, ld, uv, ld)
        torch.cuda.synchronize()
        assert torch.equal(uv, u_ref) and untouched(ub, b)
        for mode, (gf_ref, gk_ref) in refs.items():
            gb, gv = padded(b, gbar)
            ub2, uv2 = padded(a, u_ref)
            gfb, gfv = padded(a)
            gk = torch.empty_like(gk_ref)
            bwd(gv, ld, uv2, ld, mode, gfv, ld, gk)
            torch.cuda.synchronize()
            assert torch.equal(gfv, gf_ref) and torch.equal(gk, gk_ref) and untouched(gfb, a), mode
            gk2 = torch.empty_like(gk_ref)
            bwd(gv, ld, uv2, ld, mode, None, n, gk2)           # without dL/df
            torch.cuda.synchronize()
            assert torch.equal(gk2, gk_ref), mode
    # a row stride below n_nodes is rejected before any launch
    with pytest.raises(ValueError):
        fwd(f, n - 1, u_ref, n)
    with pytest.raises(ValueError):
        bwd(gbar, n, u_ref, n - 1, _native.KAPPA_SCALAR, None, n, refs[_native.KAPPA_SCALAR][1])


# =========================================================================== D. the heat rollout at the same edges
@pytest.mark.parametrize("B", [1, 17])
@pytest.mark.parametrize("name", ["r2x2", "r33x2", "r12x4", "r33x3", "r6x6_left"])
def test_heat_rollout_vs_dense(name, B):
    rng = np.random.default_rng(_seed(name) + B)
    m = _mesh(name)
    dt, N, every = 2e-2, 6, 2
    kap = torch.tensor(np.exp(rng.uniform(np.log(1e-2), np.log(10.0), m.n_elements)))
    f = torch.tensor(rng.uniform(-1.0, 1.0, m.n_nodes))
    u0 = torch.tensor(rng.uniform(-1.0, 1.0, (B, m.n_nodes)))
    W = torch.tensor(rng.standard_normal((B, N // every, m.n_nodes)))
    U, gu, gk, gf = _grads(m, kap, dt, f, u0, N, every, W)
    kr, fr, ur = kap.clone().requires_grad_(True), f.clone().requires_grad_(True), u0.clone().requires_grad_(True)
    Ur = _dense_rollout(m, kr, dt, fr, ur, N, every)
    (W * Ur).sum().backward()
    Ur = Ur.detach()
    assert float((U.cpu() - Ur).abs().max()) <= 1e-12 * float(Ur.abs().max())
    assert float((gk.cpu() - kr.grad).abs().sum()) <= 1e-10 * float(kr.grad.abs().sum())
    assert float((gu.cpu() - ur.grad).abs().max()) <= 1e-10 * float(ur.grad.abs().max())
    assert float((gf.cpu() - fr.grad).abs().max()) <= 1e-10 * float(fr.grad.abs().max())


def test_heat_stepper_full_bandwidth_vs_sparse_lu():
    """HeatStepper.step (dfe_band_solve on M_L + dt K) at half bandwidth 32 with 19 block rows, against scipy's splu."""
    import scipy.sparse as sp
    import scipy.sparse.linalg as spla
    from difffe_physics_lab_b200.timestepping import HeatStepper

    rng = np.random.default_rng(33)
    m = _mesh("r33x20")
    kap = np.exp(rng.uniform(np.log(1e-2), np.log(10.0), m.n_elements))
    f = torch.tensor(rng.uniform(-1, 1, m.n_nodes))
    dt, B = 5e-3, 37
    hs = HeatStepper(m, kap, dt, f=f)
    u0 = torch.tensor(rng.uniform(-1, 1, (B, m.n_nodes)), device="cuda")
    u = hs.step(u0, 2).cpu().numpy()
    rp, col = hs.nm.csr(0)
    A = sp.csr_matrix((hs.A.cpu().numpy(), col, rp), shape=(m.n_nodes,) * 2)
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
