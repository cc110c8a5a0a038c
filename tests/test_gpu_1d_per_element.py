"""The per-element-kappa 1-D kernels (``k1d_pe_pass1`` / ``k1d_fold`` / ``k1d_pe_pass2`` / ``k1d_gk_cols_sum`` in
csrc/dfe_1d_split.cu) at batch sizes where every CTA column walks several samples, as the (4096, 100000) benchmark does.

Host geometry restated (split1d_run): a sample has G = ceil(n_nodes / 2304) chunks of chg = ceil(n_nodes / G) nodes;
NG = min(max(1, 2 #SMs // G), B, 160) CTA columns run in one slab; sample s goes to column s % NG as that column's
iteration s // NG.  Iterations alternate the two row-buffer sets (it & 1) and the mbarrier parity ((it >> 1) & 1), prefetch
the next sample, and (shared field) accumulate dL/dkappa per column before k1d_gk_cols_sum adds the columns in order.

dL/dkappa_e is checked against ``oracle.grads_1d_exact`` on the kernel's own stored u: the float64 oracle differences
rounded lam and u, which at n_el = 1e5 costs as much as the 1e-12 tolerance (tests/test_oracle_exact_grad.py).
"""
import functools
import math

import numpy as np
import pytest
import torch

from difffe_physics_lab_b200 import _native
from diffhe.mesh import FEMesh
from diffhe.solver import DifferentiableFESolver
from oracle import oracle as O

pytestmark = pytest.mark.gpu

TOL = 1e-12
PCH = 2304        # nodes per chunk of the per-element kernels (PR * ST)
NG_CAP = 160      # bound of the per-column partial buffer
LAYOUTS = ["shared", "per_sample"]

# id: (n_el, bc_left, bc_right, log10 range of kappa, B or None = 5 NG + 3)
CASES = {
    "n41": (40, 0.0, 0.0, (-1, 1), None),
    "n42": (41, 0.3, -0.2, (-1, 1), None),
    "n2304": (2303, 0.3, -0.2, (-1, 1), None),       # one full chunk: the last thread owns 9 nodes
    "n2305": (2304, 0.0, 0.0, (-1, 1), None),        # G = 2
    "n2306": (2305, 0.5, 0.25, (-2, 2), None),
    "n4610": (4609, None, 1.5, (-1, 1), None),       # natural left end
    "n100002": (100001, 0.7, None, (-1, 1), 64),     # the benchmark's geometry; natural right end
}
LARGE = {"n100002"}


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    _native.build()


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.uint64), b.view(np.uint64))


def maxrel(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def l1rel(a, b):
    return float(np.abs(a - b).sum() / np.abs(b).sum())


def geometry(n_nodes, B):
    sm = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    G = -(-n_nodes // PCH)
    chg = -(-n_nodes // G)
    NG = min(max(1, 2 * sm // G), B, NG_CAP)
    return G, chg, NG


def n_iter(B, NG, col):
    return len(range(col, B, NG))


@functools.lru_cache(maxsize=None)
def case_data(case):
    n_el, bl, br, (klo, khi), B = CASES[case]
    nn = n_el + 1
    if B is None:
        B = 5 * geometry(nn, 10 ** 9)[2] + 3
    G, chg, NG = geometry(nn, B)
    assert n_iter(B, NG, NG - 1) >= 4, "every column must run at least 4 iterations"
    rng = np.random.default_rng(n_el)
    m = FEMesh.line(n_el, x_left=-0.2, x_right=1.3, bc_left=bl, bc_right=br)
    assert m._native(torch.cuda.current_device()).info.chain1d == 1
    f = rng.uniform(0, 1, (B, nn))
    gbar = rng.standard_normal((B, nn))
    kap = 10.0 ** rng.uniform(klo, khi, (B, n_el))
    return m, f, gbar, kap, (B, G, chg, NG)


def kappa_of(kap, layout):
    return kap[0] if layout == "shared" else kap


def api(m, f, kap, gbar, need_f=True, dev="cuda"):
    """u, dL/dkappa, dL/df (None without need_f) for L = sum(gbar * u) through the public API."""
    k = torch.as_tensor(kap, device=dev).requires_grad_(True)
    ft = torch.as_tensor(f, device=dev).requires_grad_(need_f)
    u = DifferentiableFESolver(m, kappa=k)(ft)
    (u * torch.as_tensor(gbar, device=dev)).sum().backward()
    return (u.detach().cpu().numpy(), k.grad.cpu().numpy(), ft.grad.cpu().numpy() if need_f else None)


@functools.lru_cache(maxsize=None)
def clean_run(case, layout):
    m, f, gbar, kap, _ = case_data(case)
    return api(m, f, kappa_of(kap, layout), gbar)


def oracle_rows(B, NG, large):
    """Samples from every pipeline position: iterations 0-3, a middle one and the last of columns 0 and NG-1, and B-1."""
    pos = []
    for col in (0, NG - 1):
        last = n_iter(B, NG, col) - 1
        its = [0, 1, 2, 3, last // 2, last]
        pos += [(col, it) for it in its]
    if large:   # about 6 oracle rows at n_el = 1e5 (~2 s each): alternate the two columns
        pos = [(0, 0), (NG - 1, 1), (0, 2), (NG - 1, 3), (0, n_iter(B, NG, 0) // 2), (NG - 1, n_iter(B, NG, NG - 1) - 1)]
    rows = {col + it * NG for col, it in pos} | {B - 1}
    return sorted(rows)


# ----------------------------------------------------------------------------------------------------------- A
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("case", list(CASES))
def test_a_pipeline_rows_vs_exact_oracle(case, layout):
    m, f, gbar, kap, (B, G, chg, NG) = case_data(case)
    u, gk, gf = clean_run(case, layout)
    nodes, el, bc = m.nodes.numpy(), m.elements.numpy(), m.dirichlet_nodes
    worst = {"u": 0.0, "gf": 0.0, "gk_l1": 0.0, "gk_max": 0.0, "gk_l1_exact_u": 0.0}
    for s in oracle_rows(B, NG, case in LARGE):
        kb = kappa_of(kap, layout) if layout == "shared" else kap[s]
        ue = O.forward_exact(nodes, el, bc, kb, f[s])
        uo = np.array([float(v) for v in ue])
        gko, gfo, _ = O.grads_1d_exact(nodes, el, bc, kb, u[s], gbar[s])     # exact gradient of the STORED u
        e = {"u": maxrel(u[s], uo), "gf": maxrel(gf[s], gfo)}
        if layout == "per_sample":
            e["gk_l1"], e["gk_max"] = l1rel(gk[s], gko), maxrel(gk[s], gko)
            gke, _, _ = O.grads_1d_exact(nodes, el, bc, kb, ue, gbar[s])      # exact gradient of the exact u
            e["gk_l1_exact_u"] = l1rel(gk[s], gke)
        for k, v in e.items():
            worst[k] = max(worst[k], v)
        where = f"sample {s} (column {s % NG}, iteration {s // NG})"
        assert e["u"] <= TOL, where
        assert e["gf"] <= TOL, where
        if layout == "per_sample":
            assert e["gk_l1"] <= TOL and e["gk_max"] <= TOL, where
    print(f"\n[A] {case} {layout} B={B} G={G} NG={NG} worst relative errors: "
          + ", ".join(f"{k} {v:.3g}" for k, v in worst.items()))


# ----------------------------------------------------------------------------------------------------------- B
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("case", list(CASES))
def test_b_rows_independent_of_batch(case, layout):
    m, f, gbar, kap, (B, G, chg, NG) = case_data(case)
    u, gk, gf = clean_run(case, layout)
    for lo in range(0, B, NG):                        # one iteration per column
        hi = min(B, lo + NG)
        k = kappa_of(kap, layout) if layout == "shared" else kap[lo:hi]
        ub, gkb, gfb = api(m, f[lo:hi], k, gbar[lo:hi])
        assert same_bits(ub, u[lo:hi]) and same_bits(gfb, gf[lo:hi]), f"rows {lo}:{hi}"
        if layout == "per_sample":
            assert same_bits(gkb, gk[lo:hi]), f"rows {lo}:{hi}"
    if layout == "shared":   # a per-sample field with equal rows computes exactly what the shared field computes
        ur, _, gfr = equal_rows_run(case)
        assert same_bits(ur, u) and same_bits(gfr, gf)


@functools.lru_cache(maxsize=None)
def equal_rows_run(case):
    m, f, gbar, kap, (B, *_) = case_data(case)
    return api(m, f, np.ascontiguousarray(np.broadcast_to(kap[0], kap.shape)), gbar)


# ----------------------------------------------------------------------------------------------------------- C
@pytest.mark.parametrize("case", list(CASES))
def test_c_shared_field_reduction_order(case):
    """Shared field: column col sums its samples col, col+NG, ... from 0.0 in iteration order; then the columns are
    added in order 0..NG-1.  The per-sample rows of the same data are the summands."""
    m, f, gbar, kap, (B, G, chg, NG) = case_data(case)
    _, gk, _ = clean_run(case, "shared")
    _, rows, _ = equal_rows_run(case)
    cols = np.zeros((NG, rows.shape[1]))
    for s in range(B):
        cols[s % NG] += rows[s]
    tot = np.zeros(rows.shape[1])
    for c in range(NG):
        tot += cols[c]
    assert same_bits(gk, tot)
    exact = np.array([math.fsum(rows[:, e]) for e in range(rows.shape[1])])
    mag = np.abs(rows).sum(axis=0)
    assert np.all(np.abs(gk - exact) <= 1e-13 * mag)


# ----------------------------------------------------------------------------------------------------------- D
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("case", ["n41", "n2305", "n4610", "n100002"])
def test_d_adjoint_without_df(case, layout):
    m, f, gbar, kap, _ = case_data(case)
    _, gk, _ = clean_run(case, layout)
    _, gk2, gf2 = api(m, f, kappa_of(kap, layout), gbar, need_f=False)
    assert gf2 is None and same_bits(gk2, gk)


# ----------------------------------------------------------------------------------------------------------- E
SENT = -12345.678


def padded(rows, ld, off, fill):
    """(B, n) rows at element offset ``off`` of a fresh buffer (256-byte aligned) with row stride ``ld``; every other
    element holds ``fill``."""
    B, n = rows.shape
    buf = torch.full((off + B * ld + 4,), fill, dtype=torch.float64, device="cuda")
    view = buf[off:off + B * ld].view(B, ld)[:, :n]
    view.copy_(torch.as_tensor(rows, device="cuda"))
    return buf, view


def rest_is(buf, view, off, fill):
    """Every element of ``buf`` outside ``view`` still equals ``fill`` bitwise."""
    mask = torch.ones(buf.numel(), dtype=torch.bool, device="cuda")
    B, n = view.shape
    idx = off + torch.arange(B, device="cuda")[:, None] * view.stride(0) + torch.arange(n, device="cuda")[None, :]
    mask[idx.reshape(-1)] = False
    rest = buf[mask].cpu().numpy()
    return same_bits(rest, np.full(rest.shape, fill))


def abi_run(m, B, f, ldf, kap, mode, u_out, ldu, gbar, ldg, gf_out, ldgf, gk_out):
    L = _native.lib()
    nm = m._native(torch.cuda.current_device())
    ws = torch.empty(L.dfe_solve1d_workspace_bytes(nm.handle, B), dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    rc = L.dfe_solve1d_fwd(nm.handle, B, f, ldf, kap, mode, -1, u_out, ldu, ws.data_ptr(), ws.numel(), st)
    assert rc == 0, L.dfe_last_error()
    rc = L.dfe_solve1d_bwd(nm.handle, B, gbar, ldg, u_out, ldu, kap, mode, -1, gf_out, ldgf, gk_out,
                           ws.data_ptr(), ws.numel(), st)
    assert rc == 0, L.dfe_last_error()
    torch.cuda.synchronize()


@pytest.mark.parametrize("off", [1, 2])            # 1: rows from an 8 mod 16 base (sup* = 0); 2: 16-byte base (sup* = 1)
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("case", ["n2306", "n4610"])
def test_e_abi_odd_offsets_and_strides(case, layout, off):
    m, f, gbar, kap, (B, G, chg, NG) = case_data(case)
    u, gk, gf = clean_run(case, layout)
    nn, n_el = f.shape[1], kap.shape[1]
    n0 = (G - 1) * chg                             # first node of the last chunk
    eA = max(n0 - 1, 0)                            # first kappa element the last chunk loads
    ecnt = n_el - eA

    def odd_end(start, length):                    # a 16-byte-aligned superset load would run one element past the row
        return (start % 2 + length) % 2 == 1

    # stride > n_nodes; where the parity allows it, one that makes sample B-1's last f / gbar / u chunk end oddly
    lds = [ld for ld in range(nn + 1, nn + 5) if odd_end(off + (B - 1) * ld + n0, nn - n0)]
    ld = lds[0] if lds else nn + 3
    if off % 2 == 0:   # aligned base: sample B-1 must take a `last` path of the superset loads (rows or kappa)
        kstart = off + eA + (0 if layout == "shared" else (B - 1) * n_el)
        assert lds or odd_end(kstart, ecnt)
    nan = float("nan")
    fb, fv = padded(f, ld, off, nan)
    gb, gv = padded(gbar, ld, off, nan)
    ub, uv = padded(np.zeros_like(f), ld, off, SENT)
    gfb, gfv = padded(np.zeros_like(f), ld, off, SENT)
    k = kappa_of(kap, layout).reshape(-1)
    kb, kv = padded(k[None, :], k.size, off, nan)
    nk = n_el if layout == "shared" else B * n_el
    gkb, gkv = padded(np.zeros((1, nk)), nk, off, SENT)
    mode = _native.KAPPA_PER_ELEMENT if layout == "shared" else _native.KAPPA_PER_SAMPLE_ELEMENT
    assert fv.data_ptr() % 16 == (8 if off == 1 else 0) and kv.data_ptr() % 16 == fv.data_ptr() % 16
    abi_run(m, B, fv.data_ptr(), ld, kv.data_ptr(), mode, uv.data_ptr(), ld, gv.data_ptr(), ld, gfv.data_ptr(), ld,
            gkv.data_ptr())
    assert same_bits(uv.cpu().numpy(), u)
    assert same_bits(gfv.cpu().numpy(), gf)
    assert same_bits(gkv.cpu().numpy().reshape(gk.shape), gk)
    for buf, view in ((ub, uv), (gfb, gfv), (gkb, gkv)):
        assert rest_is(buf, view, off, SENT), "a kernel wrote outside its rows"


# ----------------------------------------------------------------------------------------------------------- F
@pytest.mark.parametrize("layout", LAYOUTS)
def test_f_host_resident_rows(layout):
    """f, gbar and kappa on the CPU: the rows are streamed in 3 chunks, chunk j's kappa rows and dL/dkappa rows start
    at lo * n_el (odd), and a shared field's gradient is the chunk-ordered sum of 3 partials."""
    from difffe_physics_lab_b200.solver import _row_chunks
    n_el, B = 20001, 320
    nn = n_el + 1
    chunks = _row_chunks(B, nn, True)
    assert len(chunks) == 3 and any((lo * n_el) % 2 for lo, _ in chunks)
    rng = np.random.default_rng(20001)
    m = FEMesh.line(n_el, x_left=-0.2, x_right=1.3, bc_left=0.4, bc_right=-0.1)
    f = rng.uniform(0, 1, (B, nn))
    gbar = rng.standard_normal((B, nn))
    kap = kappa_of(10.0 ** rng.uniform(-1, 1, (B, n_el)), layout)
    ud, gkd, gfd = api(m, f, kap, gbar)
    k = torch.tensor(kap).requires_grad_(True)
    ft = torch.tensor(f).requires_grad_(True)
    uh = DifferentiableFESolver(m, kappa=k)(ft)
    assert uh.device.type == "cpu"
    (uh * torch.tensor(gbar)).sum().backward()
    assert same_bits(uh.detach().numpy(), ud) and same_bits(ft.grad.numpy(), gfd)
    if layout == "per_sample":
        assert same_bits(k.grad.numpy(), gkd)
    else:
        assert np.abs(k.grad.numpy() - gkd).max() <= 1e-13 * np.abs(gkd).max()


# ----------------------------------------------------------------------------------------------------------- G
@pytest.mark.parametrize("poison", ["kappa_last_of_prev", "kappa_first_of_next", "f_nan"])
@pytest.mark.parametrize("parity", ["even", "odd"])
def test_g_nonfinite_sample_stays_contained(poison, parity):
    """A sample with inf kappa or NaN data must not change the bits of any other sample (odd n_el: the kappa rows of
    consecutive samples alternate 16-byte alignment)."""
    case = "n4610"
    m, f, gbar, kap, (B, G, chg, NG) = case_data(case)
    assert kap.shape[1] % 2 == 1
    u, gk, gf = clean_run(case, "per_sample")
    s = 2 * NG + (4 if parity == "even" else 5)     # the sample whose neighbour is poisoned
    f2, kap2 = f.copy(), kap.copy()
    if poison == "kappa_last_of_prev":
        bad = s - 1
        kap2[bad, -1] = np.inf
    elif poison == "kappa_first_of_next":
        bad = s + 1
        kap2[bad, 0] = np.inf
    else:
        bad = s
        f2[bad, f.shape[1] // 2] = np.nan
    u2, gk2, gf2 = api(m, f2, kap2, gbar)
    keep = np.arange(B) != bad
    for name, a, b in (("u", u2, u), ("dL/df", gf2, gf), ("dL/dkappa", gk2, gk)):
        diff = [int(r) for r in np.nonzero(keep)[0] if not same_bits(a[r], b[r])]
        assert not diff, f"{name}: samples {diff[:8]} changed (poisoned sample {bad})"
