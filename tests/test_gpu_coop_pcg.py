"""The cooperative single-solve kernels, `k_pcg` (Jacobi-PCG, dfe_pcg.cu) and `k_mgpcg` (multigrid-preconditioned CG,
dfe_mg_kernel.cuh), at their partition edges and at extreme right-hand-side magnitudes, against the float64 oracle.

Every un-batched 2-D solve and its adjoint take one of these two kernels.  `k_pcg` gives each CTA a contiguous block of
`per_cta = ceil(n_slices / grid)` SELL slices of 32 rows, with `grid = min(ceil(n_slices / 24), #SMs)`, and its 24 warps
walk the block two slices at a time (slices s and s + 24).  The case table reaches one CTA with a partial last slice,
exactly 24 full slices, CTAs left without a slice, warps that make two trips with an odd last pair, slices far wider than
the 4-column batches of the SpMV (a wheel mesh whose centre has 45 neighbours), 8-neighbour rows, scattered gathers and a
1-D line.  `k_mgpcg` is reached at its smallest grid, on both sides of the 512 / 768-thread switch, with the CTA size
forced both ways, on a thin hierarchy whose shared-memory tail starts at level 1, and at every smoothing depth.

Both kernels solve for the right-hand side scaled by the power of two that brings its largest entry into [1, 2), and
scale x back at the end.  So results scale exactly with powers of two, and right-hand sides whose squares underflow
(|F| < ~1e-162) or overflow (|F| > ~1e154) are solved like any other.
"""
import functools
import re

import numpy as np
import pytest
import torch

from difffe_physics_lab_b200 import _native
from diffhe.mesh import FEMesh
from diffhe.solver import DifferentiableFESolver
from tests.test_gpu_band_edges import _grid
from tests.test_gpu_batch_pcg import _launched, _line, _permuted
from tests.test_gpu_parity import TOL2D, abi_assemble, oracle_run, relerr, run

pytestmark = pytest.mark.gpu

PW = 24            # warps per CTA of k_pcg (768 threads)
MG_SMALL_N = 65536  # grids of at most this many unknowns run the 512-thread k_mgpcg
TAIL_N = 1024      # levels of at most this many unknowns are handled by CTA 0 alone


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    _native.build()


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ============================================================================================== structure mirrors
def _slices(m):
    """(n_free, SELL slice widths) of K_free from the handle's pattern."""
    rpf, _ = m._native(torch.cuda.current_device()).csr(1)
    nf = len(rpf) - 1
    rl = np.diff(rpf)
    return nf, [int(rl[32 * s:32 * s + 32].max()) for s in range(-(-nf // 32))]


def _plan(nsl, sms):
    """plan_pcg (dfe_pcg.cu) and the block split of k_pcg: (grid, per_cta, CTAs without a slice).  One CTA per SM."""
    grid = max(1, min(-(-nsl // PW), sms))
    per = -(-nsl // grid)
    return grid, per, grid - -(-nsl // per)


def _mg_levels(nx, ny):
    """mg_dims (dfe_mg.cu): interior grid sizes of every level, and the first level of the shared-memory tail."""
    my, mx = ny - 1, nx - 1
    lev = []
    while True:
        lev.append((my, mx))
        if my * mx <= 32:
            break
        assert my >= 2 and mx >= 2
        my, mx = my // 2, mx // 2
    lc = len(lev) - 1
    while lc > 1 and lev[lc - 1][0] * lev[lc - 1][1] <= TAIL_N:
        lc -= 1
    return [a * b for a, b in lev], lc


def _square_with(pred, start):
    """The smallest n >= start whose rectangle(n, n) gives a k_pcg split with pred(n_slices, grid, per_cta, empty)."""
    sms = _sms()
    for n in range(start, 4 * start):
        nsl = -(-(n - 1) ** 2 // 32)
        if pred(nsl, *_plan(nsl, sms)):
            return n
    raise AssertionError("no rectangle size fits")


def _r_empty():
    """A full grid (one CTA per SM) in which some CTAs get no slice: rectangle(340, 340) on 148 SMs."""
    return _square_with(lambda nsl, g, per, empty: g == _sms() and empty >= 1, 340)


def _r_two_trips():
    """A full grid whose warps make two trips, the second with an odd last pair (per_cta in (2 * 24, 3 * 24)):
    rectangle(500, 500) on 148 SMs."""
    return _square_with(lambda nsl, g, per, empty: g == _sms() and 2 * PW < per < 3 * PW, 500)


def _wheel(rings):
    """A polar mesh: one centre node joined to the 45 nodes of ring 1, ring k of 45 + 6 (k - 1) nodes at radius k / rings,
    neighbouring rings stitched in angular order, the outer ring Dirichlet.  Row 0 of K_free (the centre) has 46
    entries, so slice 0 is 46 columns wide; the other slices are 6 to 8 wide."""
    counts = [45 + 6 * k for k in range(rings)]
    start = np.concatenate(([1], 1 + np.cumsum(counts)))
    xy = [(0.0, 0.0)]
    for k, c in enumerate(counts):
        t = 2 * np.pi * np.arange(c) / c
        xy += list(zip((k + 1) / rings * np.cos(t), (k + 1) / rings * np.sin(t)))
    xy = np.array(xy)
    el = [(0, start[0] + i, start[0] + (i + 1) % counts[0]) for i in range(counts[0])]
    for k in range(rings - 1):
        n1, n2, a, b = counts[k], counts[k + 1], start[k], start[k + 1]
        i = j = 0
        while i < n1 or j < n2:
            if j == n2 or (i < n1 and (i + 1) / n1 <= (j + 1) / n2):
                el.append((a + i, a + (i + 1) % n1, b + j % n2))
                i += 1
            else:
                el.append((a + i % n1, b + (j + 1) % n2, b + j))
                j += 1
    el = np.array(el, dtype=np.int64)
    p = xy[el]
    cw = (p[:, 1, 0] - p[:, 0, 0]) * (p[:, 2, 1] - p[:, 0, 1]) - (p[:, 2, 0] - p[:, 0, 0]) * (p[:, 1, 1] - p[:, 0, 1]) < 0
    el[cw] = el[cw][:, [0, 2, 1]]
    outer = range(start[rings - 1], start[rings])
    bc = {int(q): 0.2 + 0.1 * xy[q, 0] for q in outer}
    return FEMesh(nodes=torch.from_numpy(xy), elements=torch.from_numpy(el), dirichlet_nodes=bc)


def _wheel_rings():
    """Enough rings that the grid is full and slice 0 (the centre's) is paired with slice 24 (190 rings on 148 SMs)."""
    sms = _sms()
    for r in range(20, 400):
        nf = 1 + sum(45 + 6 * k for k in range(r - 1))
        if _plan(-(-nf // 32), sms)[0] == sms and _plan(-(-nf // 32), sms)[1] > PW:
            return r
    raise AssertionError


# name: (mesh factory, kappa kinds compared with the oracle)
PCG_CASES = {
    "r24": (lambda: FEMesh.rectangle(24, 24), ("scalar", "elem")),
    "r25x33": (lambda: FEMesh.rectangle(25, 33, x_range=(-1.0, 0.5), bc_value=0.4), ("scalar", "elem")),
    "r34": (lambda: FEMesh.rectangle(34, 34, bc_value=0.2), ("scalar", "elem")),
    "r100": (lambda: FEMesh.rectangle(100, 100, y_range=(0.0, 2.0), bc_value=-0.3), ("elem",)),
    "r_empty": (lambda: FEMesh.rectangle(_r_empty(), _r_empty(), bc_value=0.1), ("scalar", "elem")),
    "r_two_trips": (lambda: FEMesh.rectangle(_r_two_trips(), _r_two_trips()), ("elem",)),
    "flip60x50": (lambda: _grid(60, 50, "lrbt", 0.0, 0.5, seed=7), ("scalar", "elem")),
    "perm60x50": (lambda: _permuted(60, 50, 1), ("scalar", "elem")),
    "wheel": (lambda: _wheel(_wheel_rings()), ("scalar", "elem")),
    "line": (lambda: _line(800, 5), ("scalar", "elem")),
}
MG_GRIDS = {"mg33": (33, 33), "mg257": (257, 257), "mg258x257": (258, 257), "mg256x16": (256, 16)}
MG_CASES = {
    "mg33": (lambda: FEMesh.rectangle(33, 33, bc_value=0.25), ("scalar", "elem")),
    "mg257": (lambda: FEMesh.rectangle(257, 257, x_range=(0.0, 1.5)), ("scalar", "elem")),
    "mg258x257": (lambda: FEMesh.rectangle(258, 257, bc_value=-0.1), ("scalar", "elem")),
    "mg256x16": (lambda: FEMesh.rectangle(256, 16, y_range=(0.0, 0.1), bc_value=0.3), ("scalar", "elem")),
}
CASES = {**PCG_CASES, **MG_CASES}


@functools.lru_cache(maxsize=None)
def _mesh(name):
    return CASES[name][0]()


def _inputs(m, seed):
    rng = np.random.default_rng(seed)
    f = rng.uniform(-0.5, 1.0, m.n_nodes)
    gbar = rng.standard_normal(m.n_nodes)
    kap_e = np.exp(rng.uniform(np.log(1e-2), 0.0, m.n_elements))
    return f, gbar, kap_e


def _kappa(name, kind):
    m = _mesh(name)
    return 1.3 if kind == "scalar" else _inputs(m, 1000 + sorted(CASES).index(name))[2]


@functools.lru_cache(maxsize=None)
def _oracle(name, kind):
    """u, dL/dkappa, dL/df from the oracle, once per module."""
    m = _mesh(name)
    f, gbar, _ = _inputs(m, 1000 + sorted(CASES).index(name))
    return oracle_run(m, _kappa(name, kind), f, gbar)


def _solver2d(m):
    """solver2d that puts a k_pcg case on k_pcg: "jacobi" where multigrid would be chosen."""
    return "jacobi" if _native.lib().dfe_mg_supported(m._native(torch.cuda.current_device()).handle) else "auto"


def _route(name, m):
    """(solver2d, last_solver2d) of a case: the k_mgpcg cases on multigrid, the others on k_pcg."""
    return ("mg", "mg") if name.startswith("mg") else (_solver2d(m), "jacobi")


# ===================================================================================================== the case table
def test_case_table_structure():
    """What each mesh gives the kernels: slice counts, widths and the k_pcg block split (its counts on 148 SMs), and the
    multigrid hierarchy of the k_mgpcg meshes."""
    sms = _sms()
    L = _native.lib()
    dev = torch.cuda.current_device()
    want148 = {"r24": (529, 17, 1, 17, 0), "r25x33": (768, 24, 1, 24, 0), "r34": (1089, 35, 2, 18, 0),
               "r100": (9801, 307, 13, 24, 0), "r_empty": (339 ** 2, 3592, 148, 25, 4),
               "r_two_trips": (499 ** 2, 7782, 148, 53, 1)}
    for name in PCG_CASES:
        m = _mesh(name)
        nf, widths = _slices(m)
        nsl = len(widths)
        grid, per, empty = _plan(nsl, sms)
        assert m._native(dev).info.n_free == nf and m._native(dev).info.sell_nnz == 32 * sum(widths), name
        if sms == 148 and name in want148:
            assert (nf, nsl, grid, per, empty) == want148[name], (name, nf, nsl, grid, per, empty)
        if name == "r24":
            assert grid == 1 and nf % 32 != 0                         # one CTA, partial last slice
        if name == "r25x33":
            assert grid == 1 and nf == 32 * PW                        # exactly 24 full slices
        if name == "r34":
            assert grid == 2
        if name == "r_empty":
            assert grid == sms and empty >= 1
        if name == "r_two_trips":
            assert grid == sms and 2 * PW < per < 3 * PW              # second trip: warps with no second slice
        if name == "flip60x50":
            assert max(widths) == 9                                   # 8-neighbour rows
        if name == "perm60x50":
            rpf, colf = m._native(dev).csr(1)
            assert np.abs(np.repeat(np.arange(nf), np.diff(rpf)) - colf).max() > nf // 2   # scattered gathers
        if name == "wheel":
            assert grid == sms and per > PW                           # slice 0 is paired with slice 24
            assert widths[0] == 46 and widths[0] % 4 != 0 and widths[24] != widths[0]
            assert sum(w % 4 != 0 for w in widths) > nsl // 2
        if name == "line":
            assert m._native(dev).info.chain1d == 0
        if name in ("r34", "r100", "r_empty", "r_two_trips"):               # multigrid would take these
            assert L.dfe_mg_supported(m._native(dev).handle) == 1, name
    assert L.dfe_mg_supported(_mesh("wheel")._native(dev).handle) == 0
    # levels (unknowns) and the first level of the shared-memory tail
    levels = {"mg33": ([1024, 256, 64, 16], 1), "mg257": ([65536, 16384, 4096, 1024, 256, 64, 16], 3),
              "mg258x257": ([65792, 16384, 4096, 1024, 256, 64, 16], 3), "mg256x16": ([3825, 889, 189, 31], 1)}
    for name, want in levels.items():
        m = _mesh(name)
        nx, ny = MG_GRIDS[name]
        assert m.n_nodes == (nx + 1) * (ny + 1) and L.dfe_mg_supported(m._native(dev).handle) == 1, name
        assert m._native(dev).info.n_free == want[0][0] and _mg_levels(nx, ny) == want, name
    assert levels["mg257"][0][0] == MG_SMALL_N < levels["mg258x257"][0][0]
    assert _mg_levels(256, 16)[0] == [15 * 255, 7 * 127, 3 * 63, 1 * 31]     # every dimension odd
    assert L.dfe_mg_supported(FEMesh.rectangle(33, 32)._native(dev).handle) == 0   # 992 interior nodes: declined


# ================================================================================ route, accuracy and determinism
def _mg_widths(fn):
    """The CTA sizes of the k_mgpcg instances fn() launched (namespaces mg512 / mg768 of dfe_mg.cu)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {int(w) for e in prof.events() for w in re.findall(r"mg(512|768)::k_mgpcg", e.name.replace(" ", ""))}


def _check_case(name, solver2d="auto", want="mg", **kw):
    m = _mesh(name)
    f, gbar, _ = _inputs(m, 1000 + sorted(CASES).index(name))
    worst = {}
    for kind in CASES[name][1]:
        kap = _kappa(name, kind)
        (u, gk, gf, s), names = _launched(lambda: run(m, kap, f, gbar, solver2d=solver2d, **kw))
        assert s._opts["last_solver2d"] == want, name
        kern = "k_mgpcg" if want == "mg" else "k_pcg"
        other = "k_pcg" if want == "mg" else "k_mgpcg"
        assert kern in names and other not in names, names
        assert not any(k.startswith(("k_batch", "k_band")) for k in names), names
        assert s.last_pcg[0][0] > 0 and s._opts["last_pcg_adjoint"][0][0] > 0
        uo, gko, gfo = _oracle(name, kind)
        eu, ef = relerr(u, uo), relerr(gf, gfo)
        if kind == "scalar":
            eg = abs(float(gk) - gko.sum()) / np.abs(gko).sum()
        else:
            eg = float(np.abs(gk - gko).max() / np.abs(gko).max())
        assert eu <= TOL2D and ef <= TOL2D and eg <= TOL2D, (kind, eu, ef, eg)
        worst[kind] = (eu, ef, eg)
        u2, gk2, gf2, s2 = run(m, kap, f, gbar, solver2d=solver2d, **kw)             # same bits on a repeated call
        assert np.array_equal(u, u2) and np.array_equal(gk, gk2) and np.array_equal(gf, gf2)
        assert s2.last_pcg == s.last_pcg
    print(f"\n[{name}] {want}: " + "; ".join(f"{k}: u {a:.1e} gf {b:.1e} gk {c:.1e}" for k, (a, b, c) in worst.items()))


@pytest.mark.parametrize("name", list(PCG_CASES))
def test_pcg_vs_oracle(name):
    """k_pcg through DifferentiableFESolver: the kernel that ran, u, dL/df and dL/dkappa against the oracle, same bits
    on a repeated call."""
    _check_case(name, solver2d=_solver2d(_mesh(name)), want="jacobi")


@pytest.mark.parametrize("name", list(MG_CASES))
def test_mg_vs_oracle(name):
    """k_mgpcg: the CTA size the grid selects, u, dL/df and dL/dkappa against the oracle, same bits on a repeated call."""
    m = _mesh(name)
    n0 = _mg_levels(*MG_GRIDS[name])[0][0]
    f, gbar, _ = _inputs(m, 1)
    widths = _mg_widths(lambda: DifferentiableFESolver(m, kappa=1.0)(torch.tensor(f, device="cuda")))
    assert widths == {512 if n0 <= MG_SMALL_N else 768}, widths
    _check_case(name)


def test_mg_declines_below_1024_unknowns():
    """rectangle(33, 32) (992 interior nodes) is one row short of the smallest multigrid grid: Jacobi-PCG."""
    m = FEMesh.rectangle(33, 32, bc_value=0.25)
    f, gbar, _ = _inputs(m, 5)
    (u, gk, gf, s), names = _launched(lambda: run(m, 1.3, f, gbar))
    assert s._opts["last_solver2d"] == "jacobi" and "k_pcg" in names and "k_mgpcg" not in names
    uo, gko, gfo = oracle_run(m, 1.3, f, gbar)
    assert relerr(u, uo) <= TOL2D and relerr(gf, gfo) <= TOL2D and abs(float(gk) - gko.sum()) <= TOL2D * np.abs(gko).sum()


@pytest.mark.parametrize("mt", [512, 768])
def test_mg_cta_size_forced(monkeypatch, mt):
    """DFE_MG_MT forces either CTA size on rectangle(257, 257) (65 536 unknowns, 512 threads by default); the variable is
    read on every call.  The per-CTA node ranges differ, the results agree with the oracle either way."""
    monkeypatch.setenv("DFE_MG_MT", str(mt))
    m = _mesh("mg257")
    f, gbar, _ = _inputs(m, 1)
    assert _mg_widths(lambda: DifferentiableFESolver(m, kappa=1.0)(torch.tensor(f, device="cuda"))) == {mt}
    _check_case("mg257")


def test_mg_smoothing_depth():
    """V(nu, nu) for every nu the kernel takes (1 .. 4), per-element kappa: the same answer, the same bits on a repeated
    call, and no more iterations with four sweeps than with one."""
    m = FEMesh.rectangle(96, 80, bc_value=0.15)
    f, gbar, kap = _inputs(m, 77)
    uo, gko, gfo = oracle_run(m, kap, f, gbar)
    iters = {}
    for nu in (1, 2, 3, 4):
        (u, gk, gf, s), names = _launched(lambda: run(m, kap, f, gbar, mg_nu=nu))
        assert s._opts["last_solver2d"] == "mg" and "k_mgpcg" in names and "k_pcg" not in names
        assert relerr(u, uo) <= TOL2D and relerr(gf, gfo) <= TOL2D, nu
        assert np.abs(gk - gko).max() <= TOL2D * np.abs(gko).max(), nu
        u2, gk2, gf2, s2 = run(m, kap, f, gbar, mg_nu=nu)
        assert np.array_equal(u, u2) and np.array_equal(gk, gk2) and np.array_equal(gf, gf2) and s2.last_pcg == s.last_pcg
        iters[nu] = s.last_pcg[0][0]
    assert iters[4] <= iters[1], iters
    print(f"\n[mg_nu] forward iterations {iters}")


# ========================================================================================= right-hand-side magnitudes
MAG_CASES = ["r24", "r_empty", "mg257", "mg258x257"]


@functools.lru_cache(maxsize=None)
def _mag_mesh(name, s=1.0):
    """The case's mesh with Dirichlet data 0.3 + 0.2 x (times s)."""
    m = _mesh(name)
    x = m.nodes[:, 0].numpy()
    bc = {p: (0.3 + 0.2 * float(x[p])) * s for p in m.dirichlet_nodes}
    return FEMesh(nodes=m.nodes, elements=m.elements, dirichlet_nodes=bc)


def _mag_inputs(m, seed=3):
    rng = np.random.default_rng(seed)
    return rng.uniform(0.5, 1.0, m.n_nodes), rng.uniform(0.5, 1.0, m.n_nodes)


@pytest.mark.parametrize("name", MAG_CASES)
def test_power_of_two_scaling_is_exact(name):
    """f and the Dirichlet data times 2^-1000 with gbar times 2^1000, and the other way round: u, dL/df and dL/dkappa are
    the unscaled results times the same powers of two, bit for bit, after the same number of iterations.  The unscaled
    inputs are chosen so that no entry of F, u, lambda or dL/df, nor the products that form them, leaves the normal range
    (f in [8, 16) for the first case, gbar in [512, 1024) for the second; u, lambda > 0)."""
    for fb, gb, k in ((16.0, 1.0, -1000), (1.0, 2.0 ** 10, 1000)):
        u0, gk0, gf0, it0 = _mag_run_scaled(name, fb, gb)
        u, gk, gf, it = _mag_run_scaled(name, fb * 2.0 ** k, gb * 2.0 ** -k)
        assert it == it0 and it0[0] > 0 and it0[1] > 0, (k, it, it0)
        assert np.array_equal(u, u0 * 2.0 ** k), k
        assert np.array_equal(gf, gf0 * 2.0 ** -k), k
        assert np.array_equal(gk, gk0), k
        assert np.abs(u).min() > 0 and np.abs(gf[_free(name)]).min() > 2.3e-308


def _free(name):
    return _mag_mesh(name)._native(torch.cuda.current_device()).free_nodes()


def _mag_run_scaled(name, fs, gs):
    """run() with f in [0.5, 1) times fs, the Dirichlet data times fs and gbar in [0.5, 1) times gs."""
    m = _mag_mesh(name, fs)
    f, gbar = _mag_inputs(_mag_mesh(name))
    sv, want = _route(name, m)
    u, gk, gf, s = run(m, 1.3, f * fs, gbar * gs, solver2d=sv)
    assert s._opts["last_solver2d"] == want
    return u, gk, gf, (s.last_pcg[0][0], s._opts["last_pcg_adjoint"][0][0])


@functools.lru_cache(maxsize=None)
def _mag_oracle(name):
    m = _mag_mesh(name)
    f, gbar = _mag_inputs(m)
    return oracle_run(m, 1.3, f, gbar)


@pytest.mark.parametrize("name", MAG_CASES)
@pytest.mark.parametrize("side,scale", [("f", 1e-160), ("f", 1e-155), ("f", 1e300), ("gbar", 1e-160), ("gbar", 1e300)])
def test_extreme_magnitudes(name, side, scale):
    """f (with the Dirichlet data) or gbar times a factor that takes ||F||^2 below the smallest double or above the
    largest.  u and the gradients are linear in the scaled input, so the reference is the oracle's unscaled result times
    the factor (checked against the oracle run on the scaled input for the smallest mesh)."""
    uo, gko, gfo = _mag_oracle(name)
    fs, gs = (scale, 1.0) if side == "f" else (1.0, scale)
    u, gk, gf, it = _mag_run_scaled(name, fs, gs)
    assert it[0] > 0 and it[1] > 0
    assert relerr(u, uo * fs) <= TOL2D and relerr(gf, gfo * gs) <= TOL2D
    assert abs(float(gk) - gko.sum() * fs * gs) <= TOL2D * np.abs(gko).sum() * fs * gs
    if name == "r24":
        m = _mag_mesh(name, fs)
        f, gbar = _mag_inputs(_mag_mesh(name))
        uo2, gko2, gfo2 = oracle_run(m, 1.3, f * fs, gbar * gs)
        assert relerr(uo2, uo * fs) <= 1e-13 and relerr(gfo2, gfo * gs) <= 1e-13
        assert abs(gko2.sum() - gko.sum() * fs * gs) <= 1e-13 * np.abs(gko).sum() * fs * gs


@pytest.mark.parametrize("name", MAG_CASES)
def test_huge_kappa_with_dirichlet_data(name):
    """Scalar kappa = 1e160 with Dirichlet data 0.3 + 0.2 x: the lifted load -K_fd g is ~1e160, its square overflows.
    (With constant data u would be 0.3 to within 1e-160, and dL/dkappa would be rounding noise in any arithmetic.)"""
    m = _mag_mesh(name)
    f, gbar = _mag_inputs(m, 9)
    sv, want = _route(name, m)
    u, gk, gf, s = run(m, 1e160, f, gbar, solver2d=sv)
    assert s._opts["last_solver2d"] == want
    uo, gko, gfo = oracle_run(m, 1e160, f, gbar)
    assert relerr(u, uo) <= TOL2D and relerr(gf, gfo) <= TOL2D
    assert abs(float(gk) - gko.sum()) <= TOL2D * np.abs(gko).sum()


@pytest.mark.parametrize("name", MAG_CASES)
def test_zero_and_non_finite_right_hand_sides(name):
    """f = 0 with zero Dirichlet data: u = 0 exactly after 0 iterations (and gbar = 0: zero gradients).  A NaN or an inf in
    f or in gbar: BreakdownError that names the right-hand side, not the mesh."""
    m0 = _mesh(name)
    m = FEMesh(nodes=m0.nodes, elements=m0.elements, dirichlet_nodes={p: 0.0 for p in m0.dirichlet_nodes})
    sv, want = _route(name, m)
    z = np.zeros(m.n_nodes)
    u, gk, gf, s = run(m, 1.3, z, z, solver2d=sv)
    assert s._opts["last_solver2d"] == want and not u.any() and not gf.any() and float(gk) == 0.0
    assert s.last_pcg == [(0, 0.0)] and s._opts["last_pcg_adjoint"] == [(0, 0.0)]
    f, gbar = _mag_inputs(m)
    p = int(m._native(torch.cuda.current_device()).free_nodes()[len(z) // 7 % 50])
    for bad in (float("nan"), float("inf"), -float("inf")):
        fb = f.copy()
        fb[p] = bad
        with pytest.raises(_native.BreakdownError, match="right-hand side has a non-finite entry"):
            run(m, 1.3, fb, gbar, solver2d=sv)
        gb = gbar.copy()
        gb[p] = bad
        with pytest.raises(_native.BreakdownError, match="right-hand side has a non-finite entry"):
            run(m, 1.3, f, gb, solver2d=sv)


def test_tiny_rhs_alone_and_in_a_batch():
    """A row of f and gbar at 1e-160 solved alone (k_pcg) and inside a batch (k_batch) on a mesh both routes take."""
    m = FEMesh.rectangle(34, 20)
    L = _native.lib()
    assert L.dfe_batch_supported(m._native(torch.cuda.current_device()).handle) == 1
    rng = np.random.default_rng(12)
    f, gbar = rng.uniform(-0.5, 1.0, (3, m.n_nodes)) * 1e-160, rng.standard_normal((3, m.n_nodes)) * 1e-160

    def batch():
        k = torch.tensor(0.9, dtype=torch.float64, device="cuda", requires_grad=True)
        ft = torch.tensor(f, device="cuda", requires_grad=True)
        s = DifferentiableFESolver(m, kappa=k)
        s._opts["batch_solver"] = "pcg"
        u = s(ft)
        (u * torch.tensor(gbar, device="cuda")).sum().backward()
        return u.detach().cpu().numpy(), ft.grad.cpu().numpy()

    (ub, gfb), nb = _launched(batch)
    assert any(k.startswith("k_batch") for k in nb) and "k_pcg" not in nb, nb
    (u1, gk1, gf1, s), n1 = _launched(lambda: run(m, 0.9, f[1], gbar[1]))
    assert "k_pcg" in n1 and not any(k.startswith("k_batch") for k in n1), n1
    assert relerr(u1, ub[1]) <= 1e-12 and relerr(gf1, gfb[1]) <= 1e-12
    uo, gko, gfo = oracle_run(m, 0.9, f[1], gbar[1])
    assert relerr(u1, uo) <= TOL2D and relerr(gf1, gfo) <= TOL2D and abs(float(gk1) - gko.sum()) <= TOL2D * np.abs(gko).sum()
    Ff = abi_assemble(m, 0.9, f[1])[4]
    assert np.abs(Ff).max() < 1e-162                            # ||F||^2 underflows to 0
