"""The batched banded route for per-sample conductivity (kappa (B, 1) or (B, n_el)) on 2-D meshes: dfe_band_ps_fwd / _bwd
(dfe_band_ps.cu) against the float64 oracle, the per-sample loop (assemble / eliminate / PCG per sample) and the
shared-matrix factor dfe_band_factor, bit for bit where the kernels promise it."""
import re

import numpy as np
import pytest
import torch

from difffe_physics_lab_b200 import _native
from diffhe.mesh import FEMesh
from diffhe.solver import DifferentiableFESolver
from tests.test_gpu_band_edges import CASES, _grid, _seed
from tests.test_gpu_parity import TOL2D, oracle_run, relerr

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    _native.build()


MESHES = ["r32x32", "r2x2", "r12x4", "r33x3", "r6x6_left", "r12x9_perturbed", "r20x14_flipped"]
_cache = {}


def _mesh(name):
    if name not in _cache:
        _cache[name] = _grid(32, 32, seed=1) if name == "r32x32" else _grid(*CASES[name][0], seed=_seed(name))
    return _cache[name]


def _kappa(rng, m, B, per_element):
    """per-element fields log-uniform over [1e-3, 1]; per-sample values log-uniform over [0.1, 10]"""
    if per_element:
        return np.exp(rng.uniform(np.log(1e-3), 0.0, (B, m.n_elements)))
    return np.exp(rng.uniform(np.log(0.1), np.log(10.0), (B, 1)))


def _solve(m, kap, f, gbar, need_f=True, **opts):
    """u, dL/dkappa, dL/df (None without need_f) for L = sum(gbar * u), and the solver module."""
    k = torch.tensor(kap, dtype=torch.float64, device="cuda", requires_grad=True)
    ft = torch.tensor(f, dtype=torch.float64, device="cuda", requires_grad=need_f)
    s = DifferentiableFESolver(m, kappa=k)
    s._opts.update(opts)
    u = s(ft)
    (u * torch.tensor(gbar, device="cuda")).sum().backward()
    return u.detach(), k.grad, (ft.grad if need_f else None), s


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {m.group(1) for e in prof.events() for m in [re.search(r"(k_\w+)", e.name)] if m}


def _stream():
    return torch.cuda.current_stream().cuda_stream


# ============================================================================================================ 1. route
def test_supported_predicate():
    L = _native.lib()
    dev = torch.cuda.current_device()
    for name in MESHES + ["r33x20"]:          # r33x20: 608 unknowns at the full half bandwidth of 32
        m = _mesh(name) if name != "r33x20" else FEMesh.rectangle(33, 20)
        assert L.dfe_band_ps_supported(m._native(dev).handle) == 1, name
    for m in (FEMesh.rectangle(34, 20), FEMesh.rectangle(6, 5).to_p2(), FEMesh.line(40)):   # half bandwidth 33, P2, 1-D
        assert L.dfe_band_ps_supported(m._native(dev).handle) == 0
        assert L.dfe_band_ps_factor_bytes(m._native(dev).handle, 4) == 0


def test_route_and_loop_selection():
    rng = np.random.default_rng(11)
    m = _mesh("r32x32")
    B = 3
    f = rng.uniform(-1.0, 1.0, (B, m.n_nodes))
    gbar = rng.standard_normal((B, m.n_nodes))
    kap = _kappa(rng, m, B, True)
    (u, gk, gf, s), names = _kernels(lambda: _solve(m, kap, f, gbar))
    assert {"k_bps_assemble", "k_bps_factor", "k_band_rhs_fwd", "k_bps_solve", "k_band_grad2"} <= names, names
    assert not names & {"k_pcg", "k_mgpcg", "k_batch"}, names
    assert s.last_pcg == [(0, 0.0)]
    for opts in ({"batch_min": 10 ** 9}, {"batch_solver": "pcg"}):
        (u2, gk2, gf2, s2), names2 = _kernels(lambda: _solve(m, kap, f, gbar, **opts))
        assert "k_pcg" in names2 and not any(k.startswith("k_bps") for k in names2), (opts, names2)
        assert len(s2.last_pcg) == B and s2.last_pcg[0][0] > 0
        assert relerr(u.cpu(), u2.cpu()) <= TOL2D
        assert relerr(gk.cpu(), gk2.cpu()) <= TOL2D and relerr(gf.cpu(), gf2.cpu()) <= TOL2D


# ===================================================================================================== 2. factor bits
def _ps_fwd(m, f, kap, mode, ldf=None, ldu=None, fv=None, uv=None):
    """dfe_band_ps_fwd through the ABI; returns (factors, u, status)."""
    L = _native.lib()
    nm = m._native(torch.cuda.current_device())
    B = f.shape[0]
    factors = torch.empty(L.dfe_band_ps_factor_bytes(nm.handle, B), dtype=torch.uint8, device="cuda")
    ws = torch.empty(L.dfe_band_ps_workspace_bytes(nm.handle, B), dtype=torch.uint8, device="cuda")
    status = torch.full((B,), -1, dtype=torch.int32, device="cuda")
    u = torch.empty_like(f) if uv is None else uv
    fv = f if fv is None else fv
    _native.check(L.dfe_band_ps_fwd(nm.handle, B, fv.data_ptr(), ldf or m.n_nodes, kap.data_ptr(), mode, factors.data_ptr(),
                                    u.data_ptr(), ldu or m.n_nodes, status.data_ptr(), ws.data_ptr(), ws.numel(), _stream()))
    torch.cuda.synchronize()
    return factors, u, status


@pytest.mark.parametrize("per_element", [True, False])
@pytest.mark.parametrize("name", MESHES)
def test_factor_bits_match_shared_factor(name, per_element):
    """invd / Lr of samples 0, 18 and 36 of a batch of 37 equal the first npad * 33 doubles of
    dfe_band_factor(dfe_assemble(kappa_b)), bit for bit."""
    L = _native.lib()
    rng = np.random.default_rng(_seed(name) + 21)
    m = _mesh(name)
    nm = m._native(torch.cuda.current_device())
    I = nm.info
    B, npad = 37, L.dfe_band_npad(nm.handle)
    kap = torch.tensor(_kappa(rng, m, B, per_element), device="cuda")
    f = torch.tensor(rng.uniform(-1.0, 1.0, (B, m.n_nodes)), device="cuda")
    mode = _native.KAPPA_PER_SAMPLE_ELEMENT if per_element else _native.KAPPA_PER_SAMPLE
    factors, _, status = _ps_fwd(m, f, kap, mode)
    assert int(status.abs().max()) == 0
    fd = factors.view(torch.float64)
    off, per = 12 * I.n_elements, npad * 33
    assert factors.numel() == 8 * (off + B * per)
    vals = torch.empty(I.nnz_full, dtype=torch.float64, device="cuda")
    F = torch.empty(I.n_nodes, dtype=torch.float64, device="cuda")
    ref = torch.empty(L.dfe_band_factor_bytes(nm.handle), dtype=torch.uint8, device="cuda")
    amode = _native.KAPPA_PER_ELEMENT if per_element else _native.KAPPA_SCALAR
    for b in (0, B // 2, B - 1):
        kb = kap[b].contiguous()
        _native.check(L.dfe_assemble(nm.handle, kb.data_ptr(), amode, f[b].data_ptr(), vals.data_ptr(), F.data_ptr(), _stream()))
        _native.check(L.dfe_band_factor(nm.handle, vals.data_ptr(), ref.data_ptr(), None, _stream()))
        torch.cuda.synchronize()
        got = fd[off + b * per: off + (b + 1) * per].view(torch.int64)
        want = ref.view(torch.float64)[:per].view(torch.int64)
        assert torch.equal(got, want), (b, int((got != want).sum()))


# ========================================================================================================== 3. oracle
@pytest.mark.parametrize("per_element", [True, False])
@pytest.mark.parametrize("name", MESHES)
def test_vs_oracle(name, per_element):
    rng = np.random.default_rng(_seed(name) + 22)
    m = _mesh(name)
    B = 3 if name == "r32x32" else 5
    f = rng.uniform(-1.0, 1.0, (B, m.n_nodes))
    gbar = rng.standard_normal((B, m.n_nodes))
    kap = _kappa(rng, m, B, per_element)
    u, gk, gf, s = _solve(m, kap, f, gbar)
    assert s.last_pcg == [(0, 0.0)]
    u, gk, gf = u.cpu().numpy(), gk.cpu().numpy(), gf.cpu().numpy()
    assert gk.shape == kap.shape
    for b in range(B):
        kb = kap[b] if per_element else float(kap[b, 0])
        uo, gko, gfo = oracle_run(m, kb, f[b], gbar[b])
        assert relerr(u[b], uo) <= TOL2D, b
        assert np.abs(gf[b] - gfo).max() <= TOL2D * np.abs(gfo).max(), b
        if per_element:
            assert np.abs(gk[b] - gko).max() <= TOL2D * np.abs(gko).max(), b
        else:
            assert abs(gk[b, 0] - gko.sum()) <= TOL2D * np.abs(gko).sum(), b
    # without dL/df: the same u and dL/dkappa, bit for bit
    u2, gk2, _, _ = _solve(m, kap, f, gbar, need_f=False)
    assert np.array_equal(u2.cpu().numpy(), u) and np.array_equal(gk2.cpu().numpy(), gk)


def test_forward_without_grad_keeps_no_factors():
    rng = np.random.default_rng(23)
    m = _mesh("r12x4")
    B = 4
    f = torch.tensor(rng.uniform(-1.0, 1.0, (B, m.n_nodes)), device="cuda")
    kap = torch.tensor(_kappa(rng, m, B, True), device="cuda")
    u = DifferentiableFESolver(m, kappa=kap)(f)
    assert u.grad_fn is None
    u2, _, _, _ = _solve(m, kap.cpu().numpy(), f.cpu().numpy(), np.ones((B, m.n_nodes)))
    assert torch.equal(u, u2)


# ======================================================================================================= 4. gradcheck
@pytest.mark.parametrize("per_element", [True, False])
def test_gradcheck(per_element):
    rng = np.random.default_rng(24)
    m = FEMesh.rectangle(4, 3, bc_value=0.1)
    B = 3
    f = torch.tensor(rng.uniform(-1.0, 1.0, (B, m.n_nodes)), device="cuda", requires_grad=True)
    k = torch.tensor(np.exp(rng.uniform(np.log(0.5), np.log(2.0), (B, m.n_elements if per_element else 1))),
                     device="cuda", requires_grad=True)

    def fn(f, k):
        s = DifferentiableFESolver(m, kappa=k)
        u = s(f)
        assert s.last_pcg == [(0, 0.0)]
        return u

    assert torch.autograd.gradcheck(fn, (f, k), eps=1e-6, atol=1e-8, rtol=1e-6)


# ===================================================================================== 5. independence and determinism
def test_batch_independence_and_determinism():
    rng = np.random.default_rng(25)
    m = _mesh("r32x32")
    B = 2000
    f = rng.uniform(-1.0, 1.0, (B, m.n_nodes))
    gbar = rng.standard_normal((B, m.n_nodes))
    kap = _kappa(rng, m, B, True)
    big = _solve(m, kap, f, gbar)
    again = _solve(m, kap, f, gbar)
    for a, b in zip(big[:3], again[:3]):
        assert torch.equal(a, b)
    for idx in ([0, 1234], [B - 1, 1]):         # 2000 CTAs / warps: more than are resident at once
        small = _solve(m, kap[idx], f[idx], gbar[idx])
        for a, b in zip(big[:3], small[:3]):
            assert torch.equal(a[idx], b)


@pytest.mark.parametrize("name", ["r6x6_left", "r33x3", "r32x32"])
def test_abi_strided_rows(name):
    """dfe_band_ps_fwd / _bwd on column slices of NaN-padded buffers with odd row strides give the bits of the contiguous
    call and leave the padding untouched; a stride below n_nodes and a shared-kappa mode are rejected."""
    L = _native.lib()
    rng = np.random.default_rng(_seed(name) + 26)
    m = _mesh(name)
    nm = m._native(torch.cuda.current_device())
    n, B, st = m.n_nodes, 5, _stream()
    ld = n + 1 if n % 2 == 0 else n + 2
    f = torch.tensor(rng.uniform(-1.0, 1.0, (B, n)), device="cuda")
    gbar = torch.tensor(rng.standard_normal((B, n)), device="cuda")
    kap = torch.tensor(_kappa(rng, m, B, True), device="cuda")
    mode = _native.KAPPA_PER_SAMPLE_ELEMENT
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

    ws = torch.empty(L.dfe_band_ps_workspace_bytes(nm.handle, B), dtype=torch.uint8, device="cuda")

    def bwd(factors, gv, ldg, uv, ldu, gfv, ldgf, gk, md=mode):
        _native.check(L.dfe_band_ps_bwd(nm.handle, B, gv.data_ptr(), ldg, uv.data_ptr(), ldu, factors.data_ptr(), md,
                                        None if gfv is None else gfv.data_ptr(), ldgf, gk.data_ptr(), ws.data_ptr(),
                                        ws.numel(), st))
        torch.cuda.synchronize()

    factors, u_ref, status = _ps_fwd(m, f, kap, mode)
    assert int(status.abs().max()) == 0
    gf_ref, gk_ref = torch.empty_like(f), torch.empty_like(kap)
    bwd(factors, gbar, n, u_ref, n, gf_ref, n, gk_ref)
    for a, b in ((0, 1), (1, 0)):
        fb, fv = padded(a, f)
        ub, uv = padded(b)
        factors2, _, _ = _ps_fwd(m, f, kap, mode, ldf=ld, ldu=ld, fv=fv, uv=uv)
        assert torch.equal(uv, u_ref) and untouched(ub, b)
        assert torch.equal(factors2, factors)
        gb, gv = padded(b, gbar)
        ub2, uv2 = padded(a, u_ref)
        gfb, gfv = padded(a)
        gk = torch.empty_like(gk_ref)
        bwd(factors, gv, ld, uv2, ld, gfv, ld, gk)
        assert torch.equal(gfv, gf_ref) and torch.equal(gk, gk_ref) and untouched(gfb, a)
        gk2 = torch.empty_like(gk_ref)
        bwd(factors, gv, ld, uv2, ld, None, n, gk2)
        assert torch.equal(gk2, gk_ref)
    with pytest.raises(ValueError):
        _ps_fwd(m, f, kap, mode, ldf=n - 1)
    with pytest.raises(ValueError):
        _ps_fwd(m, f, kap[:, :1].contiguous(), _native.KAPPA_SCALAR)
    with pytest.raises(ValueError):
        bwd(factors, gbar, n, u_ref, n - 1, None, n, gk_ref)
    with pytest.raises(ValueError):
        bwd(factors, gbar, n, u_ref, n, None, n, gk_ref, md=_native.KAPPA_PER_ELEMENT)


# ======================================================================================================== 6. breakdown
def test_breakdown_names_the_sample():
    rng = np.random.default_rng(27)
    m = _mesh("r12x9_perturbed")
    B = 8
    f = rng.uniform(-1.0, 1.0, (B, m.n_nodes))
    kap = _kappa(rng, m, B, False)
    bad = kap.copy()
    bad[3, 0] = -1.0
    with pytest.raises(_native.BreakdownError, match=r"sample 3\b"):
        DifferentiableFESolver(m, kappa=torch.tensor(bad, device="cuda"))(torch.tensor(f, device="cuda"))
    u, gk, gf, s = _solve(m, kap, f, np.ones((B, m.n_nodes)))
    assert s.last_pcg == [(0, 0.0)] and bool(torch.isfinite(u).all()) and bool(torch.isfinite(gk).all())
