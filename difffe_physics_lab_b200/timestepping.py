"""Backward-Euler time stepping of the heat equation with ONE banded factorisation reused by every step.

A caller of the accelerated path from the reference's roadmap (README.md:139-143: "time-dependent heat equation"; SURVEY §8f
N4) — nothing of this exists upstream, so there is no parity burden beyond the operators it is built from:

    M_L du/dt + K(kappa) u = F(f),        (M_L + dt K) u^{n+1} = M_L u^n + dt F

with K and F exactly what ``DifferentiableFESolver`` assembles (``dfe_assemble``: reference solver.py:112-145, bit for bit) and
M_L the lumped mass matrix — the load vector of f = 1 (solver.py:143-145).  ``dfe_band_factor`` factors ``M_L + dt K`` once
(any SPD matrix on the pattern of K is accepted), ``dfe_band_solve`` applies the two triangular solves to a whole batch of
states per step (block TRSM on the FP64 tensor cores).  Meshes: half bandwidth of K_free <= 32 (``rectangle(nx, ny)``, nx <= 32).

``DifferentiableHeatSolver`` runs the same scheme as a differentiable rollout: the whole time loop is one kernel launch
(``dfe_heat_fwd``), and the backward is the discrete adjoint in time (``dfe_heat_adj``, ``dfe_heat_grad``) with optional
checkpointing.  Gradients flow to ``u0``, ``kappa`` and ``f``.  With one conductivity per sample (kappa ``(B, 1)`` or
``(B, n_el)``) every sample has its own factor and the rollout runs one warp per sample (``dfe_heat_ps_*``).  A source per
sample (``f (B, n)``) or per step (``source``) enters through per-step constants formed by ``dfe_heat_src_load`` and read by
the ``*_fwd_src`` rollouts; its gradient is ``dfe_heat_src_grad`` on the adjoint's lambda rows.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch
from torch import nn

from . import _native
from .mesh import FEMesh
from .solver import _timed


class _HeatOperator:
    """``A = M_L + dt K(kappa)`` on the pattern of K, its banded factor, and the constants of one implicit step in free
    numbering: the lumped mass ``mass_free`` and ``rhs_const = dt F_free - (A g)_free`` (the lifting of the Dirichlet values
    ``g``).  ``status`` (device int32) is 0 when the factorisation succeeded; it is not read here."""

    def __init__(self, mesh: FEMesh, kappa, dt: float, f, dev: torch.device):
        L = _native.lib()
        self.nm = nm = mesh._native(dev.index)
        I = nm.info
        kap = torch.as_tensor(kappa, dtype=torch.float64, device=dev).reshape(-1).contiguous()
        mode = _native.KAPPA_SCALAR if kap.numel() == 1 else _native.KAPPA_PER_ELEMENT
        st = torch.cuda.current_stream(dev).cuda_stream
        ones = torch.ones(I.n_nodes, dtype=torch.float64, device=dev)
        vals = torch.empty(I.nnz_full, dtype=torch.float64, device=dev)
        mass = torch.empty(I.n_nodes, dtype=torch.float64, device=dev)
        _native.check(L.dfe_assemble(nm.handle, kap.data_ptr(), mode, ones.data_ptr(), vals.data_ptr(), mass.data_ptr(), st))
        self.load = torch.zeros(I.n_nodes, dtype=torch.float64, device=dev)
        if f is not None:                                   # F(f): the reference's load vector of the source term
            fs = f.to(device=dev, dtype=torch.float64).contiguous()
            scratch = torch.empty_like(vals)
            _native.check(L.dfe_assemble(nm.handle, kap.data_ptr(), mode, fs.data_ptr(), scratch.data_ptr(), self.load.data_ptr(), st))
        rp, col = nm.csr(0)
        rows = np.repeat(np.arange(I.n_nodes), np.diff(rp))
        diag = torch.as_tensor(np.nonzero(col == rows)[0], device=dev)
        self.A = float(dt) * vals                           # M_L + dt K on the pattern of K
        self.A[diag] += mass
        self.K_vals, self.mass = vals, mass
        self.factor = torch.empty(L.dfe_band_factor_bytes(nm.handle), dtype=torch.uint8, device=dev)
        self.status = torch.zeros(1, dtype=torch.int32, device=dev)
        _native.check(L.dfe_band_factor(nm.handle, self.A.data_ptr(), self.factor.data_ptr(), self.status.data_ptr(), st))
        self.free = torch.as_tensor(np.asarray(mesh.free_nodes(), dtype=np.int64), device=dev)
        self.npad = int(L.dfe_band_npad(nm.handle))
        # Dirichlet columns of (M_L + dt K) times the boundary values: the lifting of the implicit step, per free row
        bc = mesh.dirichlet_nodes
        g = torch.zeros(I.n_nodes, dtype=torch.float64, device=dev)
        if bc:
            g[torch.as_tensor(list(bc.keys()), device=dev)] = torch.as_tensor(list(bc.values()), dtype=torch.float64, device=dev)
        self.g = g
        crow = torch.as_tensor(rows, device=dev)
        ccol = torch.as_tensor(col, device=dev)
        lift = torch.zeros(I.n_nodes, dtype=torch.float64, device=dev)
        lift.index_add_(0, crow, self.A * g[ccol])          # (A g)_p; only Dirichlet columns contribute (g = 0 elsewhere)
        self.rhs_const = (float(dt) * self.load - lift)[self.free]
        self.mass_free = mass[self.free]


class HeatStepper:
    """``step(u)`` advances a batch of states ``u`` (B, n_nodes) by ``dt``; Dirichlet nodes keep their boundary values."""

    def __init__(self, mesh: FEMesh, kappa, dt: float, f: torch.Tensor | None = None, device=None):
        if not torch.cuda.is_available():
            raise RuntimeError("HeatStepper runs on CUDA only (difffe_physics_lab_b200 has no CPU fallback)")
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.mesh, self.dt, self.dev = mesh, float(dt), dev
        L = _native.lib()
        nm = mesh._native(dev.index)
        if not L.dfe_band_supported(nm.handle):
            raise NotImplementedError("HeatStepper needs a mesh whose K_free has half bandwidth <= 32 (dfe_band_supported)")
        op = _HeatOperator(mesh, kappa, self.dt, f, dev)
        if int(op.status) != 0:
            raise _native.BreakdownError(_native.ERR_BREAKDOWN, "M_L + dt K is not positive definite")
        self.nm, self.load, self.A, self.K_vals, self.mass = op.nm, op.load, op.A, op.K_vals, op.mass
        self.factor, self.free, self.npad, self.g = op.factor, op.free, op.npad, op.g
        self.rhs_const, self.mass_free = op.rhs_const, op.mass_free
        self._X = None

    def step(self, u: torch.Tensor, n_steps: int = 1) -> torch.Tensor:
        """u (B, n_nodes) float64 on the stepper's device -> the states after ``n_steps`` steps (new tensor)."""
        L = _native.lib()
        B = u.shape[0]
        nf = self.free.numel()
        if self._X is None or self._X.shape[0] != B:
            self._X = torch.zeros((B, self.npad), dtype=torch.float64, device=self.dev)
        X = self._X
        X[:, :nf] = u[:, self.free]
        st = torch.cuda.current_stream(self.dev).cuda_stream
        for _ in range(n_steps):
            X[:, :nf].mul_(self.mass_free).add_(self.rhs_const)                 # M_L u^n + dt F - lifting
            _native.check(L.dfe_band_solve(self.nm.handle, B, X.data_ptr(), self.factor.data_ptr(), st))
        out = self.g.expand(B, -1).clone()
        out[:, self.free] = X[:, :nf]
        return out


def _heat_check_mesh(mesh: FEMesh, dev: torch.device, per_sample: bool = False):
    """NotImplementedError (with the reason) for meshes the differentiable rollout does not take; returns the native mesh.
    ``per_sample``: the per-sample-kappa route, whose gradient kernel has no shared-memory bound (dfe_band_ps_supported)."""
    if mesh.dim != 2:
        raise NotImplementedError("DifferentiableHeatSolver supports 2-D meshes only (1-D meshes are not implemented)")
    if mesh.order != 1:
        raise NotImplementedError("DifferentiableHeatSolver supports P1 meshes only (P2 is not implemented)")
    L = _native.lib()
    nm = mesh._native(dev.index)
    if not L.dfe_band_supported(nm.handle):
        raise NotImplementedError("DifferentiableHeatSolver needs a mesh whose K_free has half bandwidth <= 32 "
                                  "(dfe_band_supported; e.g. rectangle(nx, ny) with nx <= 32)")
    if not per_sample and not L.dfe_heat_supported(nm.handle):
        raise NotImplementedError("mesh too large for the trajectory gradient kernel: the per-element sums and three "
                                  "(u, lambda) rows must fit 200 KB of shared memory (dfe_heat_supported)")
    return nm


def _per_sample_kappa(kappa, n_el: int) -> bool:
    """True for the 2-D kappa forms that give every sample its own conductivity.  (1, 1), (1, n_el) and (n_el, 1) keep the
    shared meaning they had before per-sample kappa existed (the values are flattened)."""
    return torch.is_tensor(kappa) and kappa.dim() == 2 and kappa.shape[0] > 1 and tuple(kappa.shape) != (n_el, 1)


def _check_status(status: torch.Tensor, fault: torch.Tensor, who: str) -> None:
    """The one synchronisation of a call: the factorisation status and the fault word of the rollout kernels."""
    st = torch.cat([status, fault]).cpu()
    if int(st[0]) != 0:
        raise _native.BreakdownError(_native.ERR_BREAKDOWN, f"{who}: M_L + dt K is not positive definite (kappa <= 0?)")
    if int(st[1]) != 0:
        raise _native.DfeError(_native.ERR_CUDA, f"{who}: a bounded wait inside a rollout kernel expired; outputs invalid")


def _src_load(rt, n_steps, nb, q, ldq_t, ldq_b, base, ldbase, out=None):
    """c (n_steps, nb, npad): row (j, b) = fl(base_b + fl(dt F_free(q_{j,b}))), q_{j,b} at q + j ldq_t + b ldq_b"""
    if out is None:
        out = torch.empty((n_steps, nb, rt.npad), dtype=torch.float64, device=rt.dev)
    st = torch.cuda.current_stream(rt.dev).cuda_stream
    with _timed("heat_src_load", rt.dev):
        _native.check(_native.lib().dfe_heat_src_load(rt.h, n_steps, nb, rt.dt, q.data_ptr(), ldq_t, ldq_b, base.data_ptr(),
                                                       ldbase, out.data_ptr(), rt.sws.data_ptr(), rt.sws.numel(), st))
    return out


def _src_grad(rt, n_steps, nb, lam, ldl_t, ldl_b, g, ldg_t, ldg_b):
    """g row (j, b) at g + j ldg_t + b ldg_b = W^T (dt lam~_{j,b}), lam_{j,b} (free layout) at lam + j ldl_t + b ldl_b"""
    st = torch.cuda.current_stream(rt.dev).cuda_stream
    with _timed("heat_src_grad", rt.dev):
        _native.check(_native.lib().dfe_heat_src_grad(rt.h, n_steps, nb, rt.dt, lam.data_ptr(), ldl_t, ldl_b, g.data_ptr(),
                                                      ldg_t, ldg_b, rt.sws.data_ptr(), rt.sws.numel(), st))


def _src_ws(h, dev):
    return torch.empty(max(int(_native.lib().dfe_heat_src_workspace_bytes(h)), 16), dtype=torch.uint8, device=dev)


class _SharedRoute:
    """kappa shared by the batch: one factor of A = M_L + dt K(kappa), the tensor-core rollout kernels (dfe_heat_*).
    With ``f (B, n)`` each sample's constant c_b (B, npad) is formed once from the lifting-only constant and read by
    ``dfe_heat_fwd_src`` with a time stride of 0."""

    def __init__(self, mesh, kappa, dt, f, dev, B, warps):
        per_f = f is not None and f.dim() == 2
        self.op = op = _HeatOperator(mesh, kappa, dt, None if per_f else f, dev)
        self.h, self.npad, self.free, self.mass_free = op.nm.handle, op.npad, op.free, op.mass_free
        self.dt, self.warps, self.dev, self.B = dt, warps, dev, B
        nf = op.free.numel()
        self.mf = torch.zeros(self.npad, dtype=torch.float64, device=dev)
        self.cf = torch.zeros(self.npad, dtype=torch.float64, device=dev)
        self.mf[:nf], self.cf[:nf] = op.mass_free, op.rhs_const
        self.fault = torch.zeros(1, dtype=torch.int32, device=dev)
        self.cB = None
        if per_f:                                           # c_b = fl(fl(dt F_free(f_b)) - lift)
            self.sws = _src_ws(self.h, dev)
            self.cB = _src_load(self, 1, B, f, 0, f.stride(0), self.cf, 0)[0]
        # the constant a per-step source adds to: per sample (B, npad) or shared (npad,), with its row stride
        self.base, self.ldbase = (self.cf, 0) if self.cB is None else (self.cB, self.npad)

    def check(self, who):
        _check_status(self.op.status, self.fault, who)

    def fwd(self, src, X, traj, steps, c=None):
        """c: None, or (tensor, ldc_t, ldc_b): step j of sample b reads its constant at c + j ldc_t + b ldc_b"""
        st = torch.cuda.current_stream(self.dev).cuda_stream
        if c is None and self.cB is not None:
            c = (self.cB, 0, self.npad)
        with _timed("heat_fwd", self.dev):
            if c is None:
                _native.check(_native.lib().dfe_heat_fwd(
                    self.h, self.B, steps, None if src is None else src.data_ptr(), traj.shape[-1],
                    self.op.factor.data_ptr(), self.mf.data_ptr(), self.cf.data_ptr(), X.data_ptr(), traj.data_ptr(),
                    traj.stride(0), traj.stride(1), self.warps, self.fault.data_ptr(), st))
            else:
                _native.check(_native.lib().dfe_heat_fwd_src(
                    self.h, self.B, steps, None if src is None else src.data_ptr(), traj.shape[-1],
                    self.op.factor.data_ptr(), self.mf.data_ptr(), c[0].data_ptr(), c[1], c[2], X.data_ptr(),
                    traj.data_ptr(), traj.stride(0), traj.stride(1), self.warps, self.fault.data_ptr(), st))

    def begin_backward(self, N):
        self.N = N
        self.fault = torch.zeros(1, dtype=torch.int32, device=self.dev)
        self.gws = torch.empty(max(int(_native.lib().dfe_heat_grad_bytes(self.h, self.B, N)), 16), dtype=torch.uint8,
                               device=self.dev)

    def adj(self, n0, ln, gout, every, Xa, lam, lsum):
        st = torch.cuda.current_stream(self.dev).cuda_stream
        with _timed("heat_adj", self.dev):
            _native.check(_native.lib().dfe_heat_adj(
                self.h, self.B, n0, ln, gout.data_ptr(), gout.stride(0), gout.stride(1), every, self.op.factor.data_ptr(),
                self.mf.data_ptr(), Xa.data_ptr(), lam.data_ptr(), lsum.data_ptr(), self.warps, self.fault.data_ptr(), st))

    def grad(self, n0, ln, traj, lam):
        st = torch.cuda.current_stream(self.dev).cuda_stream
        with _timed("heat_grad", self.dev):
            _native.check(_native.lib().dfe_heat_grad(self.h, self.B, n0, ln, self.N, traj.data_ptr(), traj.stride(0),
                                                      traj.stride(1), lam.data_ptr(), self.gws.data_ptr(), self.gws.numel(), st))

    def gkappa(self, kappa):
        st = torch.cuda.current_stream(self.dev).cuda_stream
        gk = torch.empty(kappa.numel(), dtype=torch.float64, device=self.dev)
        mode = _native.KAPPA_SCALAR if kappa.numel() == 1 else _native.KAPPA_PER_ELEMENT
        with _timed("heat_grad", self.dev):
            _native.check(_native.lib().dfe_heat_grad_sum(self.h, self.B, self.N, self.dt, mode, gk.data_ptr(),
                                                          self.gws.data_ptr(), self.gws.numel(), st))
        return gk

    def finish_backward(self, who):
        _check_status(torch.zeros(1, dtype=torch.int32, device=self.dev), self.fault, who)


class _PerSampleRoute:
    """kappa (B, 1) or (B, n_el): one A_b = M_L + dt K(kappa_b) and one banded factor per sample (dfe_heat_ps_*), one
    warp per sample in the rollout kernels.  The factors take npad * 33 doubles per sample."""

    def __init__(self, mesh, kappa, dt, f, dev, B):
        L = _native.lib()
        nm = mesh._native(dev.index)
        I = nm.info
        self.h, self.npad, self.dt, self.dev, self.B = nm.handle, int(L.dfe_band_npad(nm.handle)), dt, dev, B
        self.n_el = I.n_elements
        self.mode = _native.KAPPA_PER_SAMPLE if kappa.shape[1] == 1 else _native.KAPPA_PER_SAMPLE_ELEMENT
        st = torch.cuda.current_stream(dev).cuda_stream
        one = torch.ones(1, dtype=torch.float64, device=dev)
        vals = torch.empty(max(I.nnz_full, 1), dtype=torch.float64, device=dev)
        mass = torch.empty(I.n_nodes, dtype=torch.float64, device=dev)   # M_L and F do not depend on kappa
        _native.check(L.dfe_assemble(nm.handle, one.data_ptr(), _native.KAPPA_SCALAR,
                                     torch.ones(I.n_nodes, dtype=torch.float64, device=dev).data_ptr(), vals.data_ptr(),
                                     mass.data_ptr(), st))
        load = None
        per_f = f is not None and f.dim() == 2
        if f is not None and not per_f:
            load = torch.empty(I.n_nodes, dtype=torch.float64, device=dev)
            fs = f.to(device=dev, dtype=torch.float64).contiguous()
            _native.check(L.dfe_assemble(nm.handle, one.data_ptr(), _native.KAPPA_SCALAR, fs.data_ptr(), vals.data_ptr(),
                                         load.data_ptr(), st))
        self.free = torch.as_tensor(np.asarray(mesh.free_nodes(), dtype=np.int64), device=dev)
        self.mass_free = mass[self.free]
        self.mf = torch.zeros(self.npad, dtype=torch.float64, device=dev)
        self.mf[:self.free.numel()] = self.mass_free
        self.factors = torch.empty(max(int(L.dfe_heat_ps_factor_bytes(nm.handle, B)), 16), dtype=torch.uint8, device=dev)
        self.cf = torch.empty((B, self.npad), dtype=torch.float64, device=dev)
        self.status = torch.empty(B, dtype=torch.int32, device=dev)
        ws = torch.empty(max(int(L.dfe_heat_ps_workspace_bytes(nm.handle, B)), 16), dtype=torch.uint8, device=dev)
        with _timed("heat_ps_setup", dev):
            _native.check(L.dfe_heat_ps_setup(nm.handle, B, kappa.data_ptr(), self.mode, dt, mass.data_ptr(),
                                              None if load is None else load.data_ptr(), self.factors.data_ptr(),
                                              self.cf.data_ptr(), self.status.data_ptr(), ws.data_ptr(), ws.numel(), st))
        if per_f:                                           # c_b += fl(dt F_free(f_b)), in place
            self.sws = _src_ws(self.h, dev)
            _src_load(self, 1, B, f, 0, f.stride(0), self.cf, self.npad, out=self.cf)
        self.base, self.ldbase = self.cf, self.npad

    def check(self, who):
        bad = self.status.cpu().nonzero()                   # the one synchronisation of a forward call
        if bad.numel():
            raise _native.BreakdownError(_native.ERR_BREAKDOWN, f"{who}: sample {int(bad[0, 0])}: M_L + dt K(kappa_b) is "
                                         "not positive definite (kappa_b <= 0?)")

    def fwd(self, src, X, traj, steps, c=None):
        """c: None, or (tensor, ldc_t, ldc_b): step j of sample b reads its constant at c + j ldc_t + b ldc_b"""
        st = torch.cuda.current_stream(self.dev).cuda_stream
        with _timed("heat_ps_fwd", self.dev):
            if c is None:
                _native.check(_native.lib().dfe_heat_ps_fwd(
                    self.h, self.B, steps, None if src is None else src.data_ptr(), traj.shape[-1],
                    self.factors.data_ptr(), self.mf.data_ptr(), self.cf.data_ptr(), X.data_ptr(), traj.data_ptr(),
                    traj.stride(0), traj.stride(1), st))
            else:
                _native.check(_native.lib().dfe_heat_ps_fwd_src(
                    self.h, self.B, steps, None if src is None else src.data_ptr(), traj.shape[-1],
                    self.factors.data_ptr(), self.mf.data_ptr(), c[0].data_ptr(), c[1], c[2], X.data_ptr(),
                    traj.data_ptr(), traj.stride(0), traj.stride(1), st))

    def begin_backward(self, N):
        self.gacc = torch.zeros((self.B, self.n_el), dtype=torch.float64, device=self.dev)   # running sums, zeroed

    def adj(self, n0, ln, gout, every, Xa, lam, lsum):
        st = torch.cuda.current_stream(self.dev).cuda_stream
        with _timed("heat_ps_adj", self.dev):
            _native.check(_native.lib().dfe_heat_ps_adj(
                self.h, self.B, n0, ln, gout.data_ptr(), gout.stride(0), gout.stride(1), every, self.factors.data_ptr(),
                self.mf.data_ptr(), Xa.data_ptr(), lam.data_ptr(), lsum.data_ptr(), st))

    def grad(self, n0, ln, traj, lam):
        st = torch.cuda.current_stream(self.dev).cuda_stream
        with _timed("heat_ps_grad", self.dev):
            _native.check(_native.lib().dfe_heat_ps_grad(self.h, self.B, ln, self.factors.data_ptr(), traj.data_ptr(),
                                                         traj.stride(0), traj.stride(1), lam.data_ptr(),
                                                         self.gacc.data_ptr(), st))

    def gkappa(self, kappa):
        st = torch.cuda.current_stream(self.dev).cuda_stream
        gk = torch.empty(kappa.shape[0] if self.mode == _native.KAPPA_PER_SAMPLE else kappa.shape, dtype=torch.float64,
                         device=self.dev)
        with _timed("heat_ps_grad_sum", self.dev):
            _native.check(_native.lib().dfe_heat_ps_grad_sum(self.h, self.B, self.dt, self.mode, self.gacc.data_ptr(),
                                                             gk.data_ptr(), st))
        return gk

    def finish_backward(self, who):
        pass                                                # no waits inside the per-sample kernels: nothing to check


class _Source:
    """A per-step source ``q``: ``(N, n)`` shared by the batch or ``(B, N, n)``.  Step n uses ``f + q[n]``: the constant of
    a launch of steps s .. s + l - 1 is c (l, nb, npad) = fl(base_b + fl(dt F_free(q_{s+j,b}))) on the route's constant
    without it (nb = 1 when both the source and that constant are shared by the batch)."""

    def __init__(self, rt, q):
        self.rt, self.q = rt, q
        self.shared = q.dim() == 2
        self.nb = 1 if self.shared and rt.ldbase == 0 else rt.B
        if not hasattr(rt, "sws"):
            rt.sws = _src_ws(rt.h, rt.dev)

    def consts(self, s, l):
        """(c, ldc_t, ldc_b) of the launch of steps s .. s + l - 1"""
        rt, q, nb = self.rt, self.q, self.nb
        qs = q[s] if self.shared else q[:, s]
        c = _src_load(rt, l, nb, qs, q.stride(-2), 0 if self.shared else q.stride(0), rt.base, rt.ldbase)
        return c, nb * rt.npad, rt.npad if nb > 1 else 0

    def grad(self, g, s, l, lam):
        """dL/dq at steps s .. s + l - 1 into g from lam (l, B, npad), whose slot j holds lambda_{s+1+j}: W^T (dt lam~), the
        batch summed first (in torch's fixed order) for a shared source"""
        rt, n = self.rt, self.q.shape[-1]
        if self.shared:
            ls = lam[:l].sum(1)
            _src_grad(rt, l, 1, ls, rt.npad, 0, g[s], n, 0)
        else:
            _src_grad(rt, l, rt.B, lam, rt.B * rt.npad, rt.npad, g[:, s], n, g.stride(0))


def _roll(rt, src, steps_per_launch, X, u0, traj, s, steps):
    """steps s .. s + steps - 1 into traj[:, :steps], from u0 or (u0 None) from the carry X.  With a source the steps are
    split into launches of at most ``steps_per_launch``: X carries the state across them exactly as across checkpoint
    segments, so the split changes no bit."""
    if src is None:
        rt.fwd(u0, X, traj, steps)
        return
    for j in range(0, steps, steps_per_launch):
        ln = min(steps_per_launch, steps - j)
        rt.fwd(u0 if j == 0 else None, X, traj[:, j:], ln, src.consts(s + j, ln))


class _HeatRollout(torch.autograd.Function):
    """(u0 (B, n), kappa, f (n,), (B, n) or None, source (N, n), (B, N, n) or None) -> the states after steps every,
    2 every, ..., N: (B, N / every, n).  kappa is (1,) or (n_el,) (shared by the batch) or, with ``per_sample``, (B, 1) or
    (B, n_el).

    All tensors are float64 and contiguous on the solver's device."""

    @staticmethod
    def forward(ctx, u0, kappa, f, source, solver, n_steps: int, every: int, per_sample: bool = False):
        dev, mesh, dt, c = u0.device, solver.mesh, solver.dt, solver.checkpoint
        B, n, N = u0.shape[0], mesh.n_nodes, n_steps
        fd = None if f is None else f.detach()
        rt = _PerSampleRoute(mesh, kappa.detach(), dt, fd, dev, B) if per_sample \
            else _SharedRoute(mesh, kappa.detach(), dt, fd, dev, B, solver._cta_warps)
        src = None if source is None else _Source(rt, source.detach())
        X = torch.zeros((B, rt.npad), dtype=torch.float64, device=dev)

        def roll(u_start, traj, s, steps):
            _roll(rt, src, solver._src_steps, X, u_start, traj, s, steps)

        if c is None:                                       # every state kept: the trajectory is the saved state
            traj = torch.empty((B, N, n), dtype=torch.float64, device=dev)
            roll(u0, traj, 0, N)
            out = traj if every == 1 else traj[:, every - 1::every].contiguous()
            saved = traj
        else:                                               # segments of c steps; only their first states are kept
            seg = torch.empty((B, min(c, N), n), dtype=torch.float64, device=dev)
            out = torch.empty((B, N // every, n), dtype=torch.float64, device=dev)
            starts = [u0]
            for s in range(0, N, c):
                ln = min(c, N - s)
                roll(u0 if s == 0 else None, seg, s, ln)    # later segments continue from the carry X
                first = (s // every + 1) * every            # first recorded step after s
                if first <= s + ln:
                    out[:, first // every - 1:(s + ln) // every] = seg[:, first - s - 1:ln:every]
                if s + ln < N:
                    starts.append(seg[:, ln - 1].clone())
            saved = torch.stack(starts)
        rt.check("DifferentiableHeatSolver")
        ctx.rt, ctx.src, ctx.solver, ctx.N, ctx.every = rt, src, solver, N, every
        ctx.need_f = f is not None
        ctx.per_f = f is not None and f.dim() == 2
        ctx.save_for_backward(saved, kappa)
        return out

    @staticmethod
    def backward(ctx, gout):
        L = _native.lib()
        saved, kappa = ctx.saved_tensors
        rt, src, solver, N, every = ctx.rt, ctx.src, ctx.solver, ctx.N, ctx.every
        mesh, dt, c = solver.mesh, solver.dt, solver.checkpoint
        dev = saved.device
        h, npad, nf, n = rt.h, rt.npad, rt.free.numel(), mesh.n_nodes
        B = saved.shape[0] if c is None else saved.shape[1]
        st = torch.cuda.current_stream(dev).cuda_stream
        gout = gout.to(dtype=torch.float64).contiguous()
        Xa = torch.zeros((B, npad), dtype=torch.float64, device=dev)       # lambda_{n+1}, zero above step N
        lsum = torch.zeros((B, npad), dtype=torch.float64, device=dev)
        rt.begin_backward(N)

        gsrc = None if src is None or not ctx.needs_input_grad[3] else \
            torch.empty(src.q.shape, dtype=torch.float64, device=dev)

        def adjoint(n0, ln, lam):
            rt.adj(n0, ln, gout, every, Xa, lam, lsum)

        if c is None:
            lam = torch.empty((N, B, npad), dtype=torch.float64, device=dev)
            adjoint(0, N, lam)
            rt.grad(0, N, saved, lam)
            if gsrc is not None:
                src.grad(gsrc, 0, N, lam)
        else:
            Xs = torch.empty((B, npad), dtype=torch.float64, device=dev)
            seg = torch.empty((B, min(c, N), n), dtype=torch.float64, device=dev)
            lam = torch.empty((min(c, N), B, npad), dtype=torch.float64, device=dev)
            for i in reversed(range(saved.shape[0])):
                s = i * c
                ln = min(c, N - s)
                # recompute the segment's states from its first one
                _roll(rt, src, solver._src_steps, Xs, saved[i], seg, s, ln)
                adjoint(s, ln, lam)
                rt.grad(s, ln, seg, lam)
                if gsrc is not None:
                    src.grad(gsrc, s, ln, lam)
        gk = rt.gkappa(kappa)
        gu0 = torch.zeros((B, n), dtype=torch.float64, device=dev)
        gu0[:, rt.free] = rt.mass_free * Xa[:, :nf]          # dL/du0[free] = m * lambda_1
        gf = None
        if ctx.need_f and ctx.per_f:                        # dL/df_b = W^T (dt sum_n lam~_{n,b})
            gf = torch.empty((B, n), dtype=torch.float64, device=dev)
            _src_grad(rt, 1, B, lsum, 0, npad, gf, 0, n)
        elif ctx.need_f:                                    # dL/df = W^T (dt sum_n sum_b lam~_n)
            lt = torch.zeros(n, dtype=torch.float64, device=dev)
            lt[rt.free] = dt * lsum[:, :nf].sum(0)
            gf = torch.empty(n, dtype=torch.float64, device=dev)
            scratch = torch.empty(mesh.n_elements, dtype=torch.float64, device=dev)
            kg = torch.ones(mesh.n_elements, dtype=torch.float64, device=dev) if isinstance(rt, _PerSampleRoute) else kappa
            with _timed("grad", dev):                       # (gf does not depend on kappa; scratch takes dL/dkappa)
                _native.check(L.dfe_grad(h, lt.data_ptr(), lt.data_ptr(), kg.data_ptr(), _native.KAPPA_PER_ELEMENT,
                                         scratch.data_ptr(), gf.data_ptr(), None, 0, st))
        rt.finish_backward("DifferentiableHeatSolver.backward")
        return gu0, gk.reshape(kappa.shape), gf, gsrc, None, None, None, None


class DifferentiableHeatSolver(nn.Module):
    """Differentiable backward-Euler rollouts of the heat equation, the scheme of :class:`HeatStepper`:

        (M_L + dt K(kappa)) u^{n+1} = M_L u^n + dt F(f),   Dirichlet nodes held at the mesh's values.

    ``solver(u0, n_steps, every=None, *, source=None)`` returns the final state (``every=None``) or the states after steps
    ``every, 2 every, ..., n_steps`` as ``(B, n_steps // every, n_nodes)``; gradients flow to ``u0``, ``kappa``, ``f`` and
    ``source`` through the discrete adjoint.  ``source`` is ``(n_steps, n_nodes)`` (one source per step, shared by the
    batch) or ``(B, n_steps, n_nodes)`` (per step and per sample, with ``u0`` of shape ``(B, n_nodes)``); step n (0-based,
    u^n -> u^{n+1}) uses ``f + source[n]``, the backward-Euler evaluation of the source at t_{n+1}.  Each call assembles ``K(kappa)``, factors ``M_L + dt K`` once and synchronises once (a failed
    factorisation, e.g. ``kappa <= 0``, raises ``BreakdownError``).

    Parameters
    ----------
    mesh : FEMesh         2-D P1, ``K_free`` of half bandwidth <= 32 (``rectangle(nx, ny)``, nx <= 32)
    kappa : number or tensor, differentiable; ``kappa.grad`` has ``kappa``'s shape
        ``()`` / ``(1,)`` / ``(n_elements,)``: shared by the batch (also ``(1, 1)``, ``(1, n_elements)`` and
        ``(n_elements, 1)``, which are flattened);
        ``(B, 1)`` / ``(B, n_elements)``: one scalar / one field per sample; ``u0`` must then be ``(B, n_nodes)`` with the
        same B.  When B = n_elements, ``(B, 1)`` keeps its shared meaning: pass per-sample scalars as ``(B, n_elements)``
        with constant rows.  Every sample gets its own ``M_L + dt K(kappa_b)`` and banded factor, ``npad * 33`` doubles
        (262 KB at ``rectangle(32, 32)``, 1.07 GB at B = 4096) kept for the backward; a sample whose matrix is not SPD
        raises ``BreakdownError`` naming the first such sample.  The trajectory and lambda buffers are those of the
        shared route.
    dt : float            not differentiable
    f : None, ``(n_nodes,)`` (shared by the batch) or ``(B, n_nodes)`` (one per sample, with ``u0`` of shape
        ``(B, n_nodes)``): a source constant in time, differentiable; ``f.grad`` has ``f``'s shape.  A per-step source goes
        to the call (``source``).
    checkpoint : keyword-only, None (keep every state for the backward) or c: keep every c-th state and recompute each
        segment of c steps in the backward.  Gradients are bit-identical either way.

    ``u0`` is ``(n_nodes,)`` or ``(B, n_nodes)`` of any float dtype; its Dirichlet entries are ignored (their gradient is 0).
    The output is float64 on ``u0``'s device (a CPU ``u0`` is computed on the current CUDA device).
    """

    # warps per CTA of the rollout kernels; 0 lets the library choose from the batch size (results do not depend on it)
    _cta_warps = 0
    # Steps per rollout launch with a per-step source (results do not depend on it).  A launch's constants take
    # (steps, B, npad) doubles: 16 steps keep them at 16 carries (0.5 GB at B = 4096 on rectangle(32, 32)) against the
    # (B, N, n_nodes) trajectory, while the launches it adds (one load kernel and one rollout per 16 steps) stay few.
    _src_steps = 16

    def __init__(self, mesh: FEMesh, kappa, dt: float, f: torch.Tensor | None = None, *, checkpoint: int | None = None):
        super().__init__()
        if not torch.cuda.is_available():
            raise RuntimeError("DifferentiableHeatSolver runs on CUDA only and no device is visible "
                               "(difffe_physics_lab_b200 has no CPU fallback)")
        if checkpoint is not None and int(checkpoint) < 1:
            raise ValueError(f"checkpoint must be None or >= 1, got {checkpoint}")
        _heat_check_mesh(mesh, torch.device("cuda", torch.cuda.current_device()),
                         per_sample=_per_sample_kappa(kappa, mesh.n_elements))
        self.mesh, self.dt = mesh, float(dt)
        self.checkpoint = None if checkpoint is None else int(checkpoint)
        self.kappa = torch.tensor(float(kappa), dtype=torch.float64) if isinstance(kappa, (int, float)) else kappa
        self.f = f

    def forward(self, u0: torch.Tensor, n_steps: int, every: int | None = None, *,
                source: torch.Tensor | None = None) -> torch.Tensor:
        mesh = self.mesh
        n_steps = int(n_steps)
        if n_steps < 1:
            raise ValueError(f"n_steps must be >= 1, got {n_steps}")
        k = n_steps if every is None else int(every)
        if k < 1 or n_steps % k != 0:
            raise ValueError(f"n_steps ({n_steps}) must be a positive multiple of every ({every})")
        if u0.dim() not in (1, 2) or u0.shape[-1] != mesh.n_nodes:
            raise ValueError(f"u0 must have shape (n_nodes,) or (B, n_nodes) with n_nodes={mesh.n_nodes}, got {tuple(u0.shape)}")
        per_sample = _per_sample_kappa(self.kappa, mesh.n_elements)
        if per_sample:
            ks = tuple(self.kappa.shape)
            if u0.dim() != 2 or ks[0] != u0.shape[0] or ks[1] not in (1, mesh.n_elements):
                raise ValueError(f"per-sample kappa must be (B, 1) or (B, n_elements={mesh.n_elements}) with u0 of shape "
                                 f"(B, n_nodes); got kappa {ks} and u0 {tuple(u0.shape)}")
            kap = self.kappa.to(dtype=torch.float64)
        else:
            kap = torch.as_tensor(self.kappa, dtype=torch.float64).reshape(-1) if not torch.is_tensor(self.kappa) \
                else self.kappa.to(dtype=torch.float64).reshape(-1)
            if kap.numel() not in (1, mesh.n_elements):
                raise ValueError(f"kappa must have 1 or n_elements={mesh.n_elements} entries, got {kap.numel()}")
        n, Bu = mesh.n_nodes, (u0.shape[0] if u0.dim() == 2 else None)
        if self.f is not None and tuple(self.f.shape) not in ((n,), (Bu, n)):
            raise ValueError(f"f must have shape ({n},) or (B, {n}) with u0 of shape (B, n_nodes); got f "
                             f"{tuple(self.f.shape)} and u0 {tuple(u0.shape)}")
        if source is not None and tuple(source.shape) not in ((n_steps, n), (Bu, n_steps, n)):
            raise ValueError(f"source must have shape (n_steps, n_nodes) = ({n_steps}, {n}) or (B, n_steps, n_nodes) with "
                             f"u0 of shape (B, n_nodes); got source {tuple(source.shape)} and u0 {tuple(u0.shape)}")
        dev = u0.device if u0.is_cuda else torch.device("cuda", torch.cuda.current_device())
        _heat_check_mesh(mesh, dev, per_sample=per_sample)
        batched = u0.dim() == 2
        u = u0.to(device=dev, dtype=torch.float64).reshape(-1, mesh.n_nodes).contiguous()
        fd = None if self.f is None else self.f.to(device=dev, dtype=torch.float64).contiguous()
        sd = None if source is None else source.to(device=dev, dtype=torch.float64).contiguous()
        with torch.cuda.device(dev):
            U = _HeatRollout.apply(u, kap.to(dev).contiguous(), fd, sd, self, n_steps, k, per_sample)
        if every is None:
            U = U[:, 0]
        if not batched:
            U = U[0]
        return U.to(u0.device)
