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
checkpointing.  Gradients flow to ``u0``, ``kappa`` and ``f``.
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


def _heat_check_mesh(mesh: FEMesh, dev: torch.device):
    """NotImplementedError (with the reason) for meshes the differentiable rollout does not take; returns the native mesh."""
    if mesh.dim != 2:
        raise NotImplementedError("DifferentiableHeatSolver supports 2-D meshes only (1-D meshes are not implemented)")
    if mesh.order != 1:
        raise NotImplementedError("DifferentiableHeatSolver supports P1 meshes only (P2 is not implemented)")
    L = _native.lib()
    nm = mesh._native(dev.index)
    if not L.dfe_band_supported(nm.handle):
        raise NotImplementedError("DifferentiableHeatSolver needs a mesh whose K_free has half bandwidth <= 32 "
                                  "(dfe_band_supported; e.g. rectangle(nx, ny) with nx <= 32)")
    if not L.dfe_heat_supported(nm.handle):
        raise NotImplementedError("mesh too large for the trajectory gradient kernel: the per-element sums and three "
                                  "(u, lambda) rows must fit 200 KB of shared memory (dfe_heat_supported)")
    return nm


def _check_status(status: torch.Tensor, fault: torch.Tensor, who: str) -> None:
    """The one synchronisation of a call: the factorisation status and the fault word of the rollout kernels."""
    st = torch.cat([status, fault]).cpu()
    if int(st[0]) != 0:
        raise _native.BreakdownError(_native.ERR_BREAKDOWN, f"{who}: M_L + dt K is not positive definite (kappa <= 0?)")
    if int(st[1]) != 0:
        raise _native.DfeError(_native.ERR_CUDA, f"{who}: a bounded wait inside a rollout kernel expired; outputs invalid")


class _HeatRollout(torch.autograd.Function):
    """(u0 (B, n), kappa (1,) or (n_el,), f (n,) or None) -> the states after steps every, 2 every, ..., N: (B, N / every, n).

    All tensors are float64 and contiguous on the solver's device."""

    @staticmethod
    def forward(ctx, u0, kappa, f, solver, n_steps: int, every: int):
        L = _native.lib()
        dev, mesh, dt, c = u0.device, solver.mesh, solver.dt, solver.checkpoint
        B, n, N = u0.shape[0], mesh.n_nodes, n_steps
        st = torch.cuda.current_stream(dev).cuda_stream
        op = _HeatOperator(mesh, kappa.detach(), dt, None if f is None else f.detach(), dev)
        h, npad, nf = op.nm.handle, op.npad, op.free.numel()
        mf = torch.zeros(npad, dtype=torch.float64, device=dev)
        cf = torch.zeros(npad, dtype=torch.float64, device=dev)
        mf[:nf], cf[:nf] = op.mass_free, op.rhs_const
        fault = torch.zeros(1, dtype=torch.int32, device=dev)
        X = torch.zeros((B, npad), dtype=torch.float64, device=dev)
        w = solver._cta_warps

        def roll(src, traj, steps):
            with _timed("heat_fwd", dev):
                _native.check(L.dfe_heat_fwd(h, B, steps, None if src is None else src.data_ptr(), n, op.factor.data_ptr(),
                                             mf.data_ptr(), cf.data_ptr(), X.data_ptr(), traj.data_ptr(), traj.stride(0),
                                             traj.stride(1), w, fault.data_ptr(), st))

        if c is None:                                       # every state kept: the trajectory is the saved state
            traj = torch.empty((B, N, n), dtype=torch.float64, device=dev)
            roll(u0, traj, N)
            out = traj if every == 1 else traj[:, every - 1::every].contiguous()
            saved = traj
        else:                                               # segments of c steps; only their first states are kept
            seg = torch.empty((B, min(c, N), n), dtype=torch.float64, device=dev)
            out = torch.empty((B, N // every, n), dtype=torch.float64, device=dev)
            starts = [u0]
            for s in range(0, N, c):
                ln = min(c, N - s)
                roll(u0 if s == 0 else None, seg, ln)       # later segments continue from the carry X
                first = (s // every + 1) * every            # first recorded step after s
                if first <= s + ln:
                    out[:, first // every - 1:(s + ln) // every] = seg[:, first - s - 1:ln:every]
                if s + ln < N:
                    starts.append(seg[:, ln - 1].clone())
            saved = torch.stack(starts)
        _check_status(op.status, fault, "DifferentiableHeatSolver")
        ctx.op, ctx.mf, ctx.solver, ctx.N, ctx.every, ctx.kmode = op, mf, solver, N, every, kappa.numel()
        ctx.need_f = f is not None
        ctx.save_for_backward(saved, kappa)
        return out

    @staticmethod
    def backward(ctx, gout):
        L = _native.lib()
        saved, kappa = ctx.saved_tensors
        op, mf, solver, N, every = ctx.op, ctx.mf, ctx.solver, ctx.N, ctx.every
        mesh, dt, c, w = solver.mesh, solver.dt, solver.checkpoint, solver._cta_warps
        dev = saved.device
        h, npad, nf, n = op.nm.handle, op.npad, op.free.numel(), mesh.n_nodes
        B = saved.shape[0] if c is None else saved.shape[1]
        st = torch.cuda.current_stream(dev).cuda_stream
        gout = gout.to(dtype=torch.float64).contiguous()
        fault = torch.zeros(1, dtype=torch.int32, device=dev)
        Xa = torch.zeros((B, npad), dtype=torch.float64, device=dev)       # lambda_{n+1}, zero above step N
        lsum = torch.zeros((B, npad), dtype=torch.float64, device=dev)
        gws = torch.empty(max(int(L.dfe_heat_grad_bytes(h, B, N)), 16), dtype=torch.uint8, device=dev)

        def adjoint(n0, ln, lam):
            with _timed("heat_adj", dev):
                _native.check(L.dfe_heat_adj(h, B, n0, ln, gout.data_ptr(), gout.stride(0), gout.stride(1), every,
                                             op.factor.data_ptr(), mf.data_ptr(), Xa.data_ptr(), lam.data_ptr(),
                                             lsum.data_ptr(), w, fault.data_ptr(), st))

        def grad(n0, ln, traj, lam):
            with _timed("heat_grad", dev):
                _native.check(L.dfe_heat_grad(h, B, n0, ln, N, traj.data_ptr(), traj.stride(0), traj.stride(1),
                                              lam.data_ptr(), gws.data_ptr(), gws.numel(), st))

        if c is None:
            lam = torch.empty((N, B, npad), dtype=torch.float64, device=dev)
            adjoint(0, N, lam)
            grad(0, N, saved, lam)
        else:
            cf = torch.zeros(npad, dtype=torch.float64, device=dev)
            cf[:nf] = op.rhs_const
            Xs = torch.empty((B, npad), dtype=torch.float64, device=dev)
            seg = torch.empty((B, min(c, N), n), dtype=torch.float64, device=dev)
            lam = torch.empty((min(c, N), B, npad), dtype=torch.float64, device=dev)
            for i in reversed(range(saved.shape[0])):
                s = i * c
                ln = min(c, N - s)
                with _timed("heat_fwd", dev):                 # recompute the segment's states from its first one
                    _native.check(L.dfe_heat_fwd(h, B, ln, saved[i].data_ptr(), n, op.factor.data_ptr(), mf.data_ptr(),
                                                 cf.data_ptr(), Xs.data_ptr(), seg.data_ptr(), seg.stride(0),
                                                 seg.stride(1), w, fault.data_ptr(), st))
                adjoint(s, ln, lam)
                grad(s, ln, seg, lam)
        gk = torch.empty(ctx.kmode, dtype=torch.float64, device=dev)
        mode = _native.KAPPA_SCALAR if ctx.kmode == 1 else _native.KAPPA_PER_ELEMENT
        with _timed("heat_grad", dev):
            _native.check(L.dfe_heat_grad_sum(h, B, N, dt, mode, gk.data_ptr(), gws.data_ptr(), gws.numel(), st))
        gu0 = torch.zeros((B, n), dtype=torch.float64, device=dev)
        gu0[:, op.free] = op.mass_free * Xa[:, :nf]          # dL/du0[free] = m * lambda_1
        gf = None
        if ctx.need_f:                                      # dL/df = W^T (dt sum_n sum_b lam~_n)
            lt = torch.zeros(n, dtype=torch.float64, device=dev)
            lt[op.free] = dt * lsum[:, :nf].sum(0)
            gf = torch.empty(n, dtype=torch.float64, device=dev)
            scratch = torch.empty(mesh.n_elements, dtype=torch.float64, device=dev)
            with _timed("grad", dev):
                _native.check(L.dfe_grad(h, lt.data_ptr(), lt.data_ptr(), kappa.data_ptr(), _native.KAPPA_PER_ELEMENT,
                                         scratch.data_ptr(), gf.data_ptr(), None, 0, st))
        _check_status(torch.zeros(1, dtype=torch.int32, device=dev), fault, "DifferentiableHeatSolver.backward")
        return gu0, gk.reshape(kappa.shape), gf, None, None, None


class DifferentiableHeatSolver(nn.Module):
    """Differentiable backward-Euler rollouts of the heat equation, the scheme of :class:`HeatStepper`:

        (M_L + dt K(kappa)) u^{n+1} = M_L u^n + dt F(f),   Dirichlet nodes held at the mesh's values.

    ``solver(u0, n_steps, every=None)`` returns the final state (``every=None``) or the states after steps ``every,
    2 every, ..., n_steps`` as ``(B, n_steps // every, n_nodes)``; gradients flow to ``u0``, ``kappa`` and ``f`` through the
    discrete adjoint.  Each call assembles ``K(kappa)``, factors ``M_L + dt K`` once and synchronises once (a failed
    factorisation, e.g. ``kappa <= 0``, raises ``BreakdownError``).

    Parameters
    ----------
    mesh : FEMesh         2-D P1, ``K_free`` of half bandwidth <= 32 (``rectangle(nx, ny)``, nx <= 32)
    kappa : number or tensor ``()`` / ``(1,)`` / ``(n_elements,)``, shared by the batch, differentiable
    dt : float            not differentiable
    f : None or ``(n_nodes,)`` source, shared by the batch, differentiable
    checkpoint : keyword-only, None (keep every state for the backward) or c: keep every c-th state and recompute each
        segment of c steps in the backward.  Gradients are bit-identical either way.

    ``u0`` is ``(n_nodes,)`` or ``(B, n_nodes)`` of any float dtype; its Dirichlet entries are ignored (their gradient is 0).
    The output is float64 on ``u0``'s device (a CPU ``u0`` is computed on the current CUDA device).
    """

    # warps per CTA of the rollout kernels; 0 lets the library choose from the batch size (results do not depend on it)
    _cta_warps = 0

    def __init__(self, mesh: FEMesh, kappa, dt: float, f: torch.Tensor | None = None, *, checkpoint: int | None = None):
        super().__init__()
        if not torch.cuda.is_available():
            raise RuntimeError("DifferentiableHeatSolver runs on CUDA only and no device is visible "
                               "(difffe_physics_lab_b200 has no CPU fallback)")
        if checkpoint is not None and int(checkpoint) < 1:
            raise ValueError(f"checkpoint must be None or >= 1, got {checkpoint}")
        _heat_check_mesh(mesh, torch.device("cuda", torch.cuda.current_device()))
        self.mesh, self.dt = mesh, float(dt)
        self.checkpoint = None if checkpoint is None else int(checkpoint)
        self.kappa = torch.tensor(float(kappa), dtype=torch.float64) if isinstance(kappa, (int, float)) else kappa
        self.f = f

    def forward(self, u0: torch.Tensor, n_steps: int, every: int | None = None) -> torch.Tensor:
        mesh = self.mesh
        n_steps = int(n_steps)
        if n_steps < 1:
            raise ValueError(f"n_steps must be >= 1, got {n_steps}")
        k = n_steps if every is None else int(every)
        if k < 1 or n_steps % k != 0:
            raise ValueError(f"n_steps ({n_steps}) must be a positive multiple of every ({every})")
        if u0.dim() not in (1, 2) or u0.shape[-1] != mesh.n_nodes:
            raise ValueError(f"u0 must have shape (n_nodes,) or (B, n_nodes) with n_nodes={mesh.n_nodes}, got {tuple(u0.shape)}")
        kap = torch.as_tensor(self.kappa, dtype=torch.float64).reshape(-1) if not torch.is_tensor(self.kappa) \
            else self.kappa.to(dtype=torch.float64).reshape(-1)
        if kap.numel() not in (1, mesh.n_elements):
            raise ValueError(f"kappa must have 1 or n_elements={mesh.n_elements} entries, got {kap.numel()}")
        if self.f is not None and tuple(self.f.shape) != (mesh.n_nodes,):
            raise ValueError(f"f must have shape ({mesh.n_nodes},), got {tuple(self.f.shape)}")
        dev = u0.device if u0.is_cuda else torch.device("cuda", torch.cuda.current_device())
        _heat_check_mesh(mesh, dev)
        batched = u0.dim() == 2
        u = u0.to(device=dev, dtype=torch.float64).reshape(-1, mesh.n_nodes).contiguous()
        fd = None if self.f is None else self.f.to(device=dev, dtype=torch.float64).contiguous()
        with torch.cuda.device(dev):
            U = _HeatRollout.apply(u, kap.to(dev).contiguous(), fd, self, n_steps, k)
        if every is None:
            U = U[:, 0]
        if not batched:
            U = U[0]
        return U.to(u0.device)
