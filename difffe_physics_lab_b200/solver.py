"""``DifferentiableFESolver`` — drop-in for reference ``diffhe/solver.py`` on B200.

Same ``nn.Module`` surface as the reference (``diffhe/solver.py:21-67``): ``DifferentiableFESolver(mesh,
kappa=1.0)``, ``.kappa``, ``solver(f) -> u`` for ``-div(kappa grad u) = f`` with P1 elements and
Dirichlet elimination, differentiable w.r.t. ``kappa`` and ``f``.  The reference's Python element
loop, dense ``K`` and ``torch.linalg.solve`` (solver.py:73-183) are replaced by ONE
``torch.autograd.Function`` whose forward/backward call hand-written sm_100a kernels through the C
ABI in ``include/dfe.h`` (``libdfe_b200.so``, loaded with ctypes).  No Triton, no dispatch, no CPU
fallback: without a CUDA device the call raises.

Extensions over the reference (semantics = a stack of independent reference calls, SURVEY §8b):
``f`` may be ``(B, n_nodes)``; ``kappa`` may be ``()``/``(1,)`` (shared scalar — the only form the
reference accepts), ``(n_el,)`` (shared per-element field), ``(B, 1)`` (per-sample scalar) or
``(B, n_el)``.  Un-batched calls keep returning ``(n_nodes,)``.

Device policy: a CPU ``f`` is copied to the current CUDA device, solved there, and ``u`` is returned
on ``f``'s device (``PhysicsLoss`` feeds CPU tensors, reference loss.py:78-83) unless ``out_device`` says
otherwise.  Large host batches on the fused 1-D path are streamed: row chunks go host -> device on a copy
stream (through pinned staging when ``f`` is pageable) while earlier chunks are being solved, and ``u`` /
``dL/df`` chunks return on a second copy stream — the host <-> device traffic overlaps the kernels.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch
import torch.nn as nn

from . import _native
from .mesh import FEMesh


# --------------------------------------------------------------------------- kernel timing hook
class KernelTimer:
    """Optional CUDA-event timer around the ABI calls (used by bench.py for the roofline numbers).

    ``with KernelTimer() as t: ...`` records one (start, stop) event pair per ABI call on the stream the
    kernels are launched on; ``t.summary()`` synchronises and returns {name: (calls, total_ms)}.
    ``launches`` counts the kernels of libdfe_b200 launched while active."""

    _active: Optional["KernelTimer"] = None
    # kernels of libdfe_b200 launched per ABI call (default pipelined 1-D path: k1d_pipe_ck + k1d_pipe [+ k1d_pipe_gk]
    # + k1d_pipe_poison)
    KERNELS_PER_CALL = {"solve1d_fwd": 3, "solve1d_bwd": 4, "solve1d_bwd_misfit": 4, "batch_fwd": 1, "batch_bwd": 1, "band_factor": 1,
                        "band_fwd": 3, "band_bwd": 3, "band_ps_fwd": 7, "band_ps_bwd": 2, "assemble": 1, "eliminate": 2, "pcg": 1, "scatter": 1,
                        "gather": 1, "grad": 3, "mg_setup": 20, "mg_pcg": 1, "heat_fwd": 1, "heat_adj": 1,
                        "heat_grad": 2, "heat_ps_setup": 6, "heat_ps_fwd": 1, "heat_ps_adj": 1, "heat_ps_grad": 1,
                        "heat_ps_grad_sum": 1}

    def __init__(self):
        self.events = []
        self.launches = 0

    def __enter__(self):
        KernelTimer._active = self
        return self

    def __exit__(self, *exc):
        KernelTimer._active = None

    def summary(self):
        torch.cuda.synchronize()
        out = {}
        for name, a, b in self.events:
            c, ms = out.get(name, (0, 0.0))
            out[name] = (c + 1, ms + a.elapsed_time(b))
        return out


class _timed:
    """Context manager: time one ABI call when a KernelTimer is active, else free."""

    def __init__(self, name: str, device: torch.device):
        self.t = KernelTimer._active
        self.name, self.device = name, device

    def __enter__(self):
        if self.t is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.a.record(torch.cuda.current_stream(self.device))

    def __exit__(self, *exc):
        if self.t is not None:
            b = torch.cuda.Event(enable_timing=True)
            b.record(torch.cuda.current_stream(self.device))
            self.t.events.append((self.name, self.a, b))
            self.t.launches += KernelTimer.KERNELS_PER_CALL.get(self.name, 1)


# --------------------------------------------------------------------------- helpers
def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _stream(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _ws(nbytes: int, device: torch.device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


def _kappa_mode(kappa: torch.Tensor, B: int, n_el: int, batched: bool) -> int:
    """Resolve the kappa layout (SURVEY §8b)."""
    if kappa.dim() <= 1 and kappa.numel() == 1:
        return _native.KAPPA_SCALAR
    if kappa.dim() == 1 and kappa.shape[0] == n_el:
        return _native.KAPPA_PER_ELEMENT
    if kappa.dim() == 2 and batched and kappa.shape[0] == B:
        if kappa.shape[1] == 1:
            return _native.KAPPA_PER_SAMPLE
        if kappa.shape[1] == n_el:
            return _native.KAPPA_PER_SAMPLE_ELEMENT
    raise ValueError(
        f"kappa of shape {tuple(kappa.shape)} is not one of (), (1,), (n_el={n_el},), (B={B}, 1), (B, n_el) "
        "[per-sample forms need a batched f of shape (B, n_nodes)]")


_PER_SAMPLE_MODES = (_native.KAPPA_PER_SAMPLE, _native.KAPPA_PER_SAMPLE_ELEMENT)


def _check_fault(nm, what: str) -> None:
    """Raise if a bounded wait inside a fused 1-D kernel expired (call after a synchronisation point)."""
    if _native.lib().dfe_mesh_fault(nm.handle):
        raise _native.DfeError(_native.ERR_CUDA, f"{what}: a fused 1-D kernel on this mesh exceeded its wait bound; the "
                               "results of that call are NaN — rebuild the mesh handle")


# --------------------------------------------------------------------------- host <-> device row streaming
_PIPE_MIN_BYTES = 32 << 20       # below this a plain copy is as fast
_PIPE_CHUNK_BYTES = 16 << 20     # smallest chunk worth a separate copy + launch
_side = {}


def _side_streams(dev: torch.device):
    st = _side.get(dev.index)
    if st is None:
        st = _side[dev.index] = (torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev))
    return st


def _row_chunks(B: int, n: int, host_io: bool):
    """Row ranges of a (B, n) float64 batch: one range unless rows cross the host boundary and the batch is large."""
    total = 8 * B * n
    if not host_io or B < 2 or total < _PIPE_MIN_BYTES:
        return [(0, B)]
    k = int(min(8, B, max(1, total // _PIPE_CHUNK_BYTES)))
    bs = -(-B // k)
    return [(lo, min(B, lo + bs)) for lo in range(0, B, bs)]


class _RowPipe:
    """Streams the rows of a batch through the device while kernels run (one instance per forward / backward call).

    ``in_host``  (B, n) CPU tensor or None: chunk j is copied into a rotating device buffer on the H2D stream (directly
                 when pinned, else through two pinned staging buffers) and handed to the kernel as ``src``.
    ``out_host`` (B, n) pinned CPU tensor or None: after the kernel of chunk j the rows of ``out_dev`` (a full device
                 tensor) — or, when ``out_dev`` is None, of a rotating device buffer handed to the kernel as ``dst`` — are
                 copied back on the D2H stream.
    The compute stream is the caller's current stream; ``finish()`` makes the host wait for the D2H copies only.
    """

    NBUF = 3

    def __init__(self, dev, n, chunks, in_host=None, out_host=None, out_dev=None):
        self.dev, self.n, self.chunks = dev, n, chunks
        self.in_host, self.out_host, self.out_dev = in_host, out_host, out_dev
        self.main = torch.cuda.current_stream(dev)
        self.h2d, self.d2h = _side_streams(dev)
        bs = max(hi - lo for lo, hi in chunks)
        nb = min(self.NBUF, len(chunks))
        self.ibuf = [torch.empty((bs, n), dtype=torch.float64, device=dev) for _ in range(nb)] if in_host is not None else None
        self.obuf = ([torch.empty((bs, n), dtype=torch.float64, device=dev) for _ in range(nb)]
                     if (out_host is not None and out_dev is None) else None)
        self.stage = None
        if in_host is not None and not in_host.is_pinned():
            self.stage = [torch.empty((bs, n), dtype=torch.float64, pin_memory=True) for _ in range(min(2, len(chunks)))]
        ev = torch.cuda.Event
        self.copied = [ev() for _ in chunks]
        self.done = [ev() for _ in chunks]
        self.back = [ev() for _ in chunks]
        # buffers were allocated on the compute stream: order the side streams after everything enqueued so far
        e0 = ev()
        e0.record(self.main)
        self.h2d.wait_event(e0)
        self.d2h.wait_event(e0)
        self._issued = 0
        if in_host is not None:                 # copies run up to NBUF - 1 chunks ahead of the kernels
            for j in range(min(nb - 1, len(chunks))):
                self._issue_h2d(j)

    def _issue_h2d(self, j):
        lo, hi = self.chunks[j]
        nb = len(self.ibuf)
        with torch.cuda.stream(self.h2d):
            if j >= nb:
                self.h2d.wait_event(self.done[j - nb])          # the kernel that read this buffer has finished
            src = self.in_host[lo:hi]
            if self.stage is not None:
                k = j % len(self.stage)
                if j >= len(self.stage):
                    self.copied[j - len(self.stage)].synchronize()   # staging buffer drained (host wait)
                self.stage[k][:hi - lo].copy_(src)
                src = self.stage[k][:hi - lo]
            self.ibuf[j % nb][:hi - lo].copy_(src, non_blocking=True)
            self.copied[j].record(self.h2d)
        self._issued = j + 1

    def run(self, kernel):
        """kernel(j, lo, hi, src, dst): enqueue the work of rows [lo, hi) on the current stream."""
        for j, (lo, hi) in enumerate(self.chunks):
            src = dst = None
            if self.in_host is not None:
                while self._issued <= min(j + len(self.ibuf) - 1, len(self.chunks) - 1):
                    self._issue_h2d(self._issued)
                self.main.wait_event(self.copied[j])
                src = self.ibuf[j % len(self.ibuf)][:hi - lo]
            if self.obuf is not None:
                nb = len(self.obuf)
                if j >= nb:
                    self.main.wait_event(self.back[j - nb])       # the D2H copy out of this buffer has finished
                dst = self.obuf[j % nb][:hi - lo]
            kernel(j, lo, hi, src, dst)
            self.done[j].record(self.main)
            if self.out_host is not None:
                with torch.cuda.stream(self.d2h):
                    self.d2h.wait_event(self.done[j])
                    self.out_host[lo:hi].copy_(dst if dst is not None else self.out_dev[lo:hi], non_blocking=True)
                    self.back[j].record(self.d2h)

    def finish(self):
        if self.out_host is not None:
            self.back[-1].synchronize()


def _pinned_like(B: int, n: int) -> torch.Tensor:
    return torch.empty((B, n), dtype=torch.float64, pin_memory=True)


def _to_host(t: torch.Tensor) -> torch.Tensor:
    """Device -> host copy of a result.  Large results land in pinned memory (torch's caching host allocator keeps the
    pages): a copy into pageable memory runs at a fraction of the PCIe rate."""
    if t.numel() * t.element_size() < _PIPE_MIN_BYTES:
        return t.cpu()
    out = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
    out.copy_(t, non_blocking=True)
    torch.cuda.current_stream(t.device).synchronize()
    return out


class _FESolve(torch.autograd.Function):
    """u = K(kappa)^{-1}-solve of the assembled P1 system; backward = adjoint solve + dL/dkappa, dL/df.

    ``f`` is (B, n) float64 contiguous, on the CPU or on ``dev``; ``kappa`` float64 contiguous on ``dev``.  ``u`` is returned
    on ``out_dev``; a device copy is kept for the adjoint either way."""

    @staticmethod
    def forward(ctx, f: torch.Tensor, kappa: torch.Tensor, mesh: FEMesh, mode: int, opts: dict, dev: torch.device,
                out_dev: torch.device):
        nm = mesh._native(dev.index)
        B, n = f.shape
        L = _native.lib()
        f_host = not f.is_cuda
        ctx.f_host = f_host
        out_host = out_dev.type != "cuda"
        # fused 1-D path: decided once, here, for both directions (dfe_solve1d_supported)
        fused = bool(nm.info.chain1d) and bool(L.dfe_solve1d_supported(nm.handle, mode, int(opts["n_refine"])))
        if bool(nm.info.chain1d) and not fused and n > 200000:
            # the only other route is Jacobi-PCG, which needs O(n) iterations on a 1-D chain: refuse instead
            raise NotImplementedError(
                f"1-D chain mesh with {n} nodes: above 2e5 nodes the fused path needs the multi-sweep kernel, which holds "
                "every chunk of a sample co-resident (about 2 * #SMs * 3328 nodes, scalar / per-sample kappa only)")
        saved_mats = None
        ctx.batch = None
        with torch.cuda.device(dev):
            u = torch.empty((B, n), dtype=torch.float64, device=dev)
            u_out = u
            if fused:
                chunks = _row_chunks(B, n, f_host or out_host)
                ws = _ws(L.dfe_solve1d_workspace_bytes(nm.handle, max(hi - lo for lo, hi in chunks)), dev)
                st = _stream(dev)
                krow = kappa.numel() // B if mode in _PER_SAMPLE_MODES else 0
                kflat = kappa.reshape(-1)
                if len(chunks) == 1 and f_host:
                    f = f.to(dev, non_blocking=f.is_pinned())
                    f_host = False
                stream_out = out_host and len(chunks) > 1
                if stream_out:
                    u_out = _pinned_like(B, n)

                def kern(j, lo, hi, src, dst):
                    fin = src if src is not None else f[lo:hi]
                    with _timed("solve1d_fwd", dev):
                        _native.check(L.dfe_solve1d_fwd(nm.handle, hi - lo, fin.data_ptr(), fin.stride(0),
                                                        kflat[lo * krow:].data_ptr(), mode, int(opts["n_refine"]),
                                                        u[lo:hi].data_ptr(), u.stride(0), ws.data_ptr(), ws.numel(), st))

                if f_host or stream_out:
                    pipe = _RowPipe(dev, n, chunks, f if f_host else None, u_out if stream_out else None, u)
                    pipe.run(kern)
                    pipe.finish()
                else:                                       # everything on the device: one launch, no events
                    kern(0, 0, B, None, None)
                if out_host:
                    if not stream_out:
                        u_out = _to_host(u)
                    _check_fault(nm, "dfe_solve1d_fwd")      # the host waited for u: the fault word is final
            else:
                if f_host:
                    f = f.to(dev, non_blocking=f.is_pinned())
                # many samples, one matrix: banded direct solver or one-CTA-per-sample PCG (config 5b)
                if B >= int(opts.get("batch_min", 2)) and mode in (_native.KAPPA_SCALAR, _native.KAPPA_PER_ELEMENT):
                    ctx.batch = _batch_solver(L, nm, opts)
                # many samples, one matrix each: per-sample banded factorisations in batched kernels
                elif (B >= int(opts.get("batch_min", 2)) and opts.get("batch_solver", "auto") in ("auto", "band")
                      and L.dfe_band_ps_supported(nm.handle)):
                    ctx.batch = "band_ps"
                if ctx.batch == "band_ps":
                    saved_mats = _band_ps_forward(L, nm, f, kappa, mode, u, opts, keep=any(ctx.needs_input_grad[:2]))
                else:
                    fwd = {"band": _band_forward, "pcg": _batch_forward, None: _general_forward}[ctx.batch]
                    saved_mats = fwd(L, nm, f, kappa, mode, u, opts)
                if out_host:
                    u_out = _to_host(u)
        ctx.mesh, ctx.mode, ctx.opts, ctx.fused, ctx.dev = mesh, mode, opts, fused, dev
        ctx.mats = saved_mats
        ctx.save_for_backward(u, kappa)
        return u_out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gbar: torch.Tensor):
        u, kappa = ctx.saved_tensors
        need_f, need_k = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        dev = ctx.dev
        nm = ctx.mesh._native(dev.index)
        L = _native.lib()
        B, n = u.shape
        mode = ctx.mode
        gbar = gbar.contiguous()
        g_host = not gbar.is_cuda
        gf_host = need_f and ctx.f_host
        gk = torch.empty_like(kappa)
        with torch.cuda.device(dev):
            if ctx.fused:
                chunks = _row_chunks(B, n, g_host or gf_host)
                ws = _ws(L.dfe_solve1d_workspace_bytes(nm.handle, max(hi - lo for lo, hi in chunks)), dev)
                st = _stream(dev)
                per_sample = mode in _PER_SAMPLE_MODES
                krow = kappa.numel() // B if per_sample else 0
                kflat, gkflat = kappa.reshape(-1), gk.reshape(-1)
                if len(chunks) == 1 and g_host:
                    gbar = gbar.to(dev, non_blocking=gbar.is_pinned())
                    g_host = False
                gf = None
                if need_f:
                    gf = _pinned_like(B, n) if (gf_host and len(chunks) > 1) else torch.empty((B, n), dtype=torch.float64, device=dev)
                stream_gf = need_f and not gf.is_cuda
                # shared kappa: one partial per chunk, added in chunk order below (deterministic)
                gk_parts = None if per_sample or len(chunks) == 1 else torch.empty((len(chunks), kappa.numel()), dtype=torch.float64, device=dev)

                def kern(j, lo, hi, src, dst):
                    gin = src if src is not None else gbar[lo:hi]
                    gout = dst if dst is not None else (gf[lo:hi] if need_f else None)
                    gko = gkflat[lo * krow:] if per_sample else (gkflat if gk_parts is None else gk_parts[j])
                    with _timed("solve1d_bwd", dev):
                        _native.check(L.dfe_solve1d_bwd(nm.handle, hi - lo, gin.data_ptr(), gin.stride(0), u[lo:hi].data_ptr(),
                                                        u.stride(0), kflat[lo * krow:].data_ptr(), mode, int(ctx.opts["n_refine"]),
                                                        _ptr(gout), gout.stride(0) if gout is not None else n, gko.data_ptr(),
                                                        ws.data_ptr(), ws.numel(), st))

                pipe = _RowPipe(dev, n, chunks, gbar if g_host else None, gf if stream_gf else None, None) if (g_host or stream_gf) else None
                if pipe is not None:
                    pipe.run(kern)
                else:
                    for j, (lo, hi) in enumerate(chunks):
                        kern(j, lo, hi, None, None)
                if gk_parts is not None:
                    gk.copy_(gk_parts.sum(dim=0).reshape(gk.shape))   # torch.sum on CUDA is deterministic (no atomics)
                if pipe is not None:
                    pipe.finish()
                if need_f and gf_host and gf.is_cuda:
                    gf = _to_host(gf)
            else:
                if g_host:
                    gbar = gbar.to(dev, non_blocking=gbar.is_pinned())
                gf = torch.empty_like(u) if need_f else None
                if ctx.batch == "band":
                    _band_backward(L, nm, gbar, u, kappa, mode, ctx.mats, gf, gk, ctx.opts)
                elif ctx.batch == "band_ps":
                    _band_ps_backward(L, nm, gbar, u, mode, ctx.mats, gf, gk, ctx.opts)
                elif ctx.batch == "pcg":
                    _batch_backward(L, nm, gbar, u, kappa, mode, ctx.mats, gf, gk, ctx.opts)
                else:
                    _general_backward(L, nm, gbar, u, kappa, mode, ctx.mats, gf, gk, ctx.opts)
                if gf_host:
                    gf = _to_host(gf)
        return gf, (gk if need_k else None), None, None, None, None, None


class _FEMisfit(torch.autograd.Function):
    """loss = (1 / n_nodes) * sum_b sum_i (u_bi - u_data_bi)^2 and its gradients in two kernels (fused 1-D path):
    the forward solve, then the misfit adjoint (``dfe_solve1d_bwd_misfit``) that forms gbar = 2 (u - u_data) / n_nodes on
    the fly and accumulates the loss next to dL/dkappa.  The gradients are computed in ``forward`` (the loss is a
    scalar, so ``backward`` only scales them) — this is the step of the reference's kappa-recovery loop
    (examples/poisson_1d_demo.py:104-110) without ever materialising gbar.

    ``out2`` (optional, shared kappa only): a persistent 2-double device buffer that receives
    [sum_b dL/dkappa, loss] — the words a data-parallel step all-reduces."""

    @staticmethod
    def forward(ctx, f, kappa, u_data, mesh, mode, opts, out2, weight):
        dev = f.device
        nm = mesh._native(dev.index)
        B, n = f.shape
        L = _native.lib()
        need_f = ctx.needs_input_grad[0]
        per_sample = mode == _native.KAPPA_PER_SAMPLE
        with torch.cuda.device(dev):
            st = _stream(dev)
            u = torch.empty((B, n), dtype=torch.float64, device=dev)
            ws = _ws(L.dfe_solve1d_workspace_bytes(nm.handle, B), dev)
            with _timed("solve1d_fwd", dev):
                _native.check(L.dfe_solve1d_fwd(nm.handle, B, f.data_ptr(), f.stride(0), kappa.data_ptr(), mode,
                                                int(opts["n_refine"]), u.data_ptr(), u.stride(0), ws.data_ptr(), ws.numel(), st))
            gf = torch.empty((B, n), dtype=torch.float64, device=dev) if need_f else None
            if per_sample:
                gk = torch.empty(B, dtype=torch.float64, device=dev)
                lossv = torch.empty(B, dtype=torch.float64, device=dev)
                gk_ptr, loss_ptr = gk.data_ptr(), lossv.data_ptr()
            else:
                if out2 is None:
                    out2 = torch.empty(2, dtype=torch.float64, device=dev)
                gk_ptr, loss_ptr = out2.data_ptr(), out2.data_ptr() + 8
            with _timed("solve1d_bwd_misfit", dev):
                _native.check(L.dfe_solve1d_bwd_misfit(nm.handle, B, u_data.data_ptr(), u_data.stride(0), u.data_ptr(),
                                                       u.stride(0), kappa.data_ptr(), mode, int(opts["n_refine"]),
                                                       2.0 * weight / n,
                                                       _ptr(gf), gf.stride(0) if gf is not None else n, gk_ptr, loss_ptr,
                                                       ws.data_ptr(), ws.numel(), st))
            if per_sample:
                loss = lossv.sum()
                gk = gk.reshape(kappa.shape)
            elif any(ctx.needs_input_grad[:2]):
                loss = out2[1].clone()
                gk = out2[0].clone().reshape(kappa.shape)
            else:                       # no graph (the sharded sweep reads out2 itself): no copy kernels
                loss = out2[1]
                gk = out2[0].reshape(kappa.shape)
        opts["last_u"] = u
        ctx.save_for_backward(gk, gf if gf is not None else torch.empty(0, device=dev))
        ctx.has_gf = gf is not None
        return loss

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gout):
        gk, gf = ctx.saved_tensors
        return (gout * gf if ctx.has_gf and ctx.needs_input_grad[0] else None,
                gout * gk if ctx.needs_input_grad[1] else None, None, None, None, None, None, None)


def _raise_batch_status(status, iters, relres, tol, what):
    """Turn the per-sample status array of the batched solver into the exceptions of the per-sample path."""
    worst = int(status.max())          # one synchronisation per call
    if worst == 0:
        return
    b = int(torch.argmax(status))
    if worst == 4:
        raise _native.NotConvergedError(_native.ERR_NOT_CONVERGED,
                                        f"{what}: sample {b} not converged after {int(iters[b])} iterations "
                                        f"(relative residual {float(relres[b]):.3e}, tol {tol:.3e})")
    raise _native.BreakdownError(_native.ERR_BREAKDOWN,
                                 f"{what}: breakdown in sample {b} at iteration {int(iters[b])} (p^T K p <= 0 or non-finite): "
                                 "K_free is not SPD — does the mesh have a Dirichlet node?")


def _batch_solver(L, nm, opts):
    """Which batched route a shared-matrix batch takes: 'band' (direct, half bandwidth <= 32), 'pcg' (one CTA per
    sample, matrix in shared memory) or None (per-sample cooperative PCG)."""
    want = opts.get("batch_solver", "auto")
    if want in ("auto", "band") and L.dfe_band_supported(nm.handle):
        return "band"
    if want in ("auto", "pcg") and L.dfe_batch_supported(nm.handle):
        return "pcg"
    return None


def _band_forward(L, nm, f, kappa, mode, u, opts):
    """Shared matrix with half bandwidth <= 32: K_free = L L^T once, two banded triangular solves per sample."""
    dev = f.device
    I = nm.info
    B = f.shape[0]
    st = _stream(dev)
    amode = _native.KAPPA_SCALAR if mode == _native.KAPPA_SCALAR else _native.KAPPA_PER_ELEMENT
    vals = torch.empty(max(I.nnz_full, 1), dtype=torch.float64, device=dev)
    F0 = torch.empty(I.n_nodes, dtype=torch.float64, device=dev)
    with _timed("assemble", dev):
        _native.check(L.dfe_assemble(nm.handle, kappa.reshape(-1).data_ptr(), amode, f[0].data_ptr(), vals.data_ptr(),
                                     F0.data_ptr(), st))
    factor = _ws(L.dfe_band_factor_bytes(nm.handle), dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    with _timed("band_factor", dev):
        _native.check(L.dfe_band_factor(nm.handle, vals.data_ptr(), factor.data_ptr(), status.data_ptr(), st))
    ws = _ws(L.dfe_band_workspace_bytes(nm.handle, B), dev)
    with _timed("band_fwd", dev):
        _native.check(L.dfe_band_fwd(nm.handle, B, f.data_ptr(), f.stride(0), vals.data_ptr(), factor.data_ptr(),
                                     u.data_ptr(), u.stride(0), ws.data_ptr(), ws.numel(), st))
    if int(status) != 0:              # one synchronisation per call
        raise _native.BreakdownError(_native.ERR_BREAKDOWN, "dfe_band_factor: a pivot of the Cholesky factorisation is <= 0: "
                                     "K_free is not SPD — does the mesh have a Dirichlet node?")
    opts["last_pcg"] = [(0, 0.0)]     # direct solve: no iterations
    return [("band", factor)]


def _band_backward(L, nm, gbar, u, kappa, mode, mats, gf, gk, opts):
    dev = u.device
    I = nm.info
    B = u.shape[0]
    st = _stream(dev)
    factor = mats[0][1]
    gmode = _native.KAPPA_SCALAR if mode == _native.KAPPA_SCALAR else _native.KAPPA_PER_ELEMENT
    nk = 1 if gmode == _native.KAPPA_SCALAR else I.n_elements
    gk_b = torch.empty((B, nk), dtype=torch.float64, device=dev)
    ws = _ws(L.dfe_band_workspace_bytes(nm.handle, B), dev)
    with _timed("band_bwd", dev):
        _native.check(L.dfe_band_bwd(nm.handle, B, gbar.data_ptr(), gbar.stride(0), u.data_ptr(), u.stride(0),
                                     factor.data_ptr(), gmode, _ptr(gf), gf.stride(0) if gf is not None else I.n_nodes,
                                     gk_b.data_ptr(), ws.data_ptr(), ws.numel(), st))
    opts["last_pcg_adjoint"] = [(0, 0.0)]
    gk.copy_(gk_b.sum(dim=0).reshape(gk.shape))   # torch.sum on CUDA is deterministic (no atomics)


def _band_ps_forward(L, nm, f, kappa, mode, u, opts, keep):
    """kappa (B, 1) or (B, n_el), half bandwidth <= 32: every sample's K_free(kappa_b) is assembled, factored and solved in
    batched kernels (dfe_band_ps_fwd).  The factors are returned for the adjoint when ``keep`` (an input needs a gradient)."""
    dev = f.device
    B = f.shape[0]
    st = _stream(dev)
    factors = _ws(L.dfe_band_ps_factor_bytes(nm.handle, B), dev)
    ws = _ws(L.dfe_band_ps_workspace_bytes(nm.handle, B), dev)
    status = torch.empty(B, dtype=torch.int32, device=dev)
    with _timed("band_ps_fwd", dev):
        _native.check(L.dfe_band_ps_fwd(nm.handle, B, f.data_ptr(), f.stride(0), kappa.data_ptr(), mode, factors.data_ptr(),
                                        u.data_ptr(), u.stride(0), status.data_ptr(), ws.data_ptr(), ws.numel(), st))
    if int(status.max()) != 0:        # one synchronisation per call
        b = int(torch.argmax(status))  # the first failing sample
        raise _native.BreakdownError(_native.ERR_BREAKDOWN, f"dfe_band_ps_fwd: sample {b}: a pivot of the Cholesky "
                                     "factorisation is <= 0: K_free(kappa_b) is not SPD — is kappa_b > 0?")
    opts["last_pcg"] = [(0, 0.0)]     # direct solve: no iterations
    return [("band_ps", factors)] if keep else None


def _band_ps_backward(L, nm, gbar, u, mode, mats, gf, gk, opts):
    dev = u.device
    B = u.shape[0]
    st = _stream(dev)
    ws = _ws(L.dfe_band_ps_workspace_bytes(nm.handle, B), dev)
    with _timed("band_ps_bwd", dev):
        _native.check(L.dfe_band_ps_bwd(nm.handle, B, gbar.data_ptr(), gbar.stride(0), u.data_ptr(), u.stride(0),
                                        mats[0][1].data_ptr(), mode, _ptr(gf), gf.stride(0) if gf is not None else nm.info.n_nodes,
                                        gk.data_ptr(), ws.data_ptr(), ws.numel(), st))
    opts["last_pcg_adjoint"] = [(0, 0.0)]


def _batch_forward(L, nm, f, kappa, mode, u, opts):
    """Shared matrix, many right-hand sides, small mesh: assemble / eliminate ONCE, then one CTA per sample
    (dfe_batch_fwd).  Returns the saved (sell, dinv) like the per-sample path."""
    dev = f.device
    I = nm.info
    B = f.shape[0]
    st = _stream(dev)
    amode = _native.KAPPA_SCALAR if mode == _native.KAPPA_SCALAR else _native.KAPPA_PER_ELEMENT
    vals = torch.empty(max(I.nnz_full, 1), dtype=torch.float64, device=dev)
    F0 = torch.empty(I.n_nodes, dtype=torch.float64, device=dev)
    sell = torch.empty(max(I.sell_nnz, 1), dtype=torch.float64, device=dev)
    dinv = torch.empty(max(I.n_free, 1), dtype=torch.float64, device=dev)
    Ff0 = torch.empty(max(I.n_free, 1), dtype=torch.float64, device=dev)
    with _timed("assemble", dev):
        _native.check(L.dfe_assemble(nm.handle, kappa.reshape(-1).data_ptr(), amode, f[0].data_ptr(), vals.data_ptr(),
                                     F0.data_ptr(), st))
    with _timed("eliminate", dev):
        _native.check(L.dfe_eliminate(nm.handle, vals.data_ptr(), F0.data_ptr(), None, sell.data_ptr(), Ff0.data_ptr(),
                                      dinv.data_ptr(), st))
    iters = torch.empty(B, dtype=torch.int32, device=dev)
    relres = torch.empty(B, dtype=torch.float64, device=dev)
    status = torch.empty(B, dtype=torch.int32, device=dev)
    tol = float(opts["pcg_tol"])
    with _timed("batch_fwd", dev):
        _native.check(L.dfe_batch_fwd(nm.handle, B, f.data_ptr(), f.stride(0), vals.data_ptr(), sell.data_ptr(),
                                      dinv.data_ptr(), u.data_ptr(), u.stride(0), tol,
                                      int(opts["pcg_maxit"] or max(10 * I.n_free, 1000)), iters.data_ptr(),
                                      relres.data_ptr(), status.data_ptr(), st))
    _raise_batch_status(status, iters, relres, tol, "dfe_batch_fwd")
    opts["last_pcg"] = [(int(iters.max()), float(relres.max()))]
    return [(sell, dinv)]


def _batch_backward(L, nm, gbar, u, kappa, mode, mats, gf, gk, opts):
    dev = u.device
    I = nm.info
    B = u.shape[0]
    st = _stream(dev)
    sell, dinv = mats[0]
    gmode = _native.KAPPA_SCALAR if mode == _native.KAPPA_SCALAR else _native.KAPPA_PER_ELEMENT
    nk = 1 if gmode == _native.KAPPA_SCALAR else I.n_elements
    gk_b = torch.empty((B, nk), dtype=torch.float64, device=dev)
    iters = torch.empty(B, dtype=torch.int32, device=dev)
    relres = torch.empty(B, dtype=torch.float64, device=dev)
    status = torch.empty(B, dtype=torch.int32, device=dev)
    tol = float(opts["pcg_tol"])
    with _timed("batch_bwd", dev):
        _native.check(L.dfe_batch_bwd(nm.handle, B, gbar.data_ptr(), gbar.stride(0), u.data_ptr(), u.stride(0),
                                      sell.data_ptr(), dinv.data_ptr(), gmode, _ptr(gf),
                                      gf.stride(0) if gf is not None else I.n_nodes, gk_b.data_ptr(), tol,
                                      int(opts["pcg_maxit"] or max(10 * I.n_free, 1000)), iters.data_ptr(),
                                      relres.data_ptr(), status.data_ptr(), st))
    _raise_batch_status(status, iters, relres, tol, "dfe_batch_bwd")
    opts["last_pcg_adjoint"] = [(int(iters.max()), float(relres.max()))]
    gk.copy_(gk_b.sum(dim=0).reshape(gk.shape))   # torch.sum on CUDA is deterministic (no atomics)


def _use_mg(L, nm, opts) -> bool:
    """Structured 2-D mesh (FEMesh.rectangle() topology): CG preconditioned by a multigrid V-cycle instead of Jacobi."""
    want = opts.get("solver2d", "auto")
    if want not in ("auto", "mg", "jacobi"):
        raise ValueError(f"solver2d must be 'auto', 'mg' or 'jacobi', got {want!r}")
    return want != "jacobi" and bool(L.dfe_mg_supported(nm.handle))


def _solve_general(L, nm, mat, rhs, x, opts, ws_j, ws_m, st, key):
    """One linear solve with the operator `mat` = ('mg', hierarchy) or ('jacobi', sell, dinv); returns (iters, relres)."""
    it, rel = C.c_int64(0), C.c_double(0.0)
    tol = float(opts["pcg_tol"])
    dev = rhs.device
    if mat[0] == "mg":
        with _timed("mg_pcg", dev):
            _native.check(L.dfe_mg_pcg(nm.handle, mat[1].data_ptr(), rhs.data_ptr(), x.data_ptr(), tol,
                                       int(opts["pcg_maxit"] or 1000), int(opts.get("mg_nu", 2)), C.byref(it), C.byref(rel),
                                       ws_m.data_ptr(), ws_m.numel(), st))
    else:
        with _timed("pcg", dev):
            _native.check(L.dfe_pcg(nm.handle, mat[1].data_ptr(), mat[2].data_ptr(), rhs.data_ptr(), x.data_ptr(), tol,
                                    int(opts["pcg_maxit"] or max(10 * nm.info.n_free, 1000)), C.byref(it), C.byref(rel),
                                    ws_j.data_ptr(), ws_j.numel(), st))
    return it.value, rel.value


def _general_forward(L, nm, f, kappa, mode, u, opts):
    """assemble -> eliminate -> PCG -> scatter, per sample; the matrix (and its multigrid hierarchy) is built once when
    kappa is shared by the batch."""
    dev = f.device
    I = nm.info
    B = f.shape[0]
    st = _stream(dev)
    n_el = I.n_elements
    shared = mode in (_native.KAPPA_SCALAR, _native.KAPPA_PER_ELEMENT)
    amode = _native.KAPPA_SCALAR if mode in (_native.KAPPA_SCALAR, _native.KAPPA_PER_SAMPLE) else _native.KAPPA_PER_ELEMENT
    kflat = kappa.reshape(-1)
    mg = _use_mg(L, nm, opts)
    ws_j = _ws(L.dfe_pcg_workspace_bytes(nm.handle), dev)
    ws_m = _ws(L.dfe_mg_workspace_bytes(nm.handle), dev) if mg else None
    vals = torch.empty(max(I.nnz_full, 1), dtype=torch.float64, device=dev)
    F = torch.empty(I.n_nodes, dtype=torch.float64, device=dev)
    x = torch.empty(max(I.n_free, 1), dtype=torch.float64, device=dev)
    Ff = torch.empty(max(I.n_free, 1), dtype=torch.float64, device=dev)
    mats = []
    iters = []
    for b in range(B):
        if mode == _native.KAPPA_PER_SAMPLE:
            kb = kflat[b:b + 1]
        elif mode == _native.KAPPA_PER_SAMPLE_ELEMENT:
            kb = kflat[b * n_el:(b + 1) * n_el]
        else:
            kb = kflat
        # assembly is repeated per sample even for shared kappa: F depends on f[b]; cheap next to the solve
        with _timed("assemble", dev):
            _native.check(L.dfe_assemble(nm.handle, kb.data_ptr(), amode, f[b].data_ptr(), vals.data_ptr(), F.data_ptr(), st))
        new_matrix = not shared or b == 0
        mat = mats[0] if not new_matrix else None
        if new_matrix and mg:
            hier = _ws(L.dfe_mg_hierarchy_bytes(nm.handle), dev)
            try:
                with _timed("mg_setup", dev):
                    _native.check(L.dfe_mg_setup(nm.handle, vals.data_ptr(), hier.data_ptr(), hier.numel(), st))
                mat = ("mg", hier)
            except NotImplementedError:          # not numerically a 5-point operator (distorted grid): Jacobi-PCG
                if opts.get("solver2d", "auto") == "mg":
                    raise
                mg = False
        if mat is None:
            sell = torch.empty(max(I.sell_nnz, 1), dtype=torch.float64, device=dev)
            dinv = torch.empty(max(I.n_free, 1), dtype=torch.float64, device=dev)
            mat = ("jacobi", sell, dinv)
        with _timed("eliminate", dev):
            if new_matrix and mat[0] == "jacobi":
                _native.check(L.dfe_eliminate(nm.handle, vals.data_ptr(), F.data_ptr(), None, mat[1].data_ptr(), Ff.data_ptr(),
                                              mat[2].data_ptr(), st))
            else:                                 # only the lifted load is needed
                if "dinv_scratch" not in opts or opts["dinv_scratch"].numel() != max(I.n_free, 1) or opts["dinv_scratch"].device != dev:
                    opts["dinv_scratch"] = torch.empty(max(I.n_free, 1), dtype=torch.float64, device=dev)
                _native.check(L.dfe_eliminate(nm.handle, vals.data_ptr(), F.data_ptr(), None, None, Ff.data_ptr(),
                                              opts["dinv_scratch"].data_ptr(), st))
        iters.append(_solve_general(L, nm, mat, Ff, x, opts, ws_j, ws_m, st, "last_pcg"))
        _native.check(L.dfe_scatter(nm.handle, x.data_ptr(), 0, u[b].data_ptr(), st))
        if new_matrix:
            mats.append(mat)
    opts["last_pcg"] = iters
    opts["last_solver2d"] = mats[0][0] if mats else None
    return mats


def _general_backward(L, nm, gbar, u, kappa, mode, mats, gf, gk, opts):
    dev = u.device
    I = nm.info
    B = u.shape[0]
    st = _stream(dev)
    shared = mode in (_native.KAPPA_SCALAR, _native.KAPPA_PER_ELEMENT)
    gmode = _native.KAPPA_SCALAR if mode in (_native.KAPPA_SCALAR, _native.KAPPA_PER_SAMPLE) else _native.KAPPA_PER_ELEMENT
    ws_j = _ws(L.dfe_pcg_workspace_bytes(nm.handle), dev)
    ws_m = _ws(L.dfe_mg_workspace_bytes(nm.handle), dev) if any(m[0] == "mg" for m in mats) else None
    gws = _ws(L.dfe_grad_workspace_bytes(nm.handle), dev)
    gfree = torch.empty(max(I.n_free, 1), dtype=torch.float64, device=dev)
    lam_free = torch.empty(max(I.n_free, 1), dtype=torch.float64, device=dev)
    lam = torch.zeros(I.n_nodes, dtype=torch.float64, device=dev)
    nk = 1 if gmode == _native.KAPPA_SCALAR else I.n_elements
    gk_b = torch.empty((B, nk), dtype=torch.float64, device=dev)
    iters = []
    for b in range(B):
        mat = mats[0] if shared else mats[b]
        _native.check(L.dfe_gather_free(nm.handle, gbar[b].data_ptr(), gfree.data_ptr(), st))
        iters.append(_solve_general(L, nm, mat, gfree, lam_free, opts, ws_j, ws_m, st, "last_pcg_adjoint"))
        _native.check(L.dfe_scatter(nm.handle, lam_free.data_ptr(), 1, lam.data_ptr(), st))
        with _timed("grad", dev):
            _native.check(L.dfe_grad(nm.handle, lam.data_ptr(), u[b].data_ptr(), None, gmode, gk_b[b].data_ptr(),
                                     gf[b].data_ptr() if gf is not None else None, gws.data_ptr(), gws.numel(), st))
    opts["last_pcg_adjoint"] = iters
    if shared:
        gk.copy_(gk_b.sum(dim=0).reshape(gk.shape))   # torch.sum on CUDA is deterministic (no atomics)
    else:
        gk.copy_(gk_b.reshape(gk.shape))


def assemble_sparse(mesh: FEMesh, kappa, f: torch.Tensor, device=None):
    """``(K, F)``: the stiffness matrix of ``mesh`` as a ``torch.sparse_csr_tensor`` on the GPU and the load vector, BEFORE
    the Dirichlet elimination — the arrays the reference builds densely in ``solver.py:82-96`` / ``:112-145`` (its roadmap
    item "sparse matrix assembly", README.md:139-143 upstream).  For P1 meshes the values and the pattern are bit-identical
    to the reference's dense ``K`` / ``F`` (rows and columns ascending; structural entries that happen to be 0 are kept);
    ``kappa`` is a number, a 0-dim / 1-element tensor or an ``(n_elements,)`` field.  No gradients flow through this call."""
    if mesh.dim not in (1, 2):
        raise NotImplementedError("Only 1D and 2D supported")
    if not torch.cuda.is_available():
        raise RuntimeError("assemble_sparse (difffe_physics_lab_b200) runs on CUDA only; there is deliberately no CPU fallback")
    dev = torch.device(device) if device is not None else (f.device if f.is_cuda else torch.device("cuda", torch.cuda.current_device()))
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    L = _native.lib()
    nm = mesh._native(dev.index)
    I = nm.info
    kap = torch.as_tensor(kappa, dtype=torch.float64).detach().reshape(-1).to(dev).contiguous()
    if kap.numel() not in (1, mesh.n_elements):
        raise ValueError(f"kappa must have 1 or n_elements={mesh.n_elements} entries, got {kap.numel()}")
    mode = _native.KAPPA_SCALAR if kap.numel() == 1 else _native.KAPPA_PER_ELEMENT
    if f.shape != (mesh.n_nodes,):
        raise ValueError(f"f must have shape ({mesh.n_nodes},), got {tuple(f.shape)}")
    fd = f.detach().to(device=dev, dtype=torch.float64).contiguous()
    with torch.cuda.device(dev):
        vals = torch.empty(max(I.nnz_full, 1), dtype=torch.float64, device=dev)
        F = torch.empty(I.n_nodes, dtype=torch.float64, device=dev)
        _native.check(L.dfe_assemble(nm.handle, kap.data_ptr(), mode, fd.data_ptr(), vals.data_ptr(), F.data_ptr(), _stream(dev)))
        rp, col = nm.csr(0)
        K = torch.sparse_csr_tensor(torch.from_numpy(rp).to(dev), torch.from_numpy(col).to(dev), vals[:I.nnz_full],
                                    size=(I.n_nodes, I.n_nodes))
    return K, F


# ----------------------------------------------------------------------------- module
class DifferentiableFESolver(nn.Module):
    """Assemble and solve the P1 FEM system for ``mesh`` and a nodal forcing ``f``.

    Parameters
    ----------
    mesh : FEMesh
    kappa : float or torch.Tensor
        Diffusion coefficient; see the module docstring for the accepted tensor shapes.
    pcg_tol, pcg_maxit : keyword-only
        2D / general path: Jacobi-PCG stops at recursive ``||r|| <= pcg_tol ||rhs||`` (default 1e-13,
        which keeps ``u`` and the gradients within 1e-9 of the reference's dense solve).
    n_refine : keyword-only
        1D fused path: number of Neumann sweeps after the structured solve (-1 = automatic).
    solver2d, mg_nu : keyword-only
        2D single-mesh solves: ``"auto"`` uses CG preconditioned by a multigrid V(mg_nu, mg_nu) cycle on meshes with
        the structure of ``FEMesh.rectangle()`` and Jacobi-PCG elsewhere; ``"jacobi"`` / ``"mg"`` force one.
    out_device : keyword-only
        where ``u`` is returned (default: the device of ``f``).
    """

    def __init__(self, mesh: FEMesh, kappa: float = 1.0, *, pcg_tol: float = 1e-13,
                 pcg_maxit: Optional[int] = None, n_refine: int = -1, out_device=None, solver2d: str = "auto",
                 mg_nu: int = 2):
        super().__init__()
        self.mesh = mesh
        # Same rule as the reference (solver.py:35-39): numbers become 0-dim float64 tensors, tensors are
        # converted with .to(float64) — which keeps the autograd graph and, for a float64 nn.Parameter,
        # returns the same object so that nn.Module registers it (SURVEY §5 checkpoint quirk).
        if isinstance(kappa, (int, float)):
            self._kappa = torch.tensor(kappa, dtype=torch.float64)
        else:
            self._kappa = kappa.to(dtype=torch.float64)
        self._opts = {"pcg_tol": pcg_tol, "pcg_maxit": pcg_maxit, "n_refine": n_refine, "solver2d": solver2d, "mg_nu": mg_nu}
        self._out_device = None if out_device is None else torch.device(out_device)

    @property
    def kappa(self) -> torch.Tensor:
        return self._kappa

    @property
    def last_pcg(self):
        """[(iterations, relative residual)] of the most recent general-path forward (diagnostics)."""
        return self._opts.get("last_pcg")

    def _resolve(self, f: torch.Tensor):
        mesh = self.mesh
        if mesh.dim not in (1, 2):
            raise NotImplementedError("Only 1D and 2D supported")
        if not torch.cuda.is_available():
            raise RuntimeError(
                "DifferentiableFESolver (difffe_physics_lab_b200) runs on CUDA only and no device is visible; "
                "there is deliberately no CPU fallback")
        batched = f.dim() == 2
        if f.dim() not in (1, 2) or f.shape[-1] != mesh.n_nodes:
            raise ValueError(f"f must have shape (n_nodes,) or (B, n_nodes) with n_nodes={mesh.n_nodes}, got {tuple(f.shape)}")
        dev = f.device if f.is_cuda else (self._out_device if self._out_device is not None and self._out_device.type == "cuda"
                                          else torch.device("cuda", torch.cuda.current_device()))
        if dev.index is None:
            dev = torch.device("cuda", torch.cuda.current_device())
        B = f.shape[0] if batched else 1
        mode = _kappa_mode(self.kappa, B, mesh.n_elements, batched)
        return dev, batched, B, mode

    def forward(self, f: torch.Tensor) -> torch.Tensor:
        """Solve ``-div(kappa grad u) = f``; ``f`` is ``(n_nodes,)`` or ``(B, n_nodes)``, any float dtype.

        ``u`` comes back on ``f``'s device (CPU in -> CPU out, as the reference's callers expect) unless the module was
        built with ``out_device="cuda"``, which keeps the solution of a host-resident ``f`` on the GPU."""
        mesh = self.mesh
        dev, batched, B, mode = self._resolve(f)
        out_dev = self._out_device if self._out_device is not None else f.device
        if out_dev.type == "cuda" and out_dev.index is None:
            out_dev = dev
        # dtype moves and reshapes are ordinary differentiable torch ops; the Function sees (B, n) float64 rows and
        # does the host <-> device transfers itself (streamed for large batches)
        f2 = f.to(dtype=torch.float64).reshape(B, mesh.n_nodes).contiguous()
        k_dev = self.kappa.to(device=dev).contiguous()
        u = _FESolve.apply(f2, k_dev, mesh, mode, self._opts, dev, out_dev)
        if not batched:
            u = u.reshape(mesh.n_nodes)
        return u

    def misfit(self, f: torch.Tensor, u_data: torch.Tensor, out2: Optional[torch.Tensor] = None,
               weight: float = 1.0) -> torch.Tensor:
        """Data-misfit loss ``weight * sum_b mean_i (u_b(f_b, kappa) - u_data_b)^2`` of the solution against ``u_data``
        (for one sample: the reference demo's ``((solver(f) - u_data) ** 2).mean()``,
        examples/poisson_1d_demo.py:104-110), differentiable w.r.t. ``kappa`` and ``f``.

        On the fused 1-D path (chain mesh, scalar or per-sample kappa, CUDA inputs) this is two kernels: the forward
        solve and a misfit adjoint that forms the upstream gradient on the fly — gbar and the squared differences never
        touch HBM.  Elsewhere it is evaluated as ``((self(f) - u_data) ** 2).sum() / n_nodes``."""
        mesh = self.mesh
        dev, batched, B, mode = self._resolve(f)
        n = mesh.n_nodes
        fast = (f.is_cuda and u_data.is_cuda and mode in (_native.KAPPA_SCALAR, _native.KAPPA_PER_SAMPLE)
                and bool(mesh._native(dev.index).info.chain1d) and n <= 163840
                and self._opts["n_refine"] in (-1, 1) and f.dtype == torch.float64 and u_data.dtype == torch.float64)
        if fast:
            f2 = f.reshape(B, n).contiguous()
            d2 = u_data.detach().reshape(B, n).contiguous()
            fast = f2.data_ptr() % 16 == 0 and d2.data_ptr() % 16 == 0
        if fast:
            k_dev = self.kappa.to(device=dev).contiguous()
            try:
                return _FEMisfit.apply(f2, k_dev, d2, mesh, mode, self._opts, out2, float(weight))
            except NotImplementedError:      # the pipelined kernel does not take this call (DFE_ERR_UNSUPPORTED)
                pass
        u = self(f)
        loss = ((u - u_data.to(u.device)) ** 2).sum() * (float(weight) / n)
        if out2 is not None:
            raise NotImplementedError("misfit(out2=...) needs the fused misfit adjoint (chain mesh, shared scalar kappa)")
        return loss
