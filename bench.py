#!/usr/bin/env python
"""bench.py — FEM fwd+adjoint solves/s on B200 (BASELINE.json metric), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c2|c5a]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (N=1, default) = BASELINE.json configs[1]: 1-D Poisson, FEMesh.line(n_elements=100000), batch of
4096 samples with random forcing f ~ U(0,1) and per-sample kappa ~ logU[0.5,2], forward + adjoint
(upstream gradient gbar ~ N(0,1), dL/df and dL/dkappa both produced).  One "step" = one fwd+adjoint pass
over the batch; with N GPUs every rank holds its own 4096 samples (weak scaling, no data-path collective:
the samples are independent systems on a replicated mesh).

  value      solves/s over all ranks, inputs resident in HBM, through the public API
             (DifferentiableFESolver(...)(f); u.backward(gbar)), CUDA events, max over ranks
  e2e        same metric with HOST inputs: every step copies f and kappa from pinned host memory and
             reads dL/dkappa back (copies inside the timed region, sub-batches pipelined on two streams)
  roofline   dominant kernel (k_solve1d<BWD>): algorithmic bytes per launch / its mean CUDA-event
             duration inside the timed region, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  oracle/fem_port.c (C restatement, OpenMP over samples) on a bounded sample, rank 0, N=1
  --impl reference  times that CPU port alone (the reference is pure Python and cannot run n=1e5:
             dense K would be 80 GB — BASELINE.md §2)
  --dump-outputs DIR  after the timed steps, write what the last timed step returned to its caller as DIR/<name>.npy
             (float64, at most 64 MB in all; see dump_outputs).  The inputs are seeded, so two builds run with the same
             arguments can be compared file by file.

Inputs per array are 3.28 GB (>> 126 MB L2), so no L2 flush is needed between iterations.
bench.py writes nothing into the source tree (it may be read-only): it loads the library build() compiled.
"""
from __future__ import annotations

import argparse
import json
import os
import pathlib
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True            # no __pycache__ for the project modules imported below: the tree stays untouched

WORKLOADS = {
    # name: (n_elements, batch per rank, kappa layout, scaling)
    "c2": dict(n_elements=100000, batch=4096, kappa="per_sample", scaling="weak",
               desc="1D Poisson batch of 4096 random forcing/kappa samples, n_elements=100000, fwd+adjoint"),
    "c2e": dict(n_elements=100000, batch=4096, kappa="per_sample_element", scaling="weak",
                desc="1D Poisson batch of 4096 samples, n_elements=100000, per-sample PER-ELEMENT kappa (4096, 100000) ~ logU[0.1,10], "
                     "fwd+adjoint with dL/df and dL/dkappa_e (SURVEY 8(d) C2 variant, 64 B/node accounting)"),
    "c5a": dict(n_elements=16384, batch=65536, kappa="shared", scaling="strong",
                desc="kappa inverse-problem sweep: 65536 1D solves (n_elements=16384), shared kappa, NCCL grad allreduce"),
    # 2-D configs (one mesh per GPU; N > 1 = replicas only).  Not the default bench line.
    "c3": dict(nx=128, kappa="scalar", scaling="weak",
               desc="2D unit-square P1 triangles 128x128 (16641 nodes), f=1, kappa=1, fwd+adjoint"),
    "c5b": dict(nx=32, batch=65536, kappa="shared", scaling="strong", small=True,
                desc="kappa inverse-problem sweep: 65536 2D solves on rectangle(32,32) (961 DOF), shared kappa, NCCL grad allreduce"),
    "c4": dict(nx=1024, kappa="per_element", scaling="weak",
               desc="2D heterogeneous per-element kappa 1024x1024 mesh, kappa_e ~ logU[1e-3,1], f=1, fwd+adjoint of sum(u)"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=None, help="override samples per rank (debugging; noted in config)")
    ap.add_argument("--n-elements", type=int, default=None, help="override mesh size (debugging; noted in config)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 0:
        ap.error("--warmup must not be negative")
    return args


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def measured_traffic(workload, kernel):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of `kernel` in the `ncu --set full` capture of
    `workload`, from the latest summary under profiles/ (tools/make_profiles.py; keys are "<workload>:<kernel name>")."""
    best = None
    for fp in sorted((ROOT / "profiles").glob("r*_traffic.json")):
        try:
            for k, v in json.loads(fp.read_text()).items():
                k = k.replace(" ", "")
                if kernel in k and (k.startswith(workload + ":") or ":" not in k.split("<")[0].split("(")[0]):
                    best = float(v)
        except Exception:
            pass
    return best


# ------------------------------------------------------------------------------- CPU baseline (oracle port)
def cpu_port_rate(n_elements, seconds_target, steps=1, warmup=0, seed=0):
    """Time oracle/fem_port.c (fwd + adjoint, all host threads) on a bounded sample of the workload.
    Returns (solves_per_s, cores, sample_description, ms_per_step)."""
    from oracle import port as P
    from oracle import oracle as O

    # every host core this process may run on — NOT omp_get_max_threads(): torch.distributed.run exports
    # OMP_NUM_THREADS=1 to its workers, which would silently turn the baseline into a single-thread run
    cores = len(os.sched_getaffinity(0))
    nodes, _, bc = O.line_mesh(n_elements)
    x = nodes[:, 0]
    nn = n_elements + 1
    rng = np.random.default_rng(seed)
    S = max(cores, 8)
    f = rng.uniform(0, 1, (S, nn))
    gbar = rng.standard_normal((S, nn))
    kap = np.exp(rng.uniform(np.log(0.5), np.log(2.0), S))
    t0 = time.perf_counter()
    P.solve1d_batch(x, bc, f, kap, gbar, nthreads=cores)       # calibration pass (also warms the pages)
    t_cal = time.perf_counter() - t0
    reps = max(1, int(seconds_target / max(t_cal, 1e-6)))
    for _ in range(warmup):
        P.solve1d_batch(x, bc, f, kap, gbar, nthreads=cores)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        for _ in range(reps):
            P.solve1d_batch(x, bc, f, kap, gbar, nthreads=cores)
        times.append(time.perf_counter() - t0)
    per_step = float(np.mean(times))
    rate = S * reps / per_step
    sample = (f"{S * reps} fwd+adjoint solves per step ({S} distinct samples x {reps} passes) of the n_elements="
              f"{n_elements} workload, OpenMP over samples, {cores} threads")
    return rate, cores, sample, per_step * 1e3



def cpu_rate_2d(mesh, kappa_np, f_np, iters_step, seconds_target=10.0):
    """CPU baseline of one 2-D fwd+adjoint step: the oracle's vectorised assembly + Dirichlet elimination (numpy, one
    thread) and the port's Jacobi-PCG (OpenMP, all host threads).  The PCG is timed on a BOUNDED number of iterations
    and scaled to the `iters_step` iterations (forward + adjoint) the same Jacobi-PCG needs on this system."""
    from oracle import oracle as O
    from oracle import port as P

    cores = len(os.sched_getaffinity(0))
    nodes, el, bc = mesh.nodes.numpy(), mesh.elements.numpy(), mesh.dirichlet_nodes
    t0 = time.perf_counter()
    rp, col, vals, F = O.assemble_csr(nodes, el, kappa_np, f_np)
    _, frp, fcol, fvals, Ff = O.apply_bc(rp, col, vals, F, bc)
    t_asm = time.perf_counter() - t0
    t0 = time.perf_counter()
    P.pcg_csr(frp, fcol, fvals, Ff, tol=0.0, maxit=20, nthreads=cores)
    t_it = (time.perf_counter() - t0) / 20
    n_run = int(max(20, min(4 * iters_step, seconds_target / max(t_it, 1e-9))))
    t0 = time.perf_counter()
    P.pcg_csr(frp, fcol, fvals, Ff, tol=0.0, maxit=n_run, nthreads=cores)
    t_it = (time.perf_counter() - t0) / n_run
    t_step = t_asm + iters_step * t_it
    return {"value": 1.0 / t_step, "unit": "solves/s", "cores": cores, "kind": "port",
            "sample": f"assembly + elimination once ({t_asm:.2f} s, numpy, 1 thread) + {n_run} timed Jacobi-PCG iterations "
                      f"({t_it * 1e3:.3f} ms each, OpenMP, {cores} threads) scaled to the {iters_step} iterations of one "
                      f"forward + adjoint solve at tol 1e-13 (count taken from the same Jacobi-PCG on the GPU)"}


def cpu_rate_2d_batch(mesh, kappa, S, seed=0):
    """CPU baseline of config 5b on S samples: shared matrix assembled once (oracle, numpy), per-sample load vectors
    (vectorised numpy), then forward and adjoint Jacobi-PCG solves of every sample (port, OpenMP over the samples)."""
    from oracle import oracle as O
    from oracle import port as P

    cores = len(os.sched_getaffinity(0))
    nodes, el, bc = mesh.nodes.numpy(), mesh.elements.numpy(), mesh.dirichlet_nodes
    nn = len(nodes)
    rng = np.random.default_rng(seed)
    f = rng.uniform(0.5, 1.5, (S, nn))
    gbar = rng.standard_normal((S, nn))
    rp, col, vals, F0 = O.assemble_csr(nodes, el, kappa, f[0])
    free, frp, fcol, fvals, Ff0 = O.apply_bc(rp, col, vals, F0, bc)
    lift = F0[free] - Ff0                                   # sample independent
    x, y = nodes[:, 0], nodes[:, 1]
    i, j, k = el[:, 0], el[:, 1], el[:, 2]
    area = 0.5 * np.abs((x[j] - x[i]) * (y[k] - y[i]) - (x[k] - x[i]) * (y[j] - y[i]))
    t0 = time.perf_counter()
    term = (area / 3.0) * ((f[:, i] + f[:, j] + f[:, k]) / 3.0)            # (S, n_el), solver.py:143-145
    F = np.zeros((S, nn))
    for loc in (i, j, k):
        for b in range(S):
            F[b] += np.bincount(loc, weights=term[b], minlength=nn)
    rhs = F[:, free] - lift
    u_free, _ = P.pcg_csr_batch(frp, fcol, fvals, rhs, nthreads=cores)
    lam, _ = P.pcg_csr_batch(frp, fcol, fvals, gbar[:, free], nthreads=cores)
    t = time.perf_counter() - t0
    return {"value": S / t, "unit": "solves/s", "cores": cores, "kind": "port",
            "sample": f"{S} samples of the 65536: load vectors (numpy) + forward and adjoint Jacobi-PCG per sample "
                      f"(oracle/fem_port.c, OpenMP over samples, {cores} threads, tol 1e-13); matrix assembled once; "
                      f"gradient evaluation not included"}


def run_reference(args):
    """--impl reference: the CPU implementation of the path on the host cores (oracle port)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = dict(WORKLOADS[args.workload])
    n_el = args.n_elements or w["n_elements"]
    subprocess.run(["make", "-s", "-C", str(ROOT / "oracle")], check=True)
    rate, cores, sample, ms = cpu_port_rate(n_el, seconds_target=4.0, steps=args.steps, warmup=args.warmup)
    line = {
        "impl": "reference", "metric": "fem_fwd_adjoint_solves_per_s", "value": rate, "unit": "solves/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": w["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "dof_per_s": rate * (n_el - 1),
        "config": {"workload": w["desc"], "n_elements": n_el, "note": "CPU port of the reference path (oracle/fem_port.c); "
                   "the pure-Python reference cannot run this size (dense K = 80 GB, BASELINE.md §2)"},
        "cpu_baseline": {"value": rate, "unit": "solves/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,utilization.gpu,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.tmp = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=self.tmp, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.tmp.flush()
        sm, sm_load, mx, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in open(self.tmp.name):
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 8 or not parts[0].isdigit() or int(parts[0]) != self.gpu_index:
                continue
            try:
                clk, cmax = float(parts[1]), float(parts[2])
            except ValueError:
                continue
            sm.append(clk)
            mx.append(cmax)
            try:
                if float(parts[3]) >= 50.0:
                    sm_load.append(clk)
            except ValueError:
                pass
            for nm, v in zip(names, parts[4:8]):
                if v == "Active":
                    reasons.add(nm)
        os.unlink(self.tmp.name)
        if sm:
            use = sm_load or sm
            out.update(sm_mhz=float(np.median(use)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons),
                       samples=len(sm), samples_under_load=len(sm_load))
        return out


def bind_to_gpu_numa_node(local_rank):
    """Pin this rank (and therefore the pinned host buffers it first-touches) to the CPUs of its GPU's NUMA node:
    with one rank per GPU the host->device copies of the e2e leg otherwise cross the socket interconnect.  Best
    effort (pynvml + sysfs); returns a short description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local_rank)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:          # nvml pads the PCI domain to 8 hex digits, sysfs uses 4
            bus = bus[4:]
        base = pathlib.Path("/sys/bus/pci/devices") / bus
        node = int((base / "numa_node").read_text().strip())
        cpus = set()
        for part in (base / "local_cpulist").read_text().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"numa node {node}, {len(cpus)} cpus"
    except Exception as exc:  # no NUMA information: leave the default placement
        return f"unbound ({type(exc).__name__})"
    return "unbound"


# ------------------------------------------------------------------------------- GPU arm
def parity_block(mesh, rows, f, kappa, gbar, u, gf, gk, shared_kappa, per_elem=False):
    """Max relative error of sampled rows of the TIMED output against the exact oracle (oracle/oracle.py: the same
    float64 system solved in 50-digit arithmetic).  Checker use of oracle/ — the rows were produced by the kernels."""
    from oracle import oracle as O

    nodes, el, bc = mesh.nodes.numpy(), mesh.elements.numpy(), mesh.dirichlet_nodes
    worst = {"u": 0.0, "gf": 0.0, "gkappa": 0.0}
    for b in rows:
        kb = kappa[b].cpu().numpy() if per_elem else float(kappa.reshape(-1)[0 if shared_kappa else b])
        uo = O.forward(nodes, el, bc, kb, f[b].cpu().numpy())
        gko, gfo, _ = O.adjoint_and_grads(nodes, el, bc, kb, uo, gbar[b].cpu().numpy())
        worst["u"] = max(worst["u"], float(np.abs(u[b].cpu().numpy() - uo).max() / np.abs(uo).max()))
        if gf is not None:
            worst["gf"] = max(worst["gf"], float(np.abs(gf[b].cpu().numpy() - gfo).max() / np.abs(gfo).max()))
        if per_elem:      # SURVEY appendix A: dL/dkappa_e relative to sum_e |dL/dkappa_e| (L1), the entry-wise maximum beside it
            gkb = gk[b].cpu().numpy()
            worst["gkappa"] = max(worst["gkappa"], float(np.abs(gkb - gko).sum() / np.abs(gko).sum()))
            worst["gkappa_entry"] = max(worst.get("gkappa_entry", 0.0), float(np.abs(gkb - gko).max() / np.abs(gko).max()))
        elif not shared_kappa:
            worst["gkappa"] = max(worst["gkappa"], float(abs(float(gk.reshape(-1)[b]) - gko.sum()) / np.abs(gko).sum()))
    return {"rows": [int(r) for r in rows], "max_rel": max(worst["u"], worst["gf"], worst["gkappa"]), "max_rel_u": worst["u"],
            "max_rel_gf": worst["gf"], "max_rel_gkappa": worst["gkappa"] if not shared_kappa else None,
            "max_rel_gkappa_entrywise": worst.get("gkappa_entry"), "tol": 1e-12,
            "oracle": "oracle/oracle.py exact (50-digit Thomas on the bit-exact float64 system)",
            "note": "rows of the last timed step, chosen from the first, a middle and the last pipeline iteration"}


def parity_block_2d(mesh, nm, kappa, f, u, gk):
    """Proof that the timed 2-D solve did the work, without a CPU solve of the 1e6-unknown system: the TRUE relative residual
    of the assembled system (dfe_assemble values on the handle's CSR pattern, sparse mat-vec in torch on the device) and the
    Euler identity of the gradient (K is linear in kappa and the boundary values are zero, so for J = sum(u):
    sum_e kappa_e dJ/dkappa_e = -J).  The oracle comparison at this size is tests/test_gpu_mg.py."""
    import torch
    import ctypes as C
    from difffe_physics_lab_b200 import _native
    L = _native.lib()
    dev = u.device
    I = nm.info
    kf = kappa.detach().reshape(-1).contiguous()
    mode = _native.KAPPA_SCALAR if kf.numel() == 1 else _native.KAPPA_PER_ELEMENT
    vals = torch.empty(I.nnz_full, dtype=torch.float64, device=dev)
    F = torch.empty(I.n_nodes, dtype=torch.float64, device=dev)
    _native.check(L.dfe_assemble(nm.handle, kf.data_ptr(), mode, f.data_ptr(), vals.data_ptr(), F.data_ptr(),
                                 torch.cuda.current_stream().cuda_stream))
    rp, col = nm.csr(0)
    K = torch.sparse_csr_tensor(torch.from_numpy(rp).to(dev), torch.from_numpy(col).to(dev), vals, size=(I.n_nodes, I.n_nodes))
    free = torch.from_numpy(nm.free_nodes()).to(dev)
    r = (F - K @ u.detach())[free]
    res = float(r.norm() / F[free].norm())
    J = float(u.detach().sum())
    euler = abs(float((kappa.detach() * gk).sum()) + J) / abs(J)
    return {"true_residual_rel": res, "euler_identity_rel": euler,
            "what": "||F - K u||_free / ||F||_free with K, F from dfe_assemble (bit-exact with the reference's dense arrays) and the "
                    "timed u; |sum_e kappa_e dJ/dkappa_e + J| / |J| for J = sum(u) with the timed gradient"}


def parity_block_small2d(mesh, rows, f, kappa, gbar, u, gf):
    """Rows of the timed config-5b output against the oracle (sparse LU + refinement): max relative error of u and dL/df."""
    from oracle import oracle as O
    nodes, el, bc = mesh.nodes.numpy(), mesh.elements.numpy(), mesh.dirichlet_nodes
    worst_u = worst_gf = 0.0
    for b in rows:
        fb, gb = f[b].detach().cpu().numpy(), gbar[b].cpu().numpy()
        uo = O.forward(nodes, el, bc, float(kappa), fb)
        _, gfo, _ = O.adjoint_and_grads(nodes, el, bc, float(kappa), uo, gb)
        worst_u = max(worst_u, float(np.abs(u[b].detach().cpu().numpy() - uo).max() / np.abs(uo).max()))
        worst_gf = max(worst_gf, float(np.abs(gf[b].cpu().numpy() - gfo).max() / np.abs(gfo).max()))
    return {"max_rel": max(worst_u, worst_gf), "u_max_rel": worst_u, "gf_max_rel": worst_gf, "rows": [int(b) for b in rows],
            "tolerance": 1e-9, "oracle": "oracle/oracle.py (sparse LU + refinement of the same float64 system)"}


DUMP_BYTES = 64 * 10 ** 6                   # --dump-outputs: all files together, .npy headers included


def dump_outputs(out_dir, whole, batched=None):
    """--dump-outputs: write the arrays the last timed step returned to its caller as <out_dir>/<name>.npy (float64).

    `whole` arrays are written entire.  `batched` arrays hold one row per sample; when they do not fit the budget left by
    `whole`, every one of them keeps the same rows: as many as fit, drawn with a fixed seed and sorted ascending.  The
    sample depends on the shapes alone, so runs with the same arguments write the same rows.  Only rank 0 dumps."""
    import torch

    out = {k: v.detach().double().cpu().numpy() for k, v in whole.items()}
    if batched:
        B = next(iter(batched.values())).shape[0]
        room = DUMP_BYTES - sum(a.nbytes for a in out.values()) - 4096 * (len(out) + len(batched))   # 4 KiB per header
        n = min(B, room // sum(8 * (v.numel() // B) for v in batched.values()))
        rows = np.sort(np.random.default_rng(0).choice(B, n, replace=False))
        idx = torch.from_numpy(rows).to(next(iter(batched.values())).device)
        out.update({k: v.detach()[idx].double().cpu().numpy() for k, v in batched.items()})
    d = pathlib.Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for k, a in out.items():
        np.save(d / f"{k}.npy", a)


def time_sweep(args, rank, world, dev, n_el, B_total, steps, warmup, dump_dir=None):
    """BASELINE config 5a as SURVEY §8(d) defines it: 65 536 samples on line(16384), shared kappa, sharded over the
    ranks (strong scaling); per step  forward -> fused misfit adjoint (gbar = 2 (u - u_data) / n formed in the kernel,
    [sum dL/dkappa, sum loss] written into the persistent reduction buffer) -> ONE NCCL all-reduce of 16 bytes -> Adam
    step replicated on every rank (examples/poisson_1d_demo.py:104-110, batched).  With `dump_dir`, the last step's
    loss, dL/dkappa and updated kappa go there (dump_outputs)."""
    import torch
    import torch.distributed as dist

    from difffe_physics_lab_b200 import DifferentiableFESolver, FEMesh
    from difffe_physics_lab_b200.distributed import MisfitSweep, shard_bounds
    from difffe_physics_lab_b200.solver import KernelTimer

    lo, hi = shard_bounds(B_total, rank, world)
    B = hi - lo
    nn = n_el + 1
    mesh = FEMesh.line(n_el)
    gen = torch.Generator(device=dev).manual_seed(4321 + rank)
    f = torch.rand((B, nn), dtype=torch.float64, device=dev, generator=gen) + 0.5
    with torch.no_grad():
        u_data = DifferentiableFESolver(mesh, kappa=torch.tensor(2.0, dtype=torch.float64, device=dev))(f)
    kappa = torch.tensor(1.0, dtype=torch.float64, device=dev, requires_grad=True)
    try:                                         # one fused kernel per Adam step instead of four
        opt = torch.optim.Adam([kappa], lr=0.05, fused=True)
    except Exception:
        opt = torch.optim.Adam([kappa], lr=0.05, capturable=True)
    sweep = MisfitSweep(mesh, f, u_data, B_total)

    def step():
        loss, grad = sweep.step(kappa)
        kappa.grad = grad.detach().reshape(())
        opt.step()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    l_first = float(step())                     # (a host read: only here, outside the timed region)
    for _ in range(max(warmup, 3) - 1):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with KernelTimer() as kt:
        e0.record()
        for _ in range(steps):
            last = step()
        e1.record()
        barrier()
    ms_total = e0.elapsed_time(e1)
    ksum = kt.summary()
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, {"loss": last, "grad_kappa": kappa.grad, "kappa": kappa})
    if world > 1:
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t[0])
    ms_step = ms_total / steps
    peak, _ = measured_peak()
    kern = {k: {"calls": c, "ms_per_launch": m / c} for k, (c, m) in ksum.items()}
    for name, bpn in (("solve1d_fwd", 16), ("solve1d_bwd_misfit", 16)):     # read f, write u / read u_data, read u
        if name in kern:
            kern[name]["algorithmic_bytes"] = bpn * nn * B
            kern[name]["achieved_gbs"] = bpn * nn * B / (kern[name]["ms_per_launch"] * 1e-3) / 1e9
            kern[name]["frac"] = kern[name]["achieved_gbs"] / peak
    out = {"workload": WORKLOADS["c5a"]["desc"], "value": B_total * steps / (ms_total * 1e-3), "unit": "solves/s",
           "ms_per_step": ms_step, "scaling": "strong", "n_gpus": world, "global_batch": B_total, "batch_per_gpu": B,
           "n_elements": n_el, "steps": steps,
           "step": "fwd + fused misfit adjoint (16 + 16 B/node) -> all-reduce [dL/dkappa, loss] -> Adam(kappa)",
           "collective": (f"NCCL all_reduce of 2 f64 per step on the compute stream, buffer "
                          f"{'registered with NCCL (ncclMemAlloc pool)' if sweep.registered else 'persistent, unregistered'}"
                          if world > 1 else "none (1 rank)"),
           "step_frac_of_peak": 32 * nn * B / (ms_step * 1e-3) / 1e9 / peak,
           "kernels": kern, "gpu_launches": kt.launches,
           "loss_first_step": l_first, "loss_last_step": float(last), "kappa_after": float(kappa.detach())}
    del sweep, f, u_data
    torch.cuda.empty_cache()
    return out


def run_b200(args):
    import torch
    import torch.distributed as dist

    from difffe_physics_lab_b200 import DifferentiableFESolver, FEMesh
    from difffe_physics_lab_b200 import _native
    from difffe_physics_lab_b200.solver import KernelTimer

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 arm has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    host_binding = bind_to_gpu_numa_node(local_rank) if world > 1 else "single rank: default placement"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    if _native.needs_build():
        print("bench.py: libdfe_b200.so is older than its sources; run __graft_entry__.build() to rebuild it", file=sys.stderr)
    _native.lib()

    w = dict(WORKLOADS[args.workload])
    if w.get("small"):
        return run_b200_small2d(args, w, rank, local_rank, world, dev)
    if "nx" in w:
        return run_b200_2d(args, w, rank, local_rank, world, dev)
    if args.workload == "c5a":
        return run_b200_sweep(args, w, rank, local_rank, world, dev)
    n_el = args.n_elements or w["n_elements"]
    B = args.batch or w["batch"]
    nn = n_el + 1

    mesh = FEMesh.line(n_el)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    f = torch.rand((B, nn), dtype=torch.float64, device=dev, generator=gen)
    per_elem = w["kappa"] == "per_sample_element"
    if per_elem:
        kappa = torch.exp(torch.empty((B, n_el), dtype=torch.float64, device=dev).uniform_(float(np.log(0.1)), float(np.log(10.0)), generator=gen))
        args.no_e2e = args.no_sweep = args.no_cpu = True   # the variant line carries the device-resident numbers only
    else:
        kappa = torch.exp(torch.empty((B, 1), dtype=torch.float64, device=dev).uniform_(float(np.log(0.5)), float(np.log(2.0)), generator=gen))
    gbar = torch.randn((B, nn), dtype=torch.float64, device=dev, generator=gen)
    keep = {}

    def step_resident():
        fr = f.requires_grad_(True)
        fr.grad = None
        kr = kappa.detach().requires_grad_(True)
        u = DifferentiableFESolver(mesh, kappa=kr)(fr)
        u.backward(gbar)
        keep["u"], keep["gk"] = u, kr.grad
        return kr.grad

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident timing (the clock sampler runs from the warm-up to the end of the e2e
    # region: all of it is under load, and nvidia-smi needs a few hundred ms to deliver its first sample)
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        step_resident()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with KernelTimer() as kt:
        e0.record()
        for _ in range(args.steps):
            step_resident()
        e1.record()
        barrier()
    ms_total = e0.elapsed_time(e1)
    ksum = kt.summary()
    launches = kt.launches
    if world > 1:
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t[0])
    ms_step = ms_total / args.steps
    value = B * world * args.steps / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:
        whole, batched = {}, {"u": keep["u"], "grad_f": f.grad}
        (batched if per_elem else whole)["grad_kappa"] = keep["gk"]
        dump_outputs(args.dump_outputs, whole, batched)

    # ---------------- parity of the timed output (rank 0): rows from the first / a middle / the last pipeline iteration
    parity = None
    if rank == 0 and not args.no_parity:
        try:
            rows = sorted({0, B // 2 + 1, B - 1})
            parity = parity_block(mesh, rows, f.detach(), kappa, gbar, keep["u"].detach(), f.grad, keep["gk"], False, per_elem)
        except Exception as exc:
            parity = {"max_rel": None, "error": f"{type(exc).__name__}: {exc}"}

    # ---------------- roofline of the dominant kernel (algorithmic bytes, SURVEY §8d: fwd 16N, adjoint 24N with gf)
    peak, peak_src = measured_peak()
    kern = {}
    # per-element kappa adds the kappa row to both directions and the dL/dkappa_e row to the adjoint (24 / 40 B per node)
    for name, bytes_per_node in (("solve1d_fwd", 24 if per_elem else 16), ("solve1d_bwd", 40 if per_elem else 24)):
        if name in ksum:
            calls, ms = ksum[name]
            alg = bytes_per_node * nn * B
            kern[name] = {"calls": calls, "ms_per_launch": ms / calls, "algorithmic_bytes": alg,
                          "achieved_gbs": alg / (ms / calls * 1e-3) / 1e9, "frac": alg / (ms / calls * 1e-3) / 1e9 / peak}
    dom = max(kern, key=lambda k: kern[k]["ms_per_launch"] * kern[k]["calls"]) if kern else None
    roofline = None
    if dom:
        knames = {"solve1d_fwd": "dfe_solve1d_fwd = k1d_pipe<fwd> (+ k1d_pipe_ck, k1d_pipe_poison, exchange-buffer memset)",
                  "solve1d_bwd": "dfe_solve1d_bwd = k1d_pipe<bwd> (+ k1d_pipe_ck, k1d_pipe_gk, k1d_pipe_poison, exchange-buffer memset)"}
        if per_elem:
            knames = {"solve1d_fwd": "dfe_solve1d_fwd = k1d_pass1<fwd> + fold + k1d_pass2<fwd> (two-pass split kernels: per-element kappa)",
                      "solve1d_bwd": "dfe_solve1d_bwd = k1d_pass1<bwd> + fold + k1d_pass2<bwd> (two-pass split kernels: per-element kappa)"}
        roofline = {"bound": "hbm", "kernel": knames[dom],
                    "achieved": kern[dom]["achieved_gbs"], "peak": peak, "unit": "GB/s",
                    "frac": kern[dom]["achieved_gbs"] / peak,
                    # <BWD, R, W, LB, LC, SK, MF, OUT, PF> of the two kernels this workload launches
                    "traffic": (measured_traffic("c2", "k1d_pipe<0,9,12,2,2,0,0,1,1>" if dom == "solve1d_fwd" else "k1d_pipe<1,11,8,2,2,0,0,1,1>")
                                if args.workload == "c2" and not args.batch and not args.n_elements else None),
                    "traffic_source": "REPLAYED from the tracked file profiles/r*_traffic.json (dram__bytes_read.sum + dram__bytes_write.sum of "
                                      "one earlier `ncu --set full` capture of this kernel on this workload) — not measured in this run",
                    "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": kern[dom]["algorithmic_bytes"],
                    "ms_per_launch": kern[dom]["ms_per_launch"], "kernels": kern,
                    "step_frac_of_peak": ((64 if per_elem else 40) * nn * B) / (ms_step * 1e-3) / 1e9 / peak}

    # ---------------- end to end through the product API with HOST buffers: u = solver(f_host); u.backward(gbar)
    # The row streaming (pinned chunks on a copy stream overlapped with the kernels) is the product's, not bench code.
    e2e = e2e_full = None
    if not args.no_e2e:
        f_host = torch.empty((B, nn), dtype=torch.float64, pin_memory=True)
        f_host.copy_(f.detach())
        k_host = kappa.detach().cpu()
        n_e2e = max(2, min(args.steps, 5))

        def time_e2e(step_fn, host_clock):
            for _ in range(2):
                step_fn()
            barrier()
            t0 = time.perf_counter()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(n_e2e):
                step_fn()
            a1.record()
            barrier()
            wall = (time.perf_counter() - t0) * 1e3           # the host waits inside the step when results land on the CPU
            ms = wall if host_clock else a0.elapsed_time(a1)
            if world > 1:
                t = torch.tensor([ms, wall], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms, wall = float(t[0]), float(t[1])
            return ms, wall

        def step_inverse():
            """f, kappa on the host -> forward + adjoint on the device -> dL/dkappa on the host (the inverse-problem step:
            f is data, dL/df is not requested; u stays on the device because the loss is formed there)."""
            kr = k_host.clone().requires_grad_(True)
            u = DifferentiableFESolver(mesh, kappa=kr, out_device=dev)(f_host)
            u.backward(gbar)
            return kr.grad                                     # a CPU tensor: autograd moved it (and waited)

        ms, wall = time_e2e(step_inverse, False)
        e2e = {"value": B * world * n_e2e / (ms * 1e-3), "unit": "solves/s", "wall_ms_per_step": wall / n_e2e,
               "h2d_bytes_per_step": int(f_host.numel() * 8 + k_host.numel() * 8), "d2h_bytes_per_step": int(k_host.numel() * 8),
               "steps": n_e2e, "ms_per_step": ms / n_e2e, "call": "u = DifferentiableFESolver(mesh, kappa_host, out_device='cuda')(f_host_pinned); "
               "u.backward(gbar_dev); kappa_host.grad", "grads": "dL/dkappa (f is host data and does not require grad)",
               "pipeline": "product-side row streaming (solver._RowPipe): 8 chunks, H2D stream + compute stream", "host_binding": host_binding}

        gbar_host = torch.empty((B, nn), dtype=torch.float64, pin_memory=True)
        gbar_host.copy_(gbar)

        def step_full():
            """Everything crosses: f, kappa, gbar from the host; u, dL/df, dL/dkappa back to the host."""
            kr = k_host.clone().requires_grad_(True)
            fr = f_host.requires_grad_(True)
            fr.grad = None
            u = DifferentiableFESolver(mesh, kappa=kr)(fr)     # CPU in -> CPU out (the reference's calling convention)
            u.backward(gbar_host)
            return kr.grad

        try:
            ms, _ = time_e2e(step_full, True)
            e2e_full = {"value": B * world * n_e2e / (ms * 1e-3), "unit": "solves/s",
                        "h2d_bytes_per_step": int(2 * f_host.numel() * 8 + k_host.numel() * 8),
                        "d2h_bytes_per_step": int(2 * f_host.numel() * 8 + k_host.numel() * 8), "steps": n_e2e, "ms_per_step": ms / n_e2e,
                        "call": "u_host = DifferentiableFESolver(mesh, kappa_host)(f_host); u_host.backward(gbar_host): u, dL/df and dL/dkappa "
                                "all return to the host (timed on the host clock: the call blocks until they have landed)"}
        except Exception as exc:                               # never sink the headline on the secondary number
            e2e_full = {"value": None, "error": f"{type(exc).__name__}: {exc}"}
        f_host.requires_grad_(False)
        del f_host, gbar_host

    clocks = sampler.stop()

    # ---------------- config 5 (the multi-GPU config north_star names): strong-scaling sweep with its collective
    sweep = None
    if not args.no_sweep:
        del f, gbar, keep
        torch.cuda.empty_cache()
        try:
            sweep = time_sweep(args, rank, world, dev, WORKLOADS["c5a"]["n_elements"], WORKLOADS["c5a"]["batch"],
                               steps=args.steps, warmup=args.warmup)
        except Exception as exc:
            sweep = {"value": None, "error": f"{type(exc).__name__}: {exc}"}

    # ---------------- CPU baseline (rank 0, N = 1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            rate, cores, sample, _ = cpu_port_rate(n_el, seconds_target=12.0)
            cpu = {"value": rate, "unit": "solves/s", "cores": cores, "kind": "port", "sample": sample}
        except Exception as exc:  # the baseline must never sink the GPU number
            cpu = {"value": None, "unit": "solves/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {exc}"}

    if rank == 0:
        line = {
            "metric": "fem_fwd_adjoint_solves_per_s", "value": value, "unit": "solves/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": w["scaling"], "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "dof_per_s": value * (n_el - 1),
            "config": {"workload": w["desc"], "n_elements": n_el, "batch_per_gpu": B, "global_batch": B * world,
                       "kappa": w["kappa"], "grads": "dL/dkappa and dL/df", "l2": "inputs (3.28 GB/array) larger than L2; no flush",
                       "accounting_bytes_per_node": 64 if per_elem else 40,
                       "parallelism": f"batch-sharded x{world}, mesh replicated, no collective (per-sample kappa); the config-5 sweep "
                                      "with its NCCL all-reduce is timed in the same run: see `sweep`"},
            "roofline": roofline, "parity": parity, "cpu_baseline": cpu, "e2e": e2e, "e2e_full": e2e_full, "sweep": sweep,
            "gpu_launches": launches, "clocks": clocks,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_b200_sweep(args, w, rank, local_rank, world, dev):
    """--workload c5a: the config-5a sweep as the main line (strong scaling, collective inside the timed region)."""
    import torch.distributed as dist

    sampler = ClockSampler(local_rank)
    sampler.start()
    r = time_sweep(args, rank, world, dev, args.n_elements or w["n_elements"], args.batch or w["batch"], args.steps, args.warmup,
                   dump_dir=args.dump_outputs)
    clocks = sampler.stop()
    peak, peak_src = measured_peak()
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            rate, cores, sample, _ = cpu_port_rate(r["n_elements"], seconds_target=8.0)
            cpu = {"value": rate, "unit": "solves/s", "cores": cores, "kind": "port", "sample": sample}
        except Exception as exc:
            cpu = {"value": None, "unit": "solves/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {exc}"}
    if rank == 0:
        dom = max((k for k in r["kernels"] if "achieved_gbs" in r["kernels"][k]), key=lambda k: r["kernels"][k]["ms_per_launch"])
        kd = r["kernels"][dom]
        line = {"metric": "fem_fwd_adjoint_solves_per_s", "value": r["value"], "unit": "solves/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "dof_per_s": r["value"] * (r["n_elements"] - 1),
                "config": {"workload": r["workload"], "n_elements": r["n_elements"], "batch_per_gpu": r["batch_per_gpu"],
                           "global_batch": r["global_batch"], "kappa": "shared", "step": r["step"], "collective": r["collective"],
                           "l2": "inputs (8.6 GB/array over all ranks) larger than L2; no flush"},
                "roofline": {"bound": "hbm", "kernel": dom, "achieved": kd["achieved_gbs"], "peak": peak, "unit": "GB/s",
                             "frac": kd["frac"], "traffic": None, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": kd["algorithmic_bytes"], "ms_per_launch": kd["ms_per_launch"],
                             "kernels": r["kernels"], "step_frac_of_peak": r["step_frac_of_peak"]},
                "cpu_baseline": cpu, "e2e": None,
                "e2e_note": "the sweep's f and u_data stay resident on the GPU across optimisation steps; only kappa (8 B) and the "
                            "reduced [dL/dkappa, loss] (16 B) would cross per step",
                "gpu_launches": r["gpu_launches"], "clocks": clocks,
                "loss_first_step": r["loss_first_step"], "loss_last_step": r["loss_last_step"], "kappa_after": r["kappa_after"]}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_b200_2d(args, w, rank, local_rank, world, dev):
    """Configs 3 / 4: one 2-D mesh per GPU (replicas only across GPUs), step = forward + adjoint of one solve."""
    import torch
    import torch.distributed as dist

    from difffe_physics_lab_b200 import DifferentiableFESolver, FEMesh
    from difffe_physics_lab_b200.solver import KernelTimer

    nx = args.n_elements or w["nx"]
    t0 = time.perf_counter()
    mesh = FEMesh.rectangle(nx, nx)
    gen = torch.Generator(device=dev).manual_seed(rank)
    if w["kappa"] == "per_element":
        kappa = torch.exp(torch.empty(mesh.n_elements, dtype=torch.float64, device=dev).uniform_(float(np.log(1e-3)), 0.0, generator=gen))
    else:
        kappa = torch.tensor(1.0, dtype=torch.float64, device=dev)
    f = torch.ones(mesh.n_nodes, dtype=torch.float64, device=dev)
    nm = mesh._native(dev.index)
    t_setup = time.perf_counter() - t0
    I = nm.info
    its = {}

    def step():
        kr = kappa.detach().requires_grad_(True)
        s = DifferentiableFESolver(mesh, kappa=kr, solver2d=os.environ.get("DFE_SOLVER2D", "auto"),
                                   mg_nu=int(os.environ.get("DFE_MG_NU", "2")))
        u = s(f)
        u.sum().backward()
        its["fwd"] = s.last_pcg[0][0]
        its["adj"] = s._opts["last_pcg_adjoint"][0][0]
        its["u"], its["gk"] = u, kr.grad
        return kr.grad

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with KernelTimer() as kt:
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        barrier()
    clocks = sampler.stop()
    ms_total = e0.elapsed_time(e1)
    ksum = kt.summary()
    if world > 1:
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t[0])
    ms_step = ms_total / args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"u": its["u"], "grad_kappa": its["gk"]})
    parity = None
    if rank == 0 and not args.no_parity:
        try:
            parity = parity_block_2d(mesh, nm, kappa, f, its.pop("u"), its.pop("gk"))
        except Exception as exc:
            parity = {"true_residual_rel": None, "error": f"{type(exc).__name__}: {exc}"}
    its.pop("u", None)
    its.pop("gk", None)
    peak, peak_src = measured_peak()
    N, nnz = I.n_free, I.nnz_free
    bytes_iter = 12 * nnz + 104 * N + 4 * (N + 1)              # SURVEY §8d accounting convention
    solver2d = "mg" if "mg_pcg" in ksum else "jacobi"
    calls, ms_pcg = ksum.get("mg_pcg") or ksum.get("pcg", (0, 0.0))
    iters_step = its.get("fwd", 0) + its.get("adj", 0)
    roofline = None
    if calls:
        ms_launch = ms_pcg / calls
        alg = bytes_iter * iters_step / 2.0                     # per PCG launch (forward and adjoint solves average)
        roofline = {"bound": "hbm", "kernel": "k_mgpcg (cooperative multigrid-preconditioned CG)" if solver2d == "mg" else "k_pcg (cooperative Jacobi-PCG)", "achieved": alg / (ms_launch * 1e-3) / 1e9,
                    "peak": peak, "unit": "GB/s", "frac": alg / (ms_launch * 1e-3) / 1e9 / peak,
                    "traffic": measured_traffic("c4", "k_pcg(") if args.workload == "c4" and not args.n_elements else None,
                    "note": "achieved = SURVEY 8(d) accounting bytes / time; the gathered vectors stay in the 126 MB L2 "
                            "(matrix loads are evict-first), so the DRAM traffic in `traffic` is lower than the accounting",
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": alg, "ms_per_launch": ms_launch,
                    "bytes_per_iteration": bytes_iter, "iterations": its, "us_per_iteration": 1e3 * ms_pcg / calls / (iters_step / 2.0),
                    "kernels": {k: {"calls": c, "ms_per_launch": m / c} for k, (c, m) in ksum.items()}}
    if roofline is not None and solver2d == "mg":
        tr = measured_traffic("c4", "k_mgpcg") if args.workload == "c4" and not args.n_elements else None
        roofline["traffic"] = tr
        roofline["traffic_source"] = ("REPLAYED from profiles/r*_traffic.json (one earlier `ncu --set full` capture of k_mgpcg on this "
                                      "workload), not measured in this run")
        roofline["note"] = ("achieved = SURVEY 8(d) Jacobi-PCG accounting bytes per iteration x MG-PCG iterations / time: the "
                            "multigrid cycle does ~10x the arithmetic of a Jacobi iteration per CG step and needs 170x fewer "
                            "steps, so this figure measures nothing useful; achieved_dram = measured DRAM bytes / time is the "
                            "honest utilisation (the hierarchy is largely L2-resident; the kernel is bound by its grid barriers)")
        if tr:
            roofline["achieved_dram"] = tr / (roofline["ms_per_launch"] * 1e-3) / 1e9
            roofline["frac_dram"] = roofline["achieved_dram"] / peak
    # ---------------- CPU baseline (rank 0, N = 1): same Jacobi-PCG the reference-faithful route runs, on the host cores
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            kr = kappa.detach().requires_grad_(True)
            sj = DifferentiableFESolver(mesh, kappa=kr, solver2d="jacobi")
            sj(f).sum().backward()
            itj = int(sj.last_pcg[0][0] + sj._opts["last_pcg_adjoint"][0][0])
            knp = kappa.detach().cpu().numpy()
            cpu = cpu_rate_2d(mesh, float(knp) if knp.ndim == 0 else knp, f.cpu().numpy(), itj)
            cpu["jacobi_iterations_fwd_plus_adjoint"] = itj
        except Exception as exc:
            cpu = {"value": None, "unit": "solves/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {exc}"}
    # ---------------- end to end through the module with HOST tensors (CPU in -> CPU out, the reference's convention)
    e2e = None
    if not args.no_e2e:
        k_host = kappa.detach().cpu()
        f_host = f.cpu().pin_memory()
        n_e2e = max(2, min(args.steps, 5))

        def step_host():
            kr = k_host.clone().requires_grad_(True)
            s = DifferentiableFESolver(mesh, kappa=kr, solver2d=os.environ.get("DFE_SOLVER2D", "auto"),
                                       mg_nu=int(os.environ.get("DFE_MG_NU", "2")))
            u = s(f_host)
            u.sum().backward()
            return u, kr.grad

        for _ in range(2):
            step_host()
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            uh, gh = step_host()
        barrier()
        wall = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([wall], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            wall = float(t[0])
        e2e = {"value": world * n_e2e / wall, "unit": "solves/s", "ms_per_step": 1e3 * wall / n_e2e, "steps": n_e2e,
               "h2d_bytes_per_step": int(8 * (f_host.numel() + k_host.numel() + uh.numel())),
               "d2h_bytes_per_step": int(8 * (uh.numel() + gh.numel())),
               "call": "u_host = DifferentiableFESolver(mesh, kappa_host)(f_host); u_host.sum().backward(): f, kappa and the upstream "
                       "gradient cross to the device, u and dL/dkappa come back (host clock; includes the host-side set-up of the call)"}
    if rank == 0:
        line = {"metric": "fem_fwd_adjoint_solves_per_s", "value": world * args.steps / (ms_total * 1e-3), "unit": "solves/s",
                "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "dof_per_s": world * args.steps / (ms_total * 1e-3) * N,
                "config": {"workload": w["desc"], "nx": nx, "n_free": int(N), "nnz_free": int(nnz), "pcg_tol": 1e-13,
                           "l2": "config 4 working set ~0.2 GB > L2; config 3 (3 MB) is L2/latency-bound by construction",
                           "mesh_setup_s": t_setup, "parallelism": f"replicas only x{world} (a single mesh stays on one GPU)"},
                "roofline": roofline, "parity": parity, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": kt.launches,
                "clocks": clocks}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_b200_small2d(args, w, rank, local_rank, world, dev):
    """Config 5b: many small 2-D systems with a shared kappa, one CTA per sample (dfe_batch_fwd / dfe_batch_bwd);
    the batch is sharded over the ranks, the only collective is the all-reduce of [dL/dkappa, loss]."""
    import torch
    import torch.distributed as dist

    from difffe_physics_lab_b200 import DifferentiableFESolver, FEMesh
    from difffe_physics_lab_b200.solver import KernelTimer

    nx = args.n_elements or w["nx"]
    B = (args.batch or w["batch"]) // world
    mesh = FEMesh.rectangle(nx, nx)
    nn = mesh.n_nodes
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    f = torch.rand((B, nn), dtype=torch.float64, device=dev, generator=gen) + 0.5
    gbar = torch.randn((B, nn), dtype=torch.float64, device=dev, generator=gen)
    kappa = torch.tensor(1.0, dtype=torch.float64, device=dev)
    red = torch.zeros(2, dtype=torch.float64, device=dev)
    its = {}

    def step():
        fr = f.requires_grad_(True)
        fr.grad = None
        kr = kappa.detach().requires_grad_(True)
        s = DifferentiableFESolver(mesh, kappa=kr)
        u = s(fr)
        u.backward(gbar)
        its["fwd"] = s.last_pcg[0][0]
        its["adj"] = s._opts["last_pcg_adjoint"][0][0]
        its["u"] = u
        if world > 1:
            red[0] = kr.grad
            dist.all_reduce(red)
        return kr.grad

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with KernelTimer() as kt:
        e0.record()
        for _ in range(args.steps):
            gk_last = step()
        e1.record()
        barrier()
    clocks = sampler.stop()
    ms_total = e0.elapsed_time(e1)
    ksum = kt.summary()
    if world > 1:
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t[0])
    ms_step = ms_total / args.steps
    value = B * world * args.steps / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"grad_kappa": gk_last}, {"u": its["u"], "grad_f": f.grad})
    parity = None
    u_last = its.pop("u", None)
    if rank == 0 and not args.no_parity and u_last is not None:
        try:
            parity = parity_block_small2d(mesh, sorted({0, B // 2 + 1, B - 1}), f, kappa, gbar, u_last, f.grad)
        except Exception as exc:
            parity = {"max_rel": None, "error": f"{type(exc).__name__}: {exc}"}
    del u_last
    peak, peak_src = measured_peak()
    kern = {k: {"calls": c, "ms_per_launch": m / c} for k, (c, m) in ksum.items()}
    roofline = None
    for key, kname, note in (("band_bwd", "dfe_band_bwd = k_band_rhs_bwd + k_band_solve_mma (block TRSM on the FP64 tensor cores) + k_band_grad3 + k_band_gksum",
                              "achieved = 24 B/node accounting (read gbar, read u, write dL/df) / time; the call itself moves more: the "
                              "right-hand sides are gathered to (B, npad), solved in place and read back by the gradient kernel"),
                             ("batch_bwd", "k_batch<adjoint> (one CTA per sample, matrix in shared memory)",
                              "shared-memory resident PCG: bound by the SpMV's shared-memory traffic, not by HBM")):
        if key in kern:
            alg = 24 * nn * B                                     # read gbar, read u, write dL/df
            ms = kern[key]["ms_per_launch"]
            roofline = {"bound": "hbm", "kernel": kname, "achieved": alg / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": alg / (ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                        "algorithmic_bytes_per_launch": alg, "ms_per_launch": ms, "note": note, "max_iterations": its,
                        "kernels": kern}
            break
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        try:
            cpu = cpu_rate_2d_batch(mesh, 1.0, 64 * len(os.sched_getaffinity(0)))
        except Exception as exc:
            cpu = {"value": None, "unit": "solves/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {exc}"}
    e2e = None
    if not args.no_e2e:
        f_host = torch.empty((B, nn), dtype=torch.float64, pin_memory=True)
        f_host.copy_(f.detach())
        g_host = torch.empty((B, nn), dtype=torch.float64, pin_memory=True)
        g_host.copy_(gbar)
        k_host = kappa.detach().cpu()
        n_e2e = max(2, min(args.steps, 5))

        def step_host():
            kr = k_host.clone().requires_grad_(True)
            u = DifferentiableFESolver(mesh, kappa=kr)(f_host)
            u.backward(g_host)
            return u, kr.grad

        for _ in range(2):
            step_host()
        barrier()
        t0 = time.perf_counter()
        for _ in range(n_e2e):
            uh, gh = step_host()
        barrier()
        wall = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([wall], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            wall = float(t[0])
        e2e = {"value": B * world * n_e2e / wall, "unit": "solves/s", "ms_per_step": 1e3 * wall / n_e2e, "steps": n_e2e,
               "h2d_bytes_per_step": int(8 * (2 * f_host.numel() + 1)), "d2h_bytes_per_step": int(8 * (f_host.numel() + 1)),
               "call": "u_host = DifferentiableFESolver(mesh, kappa_host)(f_host_pinned); u_host.backward(gbar_host_pinned): f and gbar "
                       "cross to the device, u and dL/dkappa come back (host clock; f is data, dL/df is not requested)"}
        del f_host, g_host
    if rank == 0:
        I = mesh._native(dev.index).info
        line = {"metric": "fem_fwd_adjoint_solves_per_s", "value": value, "unit": "solves/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "dof_per_s": value * int(I.n_free),
                "config": {"workload": w["desc"], "nx": nx, "n_free": int(I.n_free), "batch_per_gpu": B, "global_batch": B * world,
                           "kappa": "shared", "pcg_tol": 1e-13, "l2": "inputs 0.57 GB/array larger than L2; no flush",
                           "parallelism": f"batch-sharded x{world}, mesh replicated" + (", NCCL allreduce of [dL/dkappa, loss]" if world > 1 else "")},
                "roofline": roofline, "parity": parity, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": kt.launches,
                "clocks": clocks}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
