"""ctypes binding of libdfe_b200.so (the C ABI declared in include/dfe.h).

The shared library is built in-tree by :func:`build` (``nvcc`` for sm_100a, ``-lineinfo``) and
loaded with ``ctypes.CDLL`` — there is no torch C++ extension and no torch type crosses the
boundary: tensors are passed as ``data_ptr()`` integers plus sizes, the CUDA stream as the raw
``cudaStream_t`` of ``torch.cuda.current_stream()``.

There is no CPU fallback: if the library is missing or no CUDA device is visible, the compute
entry points raise.
"""
from __future__ import annotations

import ctypes as C
import os
import pathlib
import shutil
import subprocess

PKG = pathlib.Path(__file__).resolve().parent
ROOT = PKG.parent
LIB_PATH = PKG / "libdfe_b200.so"
SOURCES = ["dfe_mesh.cu", "dfe_1d.cu", "dfe_1d_split.cu", "dfe_1d_pipe.cu", "dfe_general.cu", "dfe_pcg.cu", "dfe_mg.cu",
           "dfe_batch.cu", "dfe_band_ps.cu", "dfe_heat.cu"]
HEADERS = [PKG / "csrc" / "dfe_internal.h", PKG / "csrc" / "dfe_1d_common.cuh", PKG / "csrc" / "dfe_gridsync.cuh", PKG / "csrc" / "dfe_exact.cuh",
           PKG / "csrc" / "dfe_p2.cuh", PKG / "csrc" / "dfe_mg_kernel.cuh", PKG / "csrc" / "dfe_band_mma.cuh",
           PKG / "csrc" / "dfe_assemble_row.cuh", PKG / "csrc" / "dfe_band_ps_solve.cuh",
           ROOT / "include" / "dfe.h"]

OK, ERR_INVALID, ERR_CUDA, ERR_UNSUPPORTED, ERR_NOT_CONVERGED, ERR_BREAKDOWN, ERR_WORKSPACE = range(7)
KAPPA_SCALAR, KAPPA_PER_SAMPLE, KAPPA_PER_ELEMENT, KAPPA_PER_SAMPLE_ELEMENT = range(4)

# every symbol include/dfe.h declares (tests check the library exports exactly these)
SYMBOLS = [
    "dfe_last_error", "dfe_abi_version", "dfe_device_count",
    "dfe_mesh_create", "dfe_mesh_create_p", "dfe_mesh_destroy", "dfe_mesh_get_info", "dfe_mesh_csr_host", "dfe_mesh_free_nodes_host",
    "dfe_solve1d_workspace_bytes", "dfe_solve1d_fwd", "dfe_solve1d_bwd", "dfe_solve1d_bwd_misfit",
    "dfe_solve1d_supported", "dfe_mesh_fault",
    "dfe_assemble", "dfe_eliminate", "dfe_pcg_workspace_bytes", "dfe_pcg", "dfe_scatter", "dfe_gather_free",
    "dfe_grad_workspace_bytes", "dfe_grad",
    "dfe_mg_supported", "dfe_mg_hierarchy_bytes", "dfe_mg_workspace_bytes", "dfe_mg_setup", "dfe_mg_pcg",
    "dfe_batch_supported", "dfe_batch_fwd", "dfe_batch_bwd",
    "dfe_band_supported", "dfe_band_factor_bytes", "dfe_band_workspace_bytes", "dfe_band_factor", "dfe_band_fwd", "dfe_band_bwd",
    "dfe_band_npad", "dfe_band_solve",
    "dfe_band_ps_supported", "dfe_band_ps_factor_bytes", "dfe_band_ps_workspace_bytes", "dfe_band_ps_fwd", "dfe_band_ps_bwd",
    "dfe_heat_supported", "dfe_heat_warps", "dfe_heat_grad_bytes", "dfe_heat_fwd", "dfe_heat_adj", "dfe_heat_grad",
    "dfe_heat_grad_sum",
    "dfe_heat_ps_factor_bytes", "dfe_heat_ps_workspace_bytes", "dfe_heat_ps_setup", "dfe_heat_ps_fwd", "dfe_heat_ps_adj",
    "dfe_heat_ps_grad", "dfe_heat_ps_grad_sum",
]


class DfeError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(message)
        self.status = status


class NotConvergedError(DfeError):
    pass


class BreakdownError(DfeError):
    pass


class MeshInfo(C.Structure):
    _fields_ = [
        ("dim", C.c_int32), ("device", C.c_int32),
        ("n_nodes", C.c_int64), ("n_elements", C.c_int64), ("n_dirichlet", C.c_int64), ("n_free", C.c_int64),
        ("nnz_full", C.c_int64), ("nnz_free", C.c_int64), ("sell_nnz", C.c_int64),
        ("max_row_nnz", C.c_int32), ("chain1d", C.c_int32),
    ]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def needs_build() -> bool:
    if not LIB_PATH.exists():
        return True
    t = LIB_PATH.stat().st_mtime
    deps = [PKG / "csrc" / s for s in SOURCES] + HEADERS
    return any(d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> pathlib.Path:
    """Compile csrc/*.cu into libdfe_b200.so for sm_100a (cross-compiles without a GPU).

    One object file per translation unit (compiled in parallel, only when the source or a header changed), then one
    link step; objects live in ``difffe_physics_lab_b200/build/`` (git-ignored)."""
    if not force and not needs_build():
        return LIB_PATH
    from concurrent.futures import ThreadPoolExecutor

    objdir = PKG / "build"
    objdir.mkdir(exist_ok=True)
    extra = (os.environ.get("DFE_NVCC_FLAGS") or "").split()      # e.g. -DDFE_SOME_DEBUG_SWITCH=1
    flags = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-Xcompiler", "-fPIC",
             "-I", str(ROOT / "include"), "-I", str(PKG / "csrc")] + extra + (["-Xptxas=-v"] if verbose else [])
    stamp = objdir / "flags.txt"
    if not stamp.exists() or stamp.read_text() != " ".join(flags):
        force = True
    hdr_t = max(h.stat().st_mtime for h in HEADERS)

    def compile_one(src: str):
        cu, obj = PKG / "csrc" / src, objdir / (src + ".o")
        if not force and obj.exists() and obj.stat().st_mtime > max(cu.stat().st_mtime, hdr_t):
            return ""
        res = subprocess.run([nvcc_path()] + flags + ["-c", str(cu), "-o", str(obj)], capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n" + res.stdout + res.stderr)
        return res.stderr

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 4)) as ex:
        logs = list(ex.map(compile_one, SOURCES))
    stamp.write_text(" ".join(flags))
    res = subprocess.run([nvcc_path(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", str(LIB_PATH)]
                         + [str(objdir / (s + ".o")) for s in SOURCES], capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
    if verbose:
        print("\n".join(logs))
    return LIB_PATH


_lib = None


def lib() -> C.CDLL:
    """Load (once) and return the shared library; raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(difffe_physics_lab_b200 has no CPU fallback)"
        )
    L = C.CDLL(str(LIB_PATH))
    vp, i64, dbl, sz, ci = C.c_void_p, C.c_int64, C.c_double, C.c_size_t, C.c_int
    L.dfe_last_error.restype = C.c_char_p
    L.dfe_last_error.argtypes = []
    L.dfe_abi_version.restype = ci
    L.dfe_device_count.restype = ci
    L.dfe_mesh_create.restype = ci
    L.dfe_mesh_create.argtypes = [ci, i64, i64, vp, vp, i64, vp, vp, ci, C.POINTER(vp)]
    L.dfe_mesh_create_p.restype = ci
    L.dfe_mesh_create_p.argtypes = [ci, ci, i64, i64, vp, vp, i64, vp, vp, ci, C.POINTER(vp)]
    L.dfe_mesh_destroy.restype = None
    L.dfe_mesh_destroy.argtypes = [vp]
    L.dfe_mesh_get_info.restype = ci
    L.dfe_mesh_get_info.argtypes = [vp, C.POINTER(MeshInfo)]
    L.dfe_mesh_csr_host.restype = ci
    L.dfe_mesh_csr_host.argtypes = [vp, ci, C.POINTER(vp), C.POINTER(vp), C.POINTER(i64), C.POINTER(i64)]
    L.dfe_mesh_free_nodes_host.restype = ci
    L.dfe_mesh_free_nodes_host.argtypes = [vp, C.POINTER(vp), C.POINTER(i64)]
    L.dfe_solve1d_workspace_bytes.restype = sz
    L.dfe_solve1d_workspace_bytes.argtypes = [vp, i64]
    L.dfe_solve1d_fwd.restype = ci
    L.dfe_solve1d_fwd.argtypes = [vp, i64, vp, i64, vp, ci, ci, vp, i64, vp, sz, vp]
    L.dfe_solve1d_bwd.restype = ci
    L.dfe_solve1d_bwd.argtypes = [vp, i64, vp, i64, vp, i64, vp, ci, ci, vp, i64, vp, vp, sz, vp]
    L.dfe_solve1d_bwd_misfit.restype = ci
    L.dfe_solve1d_bwd_misfit.argtypes = [vp, i64, vp, i64, vp, i64, vp, ci, ci, dbl, vp, i64, vp, vp, vp, sz, vp]
    L.dfe_solve1d_supported.restype = ci
    L.dfe_solve1d_supported.argtypes = [vp, ci, ci]
    L.dfe_mesh_fault.restype = ci
    L.dfe_mesh_fault.argtypes = [vp]
    L.dfe_assemble.restype = ci
    L.dfe_assemble.argtypes = [vp, vp, ci, vp, vp, vp, vp]
    L.dfe_eliminate.restype = ci
    L.dfe_eliminate.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.dfe_pcg_workspace_bytes.restype = sz
    L.dfe_pcg_workspace_bytes.argtypes = [vp]
    L.dfe_pcg.restype = ci
    L.dfe_pcg.argtypes = [vp, vp, vp, vp, vp, dbl, i64, C.POINTER(i64), C.POINTER(dbl), vp, sz, vp]
    L.dfe_scatter.restype = ci
    L.dfe_scatter.argtypes = [vp, vp, ci, vp, vp]
    L.dfe_gather_free.restype = ci
    L.dfe_gather_free.argtypes = [vp, vp, vp, vp]
    L.dfe_grad_workspace_bytes.restype = sz
    L.dfe_grad_workspace_bytes.argtypes = [vp]
    L.dfe_grad.restype = ci
    L.dfe_grad.argtypes = [vp, vp, vp, vp, ci, vp, vp, vp, sz, vp]
    L.dfe_mg_supported.restype = ci
    L.dfe_mg_supported.argtypes = [vp]
    L.dfe_mg_hierarchy_bytes.restype = sz
    L.dfe_mg_hierarchy_bytes.argtypes = [vp]
    L.dfe_mg_workspace_bytes.restype = sz
    L.dfe_mg_workspace_bytes.argtypes = [vp]
    L.dfe_mg_setup.restype = ci
    L.dfe_mg_setup.argtypes = [vp, vp, vp, sz, vp]
    L.dfe_mg_pcg.restype = ci
    L.dfe_mg_pcg.argtypes = [vp, vp, vp, vp, dbl, i64, ci, C.POINTER(i64), C.POINTER(dbl), vp, sz, vp]
    L.dfe_batch_supported.restype = ci
    L.dfe_batch_supported.argtypes = [vp]
    L.dfe_batch_fwd.restype = ci
    L.dfe_batch_fwd.argtypes = [vp, i64, vp, i64, vp, vp, vp, vp, i64, dbl, i64, vp, vp, vp, vp]
    L.dfe_batch_bwd.restype = ci
    L.dfe_batch_bwd.argtypes = [vp, i64, vp, i64, vp, i64, vp, vp, ci, vp, i64, vp, dbl, i64, vp, vp, vp, vp]
    L.dfe_band_supported.restype = ci
    L.dfe_band_supported.argtypes = [vp]
    L.dfe_band_factor_bytes.restype = sz
    L.dfe_band_factor_bytes.argtypes = [vp]
    L.dfe_band_workspace_bytes.restype = sz
    L.dfe_band_workspace_bytes.argtypes = [vp, i64]
    L.dfe_band_factor.restype = ci
    L.dfe_band_factor.argtypes = [vp, vp, vp, vp, vp]
    L.dfe_band_fwd.restype = ci
    L.dfe_band_fwd.argtypes = [vp, i64, vp, i64, vp, vp, vp, i64, vp, sz, vp]
    L.dfe_band_bwd.restype = ci
    L.dfe_band_bwd.argtypes = [vp, i64, vp, i64, vp, i64, vp, ci, vp, i64, vp, vp, sz, vp]
    L.dfe_band_npad.restype = i64
    L.dfe_band_npad.argtypes = [vp]
    L.dfe_band_solve.restype = ci
    L.dfe_band_solve.argtypes = [vp, i64, vp, vp, vp]
    L.dfe_band_ps_supported.restype = ci
    L.dfe_band_ps_supported.argtypes = [vp]
    L.dfe_band_ps_factor_bytes.restype = sz
    L.dfe_band_ps_factor_bytes.argtypes = [vp, i64]
    L.dfe_band_ps_workspace_bytes.restype = sz
    L.dfe_band_ps_workspace_bytes.argtypes = [vp, i64]
    L.dfe_band_ps_fwd.restype = ci
    L.dfe_band_ps_fwd.argtypes = [vp, i64, vp, i64, vp, ci, vp, vp, i64, vp, vp, sz, vp]
    L.dfe_band_ps_bwd.restype = ci
    L.dfe_band_ps_bwd.argtypes = [vp, i64, vp, i64, vp, i64, vp, ci, vp, i64, vp, vp, sz, vp]
    L.dfe_heat_supported.restype = ci
    L.dfe_heat_supported.argtypes = [vp]
    L.dfe_heat_warps.restype = ci
    L.dfe_heat_warps.argtypes = [vp, i64]
    L.dfe_heat_grad_bytes.restype = sz
    L.dfe_heat_grad_bytes.argtypes = [vp, i64, i64]
    L.dfe_heat_fwd.restype = ci
    L.dfe_heat_fwd.argtypes = [vp, i64, i64, vp, i64, vp, vp, vp, vp, vp, i64, i64, ci, vp, vp]
    L.dfe_heat_adj.restype = ci
    L.dfe_heat_adj.argtypes = [vp, i64, i64, i64, vp, i64, i64, i64, vp, vp, vp, vp, vp, ci, vp, vp]
    L.dfe_heat_grad.restype = ci
    L.dfe_heat_grad.argtypes = [vp, i64, i64, i64, i64, vp, i64, i64, vp, vp, sz, vp]
    L.dfe_heat_grad_sum.restype = ci
    L.dfe_heat_grad_sum.argtypes = [vp, i64, i64, dbl, ci, vp, vp, sz, vp]
    L.dfe_heat_ps_factor_bytes.restype = sz
    L.dfe_heat_ps_factor_bytes.argtypes = [vp, i64]
    L.dfe_heat_ps_workspace_bytes.restype = sz
    L.dfe_heat_ps_workspace_bytes.argtypes = [vp, i64]
    L.dfe_heat_ps_setup.restype = ci
    L.dfe_heat_ps_setup.argtypes = [vp, i64, vp, ci, dbl, vp, vp, vp, vp, vp, vp, sz, vp]
    L.dfe_heat_ps_fwd.restype = ci
    L.dfe_heat_ps_fwd.argtypes = [vp, i64, i64, vp, i64, vp, vp, vp, vp, vp, i64, i64, vp]
    L.dfe_heat_ps_adj.restype = ci
    L.dfe_heat_ps_adj.argtypes = [vp, i64, i64, i64, vp, i64, i64, i64, vp, vp, vp, vp, vp, vp]
    L.dfe_heat_ps_grad.restype = ci
    L.dfe_heat_ps_grad.argtypes = [vp, i64, i64, vp, vp, i64, i64, vp, vp, vp]
    L.dfe_heat_ps_grad_sum.restype = ci
    L.dfe_heat_ps_grad_sum.argtypes = [vp, i64, dbl, ci, vp, vp, vp]
    if L.dfe_abi_version() != 1:
        raise RuntimeError("libdfe_b200.so ABI version mismatch")
    _lib = L
    return L


def check(status: int) -> None:
    """Turn a dfe_status into the Python exception the reference-facing API documents."""
    if status == OK:
        return
    msg = lib().dfe_last_error().decode("utf-8", "replace")
    if status == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)          # reference: NotImplementedError (solver.py:66-67)
    if status == ERR_INVALID:
        raise ValueError(msg)
    if status == ERR_NOT_CONVERGED:
        raise NotConvergedError(status, msg)
    if status == ERR_BREAKDOWN:
        raise BreakdownError(status, msg)
    raise DfeError(status, msg)
