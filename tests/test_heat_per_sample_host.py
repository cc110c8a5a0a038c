"""The per-sample-kappa heat rollout entry points (dfe_heat_ps_*) on a host-only mesh handle: they refuse with
DFE_ERR_CUDA (the library has no CPU path) and report no sizes."""
from difffe_physics_lab_b200 import FEMesh, _native


def test_host_only_handle_refuses():
    L = _native.lib()
    nm = FEMesh.rectangle(5, 4)._native(-1)   # kept alive: the handle belongs to it
    h = nm.handle
    assert L.dfe_heat_ps_factor_bytes(h, 4) == 0 and L.dfe_heat_ps_workspace_bytes(h, 4) == 0
    ps = _native.KAPPA_PER_SAMPLE_ELEMENT
    assert L.dfe_heat_ps_setup(h, 2, 8, ps, 1e-2, 8, None, 16, 8, 8, 8, 1 << 20, None) == _native.ERR_CUDA
    assert L.dfe_heat_ps_fwd(h, 2, 3, 8, 30, 16, 8, 8, 8, 8, 90, 30, None) == _native.ERR_CUDA
    assert L.dfe_heat_ps_adj(h, 2, 0, 3, 8, 90, 30, 1, 16, 8, 8, 8, 8, None) == _native.ERR_CUDA
    assert L.dfe_heat_ps_grad(h, 2, 3, 16, 8, 90, 30, 8, 8, None) == _native.ERR_CUDA
    assert L.dfe_heat_ps_grad_sum(h, 2, 1e-2, ps, 8, 8, None) == _native.ERR_CUDA
    assert b"no CUDA device" in L.dfe_last_error()


def test_null_handle_is_invalid():
    L = _native.lib()
    assert L.dfe_heat_ps_fwd(None, 2, 3, 8, 30, 16, 8, 8, 8, 8, 90, 30, None) == _native.ERR_INVALID
    assert L.dfe_heat_ps_grad_sum(None, 2, 1e-2, _native.KAPPA_PER_SAMPLE, 8, 8, None) == _native.ERR_INVALID
