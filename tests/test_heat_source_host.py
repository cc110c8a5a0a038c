"""The heat-source entry points (dfe_heat_src_*, dfe_heat_fwd_src, dfe_heat_ps_fwd_src) on a host-only mesh handle refuse
with DFE_ERR_CUDA (the library has no CPU path) and report no sizes; a null handle is DFE_ERR_INVALID."""
from difffe_physics_lab_b200 import FEMesh, _native


def test_host_only_handle_refuses():
    L = _native.lib()
    nm = FEMesh.rectangle(5, 4)._native(-1)   # kept alive: the handle belongs to it
    h = nm.handle
    assert L.dfe_heat_src_workspace_bytes(h) == 0
    assert L.dfe_heat_src_load(h, 3, 2, 1e-2, 8, 30, 90, 16, 0, 16, 8, 1 << 20, None) == _native.ERR_CUDA
    assert L.dfe_heat_fwd_src(h, 2, 3, 8, 30, 16, 16, 16, 64, 32, 16, 8, 90, 30, 0, 8, None) == _native.ERR_CUDA
    assert L.dfe_heat_ps_fwd_src(h, 2, 3, 8, 30, 16, 16, 16, 64, 32, 16, 8, 90, 30, None) == _native.ERR_CUDA
    assert L.dfe_heat_src_grad(h, 3, 2, 1e-2, 16, 64, 32, 8, 30, 90, 8, 1 << 20, None) == _native.ERR_CUDA
    assert b"no CUDA device" in L.dfe_last_error()


def test_null_handle_is_invalid():
    L = _native.lib()
    assert L.dfe_heat_src_workspace_bytes(None) == 0
    assert L.dfe_heat_src_load(None, 3, 2, 1e-2, 8, 30, 90, 16, 0, 16, 8, 1 << 20, None) == _native.ERR_INVALID
    assert L.dfe_heat_fwd_src(None, 2, 3, 8, 30, 16, 16, 16, 64, 32, 16, 8, 90, 30, 0, 8, None) == _native.ERR_INVALID
    assert L.dfe_heat_ps_fwd_src(None, 2, 3, 8, 30, 16, 16, 16, 64, 32, 16, 8, 90, 30, None) == _native.ERR_INVALID
    assert L.dfe_heat_src_grad(None, 3, 2, 1e-2, 16, 64, 32, 8, 30, 90, 8, 1 << 20, None) == _native.ERR_INVALID
