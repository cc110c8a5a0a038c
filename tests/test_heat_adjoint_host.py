"""DifferentiableHeatSolver without a CUDA device: it raises instead of falling back to the CPU."""
import pytest
import torch

from difffe_physics_lab_b200 import DifferentiableHeatSolver, FEMesh


def test_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is visible")
    mesh = FEMesh.rectangle(4, 4)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        DifferentiableHeatSolver(mesh, 1.0, 1e-2)(torch.zeros(mesh.n_nodes), 2)
