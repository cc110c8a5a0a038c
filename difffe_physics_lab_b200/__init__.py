"""difffe_physics_lab_b200 — B200-native differentiable P1-FEM Poisson solver behind the
DiffFE-Physics-Lab API (``FEMesh``, ``DifferentiableFESolver``, ``PhysicsLoss``, ``NeuralPDE``).

Only the hot path is accelerated: assembly -> Dirichlet elimination -> linear solve -> adjoint ->
dL/dkappa, as hand-written sm_100a CUDA behind the C ABI of ``include/dfe.h``.  ``import diffhe``
(the reference's package name) resolves to thin aliases of these modules.
"""
from .mesh import FEMesh
from .solver import DifferentiableFESolver, assemble_sparse
from .loss import PhysicsLoss
from .neural import NeuralPDE
from .timestepping import DifferentiableHeatSolver

__version__ = "0.1.0"
__all__ = ["FEMesh", "DifferentiableFESolver", "PhysicsLoss", "NeuralPDE", "assemble_sparse", "DifferentiableHeatSolver"]
