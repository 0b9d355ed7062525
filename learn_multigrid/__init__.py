"""Drop-in import path: `learn_multigrid.*` resolves to the B200 engine's mirror modules, so scripts written
against claudiotomasi/LearnMultigrid (`from learn_multigrid.solvers.Multigrid import *`, test/testMG.py:1-7)
run unchanged.  All code lives in learnmultigrid_b200/."""
import importlib
import sys

_SUBMODULES = [
    "solvers", "solvers.Solver", "solvers.Jacobi", "solvers.GaussSeidel", "solvers.CG", "solvers.GMRES", "solvers.Multigrid",
    "L2_projection", "L2_projection.L2Projection", "L2_projection.CouplingOperator", "L2_projection.Intersection",
    "assembly", "assembly.MassMatrix", "assembly.StiffnessMatrix", "assembly.LoadVector", "assembly.LoadFunction",
    "assembly.Quadrature", "assembly.ShapeFunction", "assembly.MapReferenceElement",
    "mesh", "mesh.Mesh1D", "mesh.Mesh2D", "mesh.Element1D",
    "utilities", "utilities.laplacian", "utilities.plots",
]

for _name in _SUBMODULES:
    _mod = importlib.import_module("learnmultigrid_b200." + _name)
    sys.modules[__name__ + "." + _name] = _mod
    if "." not in _name:
        setattr(sys.modules[__name__], _name, _mod)
