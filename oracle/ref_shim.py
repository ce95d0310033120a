"""ORACLE (test infrastructure): import the UNMODIFIED reference hot-path classes from
/root/reference in this container, with FEniCS/PETSc/matplotlib replaced by empty stand-ins.

Used only by tests/golden/make_golden.py, which regenerates the golden fixtures the tests
compare against.  No test and nothing under generative-physics-informed-pde_b200/ imports this.

Recipe = SURVEY.md Appendix B: the classes on the hot path (bottleneck/ROM.py,
bottleneck/components.py:260-323, bottleneck/VirtualObservables.py) are pure
torch/numpy/scipy; only their *constructors from FEniCS objects* are not runnable.
"""
import os
import sys
import types

import numpy as np
import torch

REFERENCE_ROOT = os.environ.get("GPDE_REFERENCE_ROOT", "/root/reference")


def available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "bottleneck", "ROM.py"))


class _Dummy(object):
    def __init__(self, *a, **k):
        pass


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


_loaded = {}


def load():
    """Returns a dict with the reference modules ROM, components, VirtualObservables."""
    if _loaded:
        return _loaded
    if not available():
        raise RuntimeError("reference tree not present at %s" % REFERENCE_ROOT)
    dummies = dict(UserExpression=_Dummy, SubDomain=_Dummy, DirichletBC=_Dummy, Cell=_Dummy,
                   Function=_Dummy, Expression=_Dummy, plot=lambda *a, **k: None)
    for name in ("fenics", "dolfin"):
        if name not in sys.modules:
            _stub(name, **dummies)
    if "petsc4py" not in sys.modules:
        p = _stub("petsc4py")
        p.PETSc = _stub("petsc4py.PETSc")
    try:
        import matplotlib  # noqa: F401
    except Exception:
        mpl = _stub("matplotlib")
        mpl.pyplot = _stub("matplotlib.pyplot", switch_backend=lambda *a, **k: None)
    # removed-API shims (SURVEY.md Appendix B.2)
    if not hasattr(torch, "solve") or True:
        torch.solve = lambda B, A: (torch.linalg.solve(A, B), None)
    if not hasattr(np, "int"):
        np.int = int
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import importlib
    _loaded["ROM"] = importlib.import_module("bottleneck.ROM")
    _loaded["components"] = importlib.import_module("bottleneck.components")
    _loaded["VirtualObservables"] = importlib.import_module("bottleneck.VirtualObservables")
    return _loaded


class PhysicsLike(object):
    """What ROM.__init__ needs from a LinearEllipticPhysics (bottleneck/ROM.py:14-15) and what
    QuerryPoint needs (VirtualObservables.py:12-15, 52-59): dof sets, Vc.dim(), dim_out,
    assemble_system."""

    class _Vc(object):
        def __init__(self, n):
            self._n = n

        def dim(self):
            return self._n

    def __init__(self, constrained_dofs, free_dofs, num_cells, assemble_system=None):
        self.constrained_dofs = np.asarray(constrained_dofs)
        self.free_dofs = np.asarray(free_dofs)
        self.Vc = PhysicsLike._Vc(num_cells)
        self._assemble = assemble_system

    @property
    def dim_out(self):
        return self.free_dofs.size

    def assemble_system(self, x, bc=None, only_free_dofs=True):
        return self._assemble(x, bc)
