"""B200-native batched NMPC solver behind the reference's CasADi-shaped solver call.

Scope: the hot path of devsonni/MPC-Implementation only -- `sol = solver(x0,lbx,ubx,lbg,ubg,p)`
(Python/NMPC_TT.py:358-365) and the shift-and-apply-first-input loop around it (:13-30, :346-402).
Import as `import b200nmpc` (root shim; this directory's name is not a valid module name).
"""
from . import _ffi, scenarios
from .nlpsol import SolveFunction, Solver, nlpsol
from .scenarios import SCENARIOS, Scenario, random_instances

__all__ = ["nlpsol", "Solver", "SolveFunction", "Scenario", "SCENARIOS", "scenarios", "random_instances", "_ffi"]
