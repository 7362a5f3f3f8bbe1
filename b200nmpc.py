"""Import shim: `import b200nmpc` loads the package kept in ./mpc-implementation_b200/ (whose directory
name, fixed by the project layout, is not a valid Python identifier)."""
import importlib.util
import sys
from pathlib import Path

_PKG_DIR = Path(__file__).resolve().parent / "mpc-implementation_b200"
_NAME = "mpc_implementation_b200"

if _NAME not in sys.modules:
    _spec = importlib.util.spec_from_file_location(_NAME, _PKG_DIR / "__init__.py",
                                                   submodule_search_locations=[str(_PKG_DIR)])
    _mod = importlib.util.module_from_spec(_spec)
    sys.modules[_NAME] = _mod
    _spec.loader.exec_module(_mod)
_pkg = sys.modules[_NAME]

nlpsol = _pkg.nlpsol
Solver = _pkg.Solver
SolveFunction = _pkg.SolveFunction
Scenario = _pkg.Scenario
SCENARIOS = _pkg.SCENARIOS
scenarios = _pkg.scenarios
random_instances = _pkg.random_instances
_ffi = _pkg._ffi

# closed-loop drivers (need torch + a GPU at call time, not at import time)
from mpc_implementation_b200.closed_loop import ClosedLoop, PipelinedClosedLoop  # noqa: E402
