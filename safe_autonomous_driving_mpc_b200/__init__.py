"""Import shim: the product package lives in the directory ``safe-autonomous-driving-mpc_b200/`` (the name
the build contract fixes; a hyphen cannot be imported), so this package only points ``__path__`` there."""
import os as _os

__path__.insert(0, _os.path.join(_os.path.dirname(_os.path.dirname(_os.path.abspath(__file__))),
                                 "safe-autonomous-driving-mpc_b200"))

from .tracker import BatchedTracker, TrajectoryLoader, TrackerParams  # noqa: E402,F401
from .environment import ObstaclesFSM, run_simulation  # noqa: E402,F401
from .planner import PlannerEvaluator  # noqa: E402,F401
from . import planner_driver  # noqa: E402,F401
from .simulation import BatchedSimulation, make_scenario, FLEET_SOLVER_CAPS  # noqa: E402,F401
from . import rare_events  # noqa: E402,F401
from . import _lib, sharding  # noqa: E402,F401
