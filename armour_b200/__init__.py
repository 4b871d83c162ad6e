"""armour_b200 — B200-native reach-set construction and constraint evaluation for the ARMOUR planner.

The compute path is the CUDA library armour_b200/libarmour_b200.so behind the C ABI of
include/armour_b200.h; this package is the thin host-side mirror used by tests and bench.py.
Importing the package loads the shared library and fails loudly when it has not been built.
"""
from . import _lib
from ._lib import ArmourError, NF

_lib.load()  # no CPU fallback: a missing extension is an ImportError here

from .planner import ReachSetEngine  # noqa: E402
from .controller import RobustController  # noqa: E402
from .armtd import ArmtdBatch, ArmtdPlanner  # noqa: E402
from . import worlds  # noqa: E402
from . import sharding  # noqa: E402

__all__ = ["ReachSetEngine", "RobustController", "ArmtdPlanner", "ArmtdBatch", "ArmourError", "NF", "worlds", "sharding"]
