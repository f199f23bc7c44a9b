"""B200-native spatial feature memory (drop-in for the memory path of nhcha6/embodied-object-detection).

The directory name carries a hyphen, so import it with
    eod = importlib.import_module("embodied-object-detection_b200")
or through the top-level shim ``import eod_b200``.
"""
from . import _lib, build, config, episodes, formats, fpn_fusion, geometry, memory, ops, runner, sharding  # noqa: F401
from ._lib import EodError  # noqa: F401
from .fpn_fusion import CustomRecurrentFPN, MemoryFusion  # noqa: F401
from .geometry import Projector, compute_intrinsics, transform3d  # noqa: F401
from .memory import EpisodeBatch, HeightMaxBatch, SpatialFeatureMemory  # noqa: F401
from .runner import EpisodeRunner, HostEpisodeProvider, LockStepSchedule  # noqa: F401

__version__ = "0.1.0"
