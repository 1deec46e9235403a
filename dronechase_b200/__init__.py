"""dronechase_b200 -- B200-native batched simulator for the per-step hot path of
DaviGuanabara/dronechase's threatengage stage03 environments (see DESIGN.md)."""
from .config import CF2X, PRESETS, TaskConfig, calculate_rounds, preset, quad_param_vector  # noqa: F401
from ._lib import DroneChaseError, LIB_PATH  # noqa: F401


def __getattr__(name):
    if name in ("BatchedThreatEngageEnv", "lidar_project", "lidar_raycast", "INFO_KEYS"):
        from . import sim
        return getattr(sim, name)
    if name in ("DeviceRollout", "PPORollout"):
        from . import rollout
        return getattr(rollout, name)
    if name in ("DatasetWriter", "MultiFileDataset", "IOData", "collect_data", "collect_data_multiobs"):
        from . import io_data
        return getattr(io_data, name)
    if name in ("LidarInertialActionPolicy", "LidarInertialActorCritic"):
        from . import policy
        return getattr(policy, name)
    if name == "VecMonitor":
        from .vec_monitor import VecMonitor
        return VecMonitor
    if name == "evaluate_2bt":
        from .evaluation import evaluate_2bt
        return evaluate_2bt
    raise AttributeError(name)
