"""ctypes binding of the C ABI in include/dronechase_b200.h.

The CUDA extension is the product: if the shared library is missing this module raises --
there is no CPU or PyTorch fallback (build it with ``python -c "import __graft_entry__ as g; g.build()"``).
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libdronechase_b200.so")

DC_ABI_VERSION = 10
DC_QUAD_PARAM_WORDS = 88
DC_INFO_WORDS = 8
DC_STATE_QUADS = 13
DC_ENV_WORDS = 16
N_THETA, N_PHI = 13, 26
DC_LIDAR_STACK = 6


class dc_config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "abi_version", "n_envs", "n_lw", "n_lm", "munition", "step_increment", "max_step", "initial_round",
        "substeps", "lm_nav", "ally_mode", "reward", "lidar", "fixed_lw_spawn", "auto_reset", "precision",
        "env_offset", "family")] + [("seed", C.c_uint64)] + [(n, C.c_double) for n in (
            "dome_radius", "born_radius", "lw_spawn_radius", "explosion_range", "shoot_range", "cooldown_steps",
            "fire_probability", "lm_speed", "bt_speed", "ally_stop_mag", "vel_bonus")] + [
        ("building", C.c_double * 3), ("quad", C.c_double * DC_QUAD_PARAM_WORDS),
        ("respawn_r_min", C.c_double), ("respawn_r_max", C.c_double), ("support_munition", C.c_int32),
        ("initial_invaders", C.c_int32), ("invaders_per_round", C.c_int32), ("max_rounds", C.c_int32),
        ("sub_batches", C.c_int32), ("level5_base_env", C.c_int32), ("level5_multi_obs", C.c_int32),
        ("lw_driver", C.c_int32 * 8), ("eval_task", C.c_int32), ("time_is_limited", C.c_int32)]


class dc_buffers(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "actions", "obs_lidar", "obs_inertial", "obs_last_action", "reward", "done", "info", "lidar_ids",
        "term_inertial", "term_last_action", "stats", "obs_mask", "lidar_hits", "student_lidar", "student_mask",
        "student_hits", "mo_lidar", "mo_mask", "mo_inertial", "mo_last_action", "mo_present", "mo_hits",
        "lw_actions", "lw_lidar", "lw_inertial", "lw_present", "lw_info")]


class dc_policy_weights(C.Structure):
    _F = C.POINTER(C.c_float)
    _fields_ = [("lidar_channels", C.c_int32), ("features_dim", C.c_int32), ("n_pi", C.c_int32), ("pi", C.c_int32 * 8),
                ("activation", C.c_int32), ("conv1_w", _F), ("conv1_b", _F), ("conv2_w", _F), ("conv2_b", _F),
                ("inertial_w", _F * 3), ("inertial_b", _F * 3), ("action_w", _F * 3), ("action_b", _F * 3),
                ("final_w", _F), ("final_b", _F), ("pi_w", _F * 8), ("pi_b", _F * 8), ("head_w", _F), ("head_b", _F),
                ("low", C.c_float * 4), ("high", C.c_float * 4)]


class dc_value_weights(C.Structure):
    _F = C.POINTER(C.c_float)
    _fields_ = [("n_vf", C.c_int32), ("vf", C.c_int32 * 8), ("vf_w", _F * 8), ("vf_b", _F * 8), ("value_w", _F), ("value_b", _F),
                ("log_std", _F)]


class DroneChaseError(RuntimeError):
    pass


_lib = None


def lib():
    """Load libdronechase_b200.so once; fail loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DroneChaseError(
            f"{LIB_PATH} is missing: build the CUDA extension first (__graft_entry__.build()); "
            "dronechase_b200 has no CPU fallback")
    L = C.CDLL(LIB_PATH)
    L.dc_create.argtypes = [C.POINTER(dc_config), C.c_int, C.POINTER(C.c_void_p)]
    L.dc_bind.argtypes = [C.c_void_p, C.POINTER(dc_buffers)]
    L.dc_reset.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
    L.dc_step.argtypes = [C.c_void_p, C.c_void_p]
    L.dc_set_actions.argtypes = [C.c_void_p, C.c_void_p]
    L.dc_lw_observe.argtypes = [C.c_void_p, C.c_void_p]
    L.dc_lw_observe.restype = C.c_int
    L.dc_note_graph_replay.argtypes = [C.c_void_p]
    L.dc_note_graph_replay.restype = C.c_int
    L.dc_set_ray_radii.argtypes = [C.c_void_p, C.c_float, C.c_float]
    L.dc_set_ray_radii.restype = C.c_int
    L.dc_scatter_hits.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    L.dc_scatter_hits.restype = C.c_int
    L.dc_scatter_stack.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p]
    L.dc_scatter_stack.restype = C.c_int
    L.dc_abi_info.argtypes = [C.c_int]
    L.dc_abi_info.restype = C.c_size_t
    got = (L.dc_abi_info(0), L.dc_abi_info(1), L.dc_abi_info(2))
    want = (DC_ABI_VERSION, C.sizeof(dc_config), C.sizeof(dc_buffers))
    if got != want:          # a stale .so or a hand-mirrored struct out of step with include/dronechase_b200.h
        raise DroneChaseError(f"{LIB_PATH}: ABI (version, sizeof dc_config, sizeof dc_buffers) = {got}, this binding expects "
                              f"{want}; rebuild the extension (__graft_entry__.build(force=True))")
    L.dc_destroy.argtypes = [C.c_void_p]
    L.dc_destroy.restype = None
    L.dc_last_error.restype = C.c_char_p
    L.dc_copy_state.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_int]
    L.dc_state_bytes.argtypes = [C.c_void_p, C.c_int]
    L.dc_state_bytes.restype = C.c_size_t
    L.dc_lidar_project.argtypes = [C.c_void_p] * 5 + [C.c_int32] * 4 + [C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
    L.dc_lidar_raycast.argtypes = [C.c_void_p] * 6 + [C.c_int32] * 3 + [C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
    L.dc_lidar_raycast.restype = C.c_int
    L.dc_launch_count.restype = C.c_uint64
    L.dc_host_scatter_sphere.argtypes = [C.c_void_p] * 3 + [C.c_int32] * 5
    L.dc_host_scatter_sphere.restype = C.c_int
    L.dc_host_scatter_stack.argtypes = [C.c_void_p] * 3 + [C.c_int32] * 3
    L.dc_host_scatter_stack.restype = C.c_int
    L.dc_host_register.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]
    L.dc_host_register.restype = C.c_int
    L.dc_host_unregister.argtypes = [C.c_void_p]
    L.dc_host_unregister.restype = C.c_int
    L.dc_mirror_hits.argtypes = [C.c_void_p, C.c_void_p] + [C.c_int32] * 4 + [C.c_void_p, C.c_void_p]
    L.dc_mirror_hits.restype = C.c_int
    L.dc_diff_hits.argtypes = [C.c_void_p, C.c_void_p] + [C.c_int32] * 4 + [C.c_void_p, C.c_void_p]
    L.dc_diff_hits.restype = C.c_int
    L.dc_host_apply_pairs.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32]
    L.dc_host_apply_pairs.restype = C.c_int
    L.dc_policy_create.argtypes = [C.POINTER(dc_policy_weights), C.c_int, C.POINTER(C.c_void_p)]
    L.dc_policy_create.restype = C.c_int
    L.dc_policy_forward.argtypes = [C.c_void_p] * 4 + [C.c_int64, C.c_void_p, C.c_int32, C.c_void_p]
    L.dc_policy_forward.restype = C.c_int
    L.dc_policy_create_ac.argtypes = [C.POINTER(dc_policy_weights), C.POINTER(dc_value_weights), C.c_int, C.POINTER(C.c_void_p)]
    L.dc_policy_create_ac.restype = C.c_int
    L.dc_policy_act.argtypes = ([C.c_void_p] * 4 + [C.c_int64, C.c_uint64, C.c_int64, C.c_uint32, C.c_int32] + [C.c_void_p] * 4
                                + [C.c_int32, C.c_void_p])
    L.dc_policy_act.restype = C.c_int
    L.dc_gae.argtypes = [C.c_void_p] * 4 + [C.c_int64, C.c_int64, C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
    L.dc_gae.restype = C.c_int
    L.dc_policy_serve.argtypes = [C.c_void_p] * 4 + [C.c_int32, C.c_int32, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]
    L.dc_policy_serve.restype = C.c_int
    L.dc_policy_destroy.argtypes = [C.c_void_p]
    L.dc_policy_destroy.restype = None
    L.dc_quad_is_builtin.argtypes = [C.c_void_p]
    L.dc_quad_is_builtin.restype = C.c_int
    for f in (L.dc_create, L.dc_bind, L.dc_reset, L.dc_step, L.dc_set_actions, L.dc_copy_state, L.dc_lidar_project):
        f.restype = C.c_int
    _lib = L
    return L


EXPORTS = ("dc_create", "dc_bind", "dc_reset", "dc_step", "dc_set_actions", "dc_note_graph_replay", "dc_destroy", "dc_last_error", "dc_copy_state",
           "dc_state_bytes", "dc_lidar_project", "dc_lidar_raycast", "dc_launch_count", "dc_host_scatter_sphere", "dc_host_scatter_stack", "dc_scatter_hits",
           "dc_scatter_stack", "dc_abi_info", "dc_host_register", "dc_host_unregister", "dc_mirror_hits", "dc_lw_observe", "dc_quad_is_builtin", "dc_diff_hits", "dc_host_apply_pairs",
           "dc_policy_create", "dc_policy_forward", "dc_policy_destroy", "dc_policy_create_ac", "dc_policy_act", "dc_gae", "dc_policy_serve", "dc_set_ray_radii")


def check(code: int, what: str):
    if code != 0:
        raise DroneChaseError(f"{what} failed ({code}): {lib().dc_last_error().decode()}")
