"""The ray-cast LiDAR as the agent's sensor (TaskConfig(lidar="raycast")) without a GPU: configuration refusals, the C ABI's
new export and struct mirror, and the properties that pin the CPU oracle's env flavour (oracle/env_raycast.py) -- zero radii
give the pinned projection, and away from ties and inside observers it agrees with the stand-alone ray-cast oracle."""
import ctypes as C
from types import SimpleNamespace

import numpy as np
import pytest

from dronechase_b200 import _lib
from dronechase_b200.config import evaluation_preset, preset
from oracle.env_oracle import EnvOracle, N_PHI, N_THETA, lidar_project
from oracle.env_raycast import RaycastEnvOracle, lidar_raycast_env
from oracle.lidar_raycast import lidar_raycast
from tests.util import kite_actions, oracle_cfg

SCOPE = ["exp02_vFinal", "exp03_vFinal", "exp04_vFinal", "exp02_v2_full", "swarm"]


@pytest.mark.parametrize("name", SCOPE)
def test_config_accepts_the_stage03_presets(name):
    cfg = preset(name, lidar="raycast", ray_radius=(0.1, 0.05))
    assert cfg.ray_radius == (0.1, 0.05) and cfg.lidar_channels == 3


@pytest.mark.parametrize("name", ["level5_c1", "level5_fusion", "stage02", "stage01", "exp05_vFinal"])
def test_config_refuses_out_of_scope_presets(name):
    with pytest.raises(ValueError, match="stage03 family without lw_driver / eval_task"):
        preset(name, lidar="raycast", ray_radius=(0.1, 0.1))


def test_config_refuses_evaluation_tasks_and_stray_radii():
    with pytest.raises(ValueError, match="stage03 family without lw_driver / eval_task"):
        evaluation_preset({"drivers": [{"type": "bt"}]}, lidar="raycast", ray_radius=(0.1, 0.1))
    for flavour in ("fused", "classic"):
        with pytest.raises(ValueError, match="ray_radius"):
            preset("exp02_vFinal", lidar=flavour, ray_radius=(0.1, 0.1))


@pytest.mark.parametrize("radius", [None, (0.1,), (-0.1, 0.1), (0.1, -1e-9), (float("nan"), 0.1), (0.1, float("inf"))])
def test_config_refuses_missing_or_bad_radii(radius):
    with pytest.raises(ValueError, match="ray_radius"):
        preset("exp02_vFinal", lidar="raycast", ray_radius=radius)


def test_hit_list_consumers_refuse_raycast():
    from dronechase_b200 import BatchedThreatEngageEnv
    from dronechase_b200.vec_env import DroneChaseVecEnv
    from dronechase_b200.rollout import DeviceRollout, PPORollout
    cfg = preset("exp02_v2_full", lidar="raycast", ray_radius=(0.1, 0.1))
    with pytest.raises(ValueError, match="cannot describe a ray-cast sphere"):
        BatchedThreatEngageEnv(cfg, n_envs=4, with_hits=True)
    fake = SimpleNamespace(cfg=cfg, lidar_hits=None)
    for cls in (DeviceRollout, PPORollout):
        with pytest.raises(_lib.DroneChaseError, match="cannot describe a ray-cast sphere"):
            cls(fake, 4)
    for kw in ({"pairs_lidar": True}, {"mapped_lidar": True}):
        with pytest.raises(ValueError, match="moves the sphere dense"):
            DroneChaseVecEnv(cfg, n_envs=4, **kw)


def test_set_ray_radii_argument_checks():
    L = _lib.lib()
    assert L.dc_set_ray_radii(None, 0.1, 0.1) == -1          # DC_ERR_ARG
    assert b"null sim" in L.dc_last_error()


def test_abi_mirror_unchanged():
    L = _lib.lib()
    assert L.dc_abi_info(0) == 10 == _lib.DC_ABI_VERSION
    assert L.dc_abi_info(1) == C.sizeof(_lib.dc_config)
    assert L.dc_abi_info(2) == C.sizeof(_lib.dc_buffers)


# attitudes whose float32 quaternion is exactly unit: the rotation matrix is then exactly orthonormal, and the world-frame
# test of oracle.lidar_raycast and the body-frame one of the env flavour see the same geometry
UNIT_Q = [(0, 0, 0, 1), (1, 0, 0, 0), (0, 1, 0, 0), (0, 0, 1, 0), (0.5, 0.5, 0.5, 0.5), (0.5, -0.5, 0.5, -0.5),
          (-0.5, 0.5, 0.5, 0.5), (0.5, 0.5, -0.5, 0.5), (0.5, 0.5, 0.5, -0.5), (-0.5, -0.5, 0.5, 0.5)]


def _scene(rng, n, exact_q=False):
    own = rng.uniform(-3, 3, 3)
    q = rng.normal(size=4); q /= np.linalg.norm(q)
    if exact_q:
        q = np.array(UNIT_Q[rng.randint(len(UNIT_Q))], dtype=np.float64)
    ents = own + rng.uniform(-6, 6, (n, 3))
    types = [3 if k < 2 else 1 for k in range(n)]
    return own, q, ents, types, list(range(1, n + 1))


def test_zero_radii_is_the_fused_projection():
    rng = np.random.RandomState(0)
    for _ in range(200):
        own, q, ents, types, ids = _scene(rng, rng.randint(1, 12))
        s_ref, i_ref = lidar_project(own, q, ents, types, ids, "fused", 40.0)
        s, i, _ = lidar_raycast_env(own, q, ents, types, ids, [0.0] * len(ids), 40.0)
        assert np.array_equal(i, i_ref)
        assert np.array_equal(s.view(np.int32), s_ref.view(np.int32))


def test_agrees_with_the_standalone_raycast_oracle():
    """Observer outside every bounding sphere: the env flavour's sphere is lidar_raycast's wherever neither is near a
    decision (radii exactly representable in float32, so both use the same spheres)."""
    rng = np.random.RandomState(1)
    compared = marked = 0
    for _ in range(60):
        own, q, ents, types, ids = _scene(rng, rng.randint(1, 10), exact_q=True)
        radii = rng.choice([0.25, 0.5, 1.0, 1.5], len(ids))
        if (np.linalg.norm(ents.astype(np.float32) - own.astype(np.float32), axis=1) <= radii + 1e-3).any():
            continue
        s, i, m = lidar_raycast_env(own, q, ents, types, ids, radii, 40.0)
        s_ref, i_ref, m_ref = lidar_raycast(own, q, ents, radii, types, ids, 40.0)
        ok = (m > 1e-6) & (m_ref > 1e-6)
        assert np.array_equal(i[ok], i_ref[ok])
        assert np.abs(s[:, ok] - s_ref[:, ok]).max() <= 1e-6
        compared += int(ok.sum()); marked += int((i[ok] >= 0).sum())
    assert compared > 10000 and marked > 500


def test_observer_inside_a_sphere_sees_it_everywhere():
    own, q = np.zeros(3), np.array([0.0, 0.0, 0.0, 1.0])
    ents = np.array([[0.2, 0.1, 0.0], [3.0, 0.0, 0.0]])
    s, i, _ = lidar_raycast_env(own, q, ents, [3, 1], [1, 5], [0.5, 0.1], 40.0)
    assert (i == 1).all() and (s[0] == 0).all() and np.allclose(s[1], 0.6) and np.allclose(s[2], 0.1)


def test_occlusion_along_a_cell_ray():
    """A munition straight behind a wingman on the centre ray of a cell is hidden there; moved aside, it reappears."""
    own, q = np.zeros(3), np.array([0.0, 0.0, 0.0, 1.0])
    ti, pj = 6, 20
    th, ph = (ti + 0.5) / N_THETA * np.pi, -np.pi + (pj + 0.5) / N_PHI * 2 * np.pi
    d = np.array([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)])
    ents = np.array([2.0 * d, 5.0 * d])
    _, i, _ = lidar_raycast_env(own, q, ents, [3, 1], [1, 4], [0.3, 0.1], 40.0)
    assert i[ti, pj] == 1 and (i == 4).sum() == 0
    side = np.cross(d, [0.0, 0.0, 1.0]); side /= np.linalg.norm(side)
    ents[0] += 0.9 * side
    _, i, _ = lidar_raycast_env(own, q, ents, [3, 1], [1, 4], [0.3, 0.1], 40.0)
    assert i[ti, pj] == 4


@pytest.mark.parametrize("name", ["exp02_vFinal", "exp03_vFinal"])
def test_zero_radii_oracle_closed_loop_is_the_fused_oracle(name):
    E, K = 4, 40
    a_orc = EnvOracle(oracle_cfg(name), E, seed=3, auto_reset=True)
    b_orc = RaycastEnvOracle(oracle_cfg(name), E, (0.0, 0.0), seed=3, auto_reset=True)
    a_orc.reset(); b_orc.reset()
    rng = np.random.RandomState(5)
    for _ in range(K):
        act = kite_actions(a_orc, rng)
        ra = a_orc.step(act.astype(np.float64))[0]
        rb = b_orc.step(act.astype(np.float64))[0]
        assert np.array_equal(ra["lidar"].view(np.int32), rb["lidar"].view(np.int32))
        assert np.array_equal(a_orc.lidar_ids, b_orc.lidar_ids)
