"""The ray-cast LiDAR as the agent's sensor of a stage03 env (TaskConfig(lidar="raycast"), raycast_sphere_kernel) -- needs a B200.

Parity is property-pinned (the reference has no ray cast): with zero radii the env is bit for bit the fused flavour; with
radii it matches the CPU oracle's env flavour (oracle/env_raycast.py) cell by cell, excusing only the cells the oracle
reports as near a decision (f64 build: 1e-9 m, f32 build: 1e-4 m)."""
import numpy as np
import pytest
import torch

from oracle.env_raycast import RaycastEnvOracle
from tests.util import kite_actions, oracle_cfg, oracle_state_dict

pytestmark = pytest.mark.gpu

SCOPE = ["exp02_vFinal", "exp03_vFinal", "exp04_vFinal", "exp02_v2_full", "swarm"]


def _env(name, E, seed, precision="f32", radius=None, sub_batches=0, auto_reset=True, **kw):
    from dronechase_b200 import BatchedThreatEngageEnv, preset
    cfg = preset(name) if radius is None else preset(name, lidar="raycast", ray_radius=radius)
    return BatchedThreatEngageEnv(cfg, n_envs=E, seed=seed, device=0, auto_reset=auto_reset, precision=precision,
                                  with_ids=True, sub_batches=sub_batches, **kw)


def _actions(E, g):
    a = torch.rand(E, 4, generator=g, device="cuda") * 2 - 1
    a[:, 3] = (a[:, 3] + 1) / 2
    return a


def _same_bits(a, b):
    return torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


@pytest.mark.parametrize("sub_batches", [1, 2])
@pytest.mark.parametrize("precision", ["f32", "f64"])
@pytest.mark.parametrize("name", SCOPE)
def test_zero_radii_is_the_fused_sphere(name, precision, sub_batches):
    """Closed loop with auto-reset: obs_lidar and lidar_ids equal the fused flavour's bit for bit at every step (K passes
    max_step, so every env is reset at least once)."""
    E, K = 128, 320
    ray = _env(name, E, 5, precision, (0.0, 0.0), sub_batches)
    fused = _env(name, E, 5, precision, None, sub_batches)
    o1, o2 = ray.reset(), fused.reset()
    g = torch.Generator(device="cuda"); g.manual_seed(3)
    dones = 0
    for t in range(K):
        a = _actions(E, g)
        o1, _, d1, _ = ray.step(a)
        o2, _, d2, _ = fused.step(a)
        assert _same_bits(o1["lidar"], o2["lidar"]), f"step {t}: sphere"
        assert torch.equal(ray.lidar_ids, fused.lidar_ids), f"step {t}: ids"
        assert torch.equal(d1, d2) and _same_bits(o1["inertial_data"], o2["inertial_data"])
        dones += int(d1.sum())
    assert dones > 0, "no episode ended: auto-reset not exercised"
    assert int((o1["lidar"][:, 0] < 1).sum()) > 0


def test_zero_radii_through_step_graph():
    E, K = 256, 80
    ray = _env("exp02_v2_full", E, 9, "f32", (0.0, 0.0), 2)
    fused = _env("exp02_v2_full", E, 9, "f32", None, 2)
    ray.reset(); fused.reset()
    g = torch.Generator(device="cuda"); g.manual_seed(1)
    for t in range(K):
        a = _actions(E, g)
        o1 = ray.step_graph(a)[0]
        o2 = fused.step(a)[0]
        assert _same_bits(o1["lidar"], o2["lidar"]) and torch.equal(ray.lidar_ids, fused.lidar_ids), f"step {t}"


def _compare(got, gid, ref, rid, margin, excuse, tol_rn):
    """Cells of the oracle's margin >= excuse: ids, type and age channels exact, r_n within tol_rn."""
    ok = margin >= excuse
    assert np.array_equal(gid[ok], rid[ok])
    assert np.array_equal(got[1:][:, ok], ref[1:][:, ok])
    assert np.abs(got[0][ok] - ref[0][ok]).max(initial=0.0) <= tol_rn
    return int(ok.sum()), int((~ok).sum())


@pytest.mark.parametrize("radius", [(0.1, 0.1), (0.3, 0.05)])
@pytest.mark.parametrize("name", ["exp02_vFinal", "exp03_vFinal", "exp04_vFinal", "exp02_v2_full"])
def test_closed_loop_f64_against_the_oracle(name, radius):
    E, K = 48, 200
    env = _env(name, E, 11, "f64", radius)
    orc = RaycastEnvOracle(oracle_cfg(name), E, radius, seed=11, auto_reset=True)
    env.reset(); orc.reset()
    rng = np.random.RandomState(3)
    ram_envs = np.arange(E) % 4 == 0
    excused = ray_cells = kept = 0
    prev = None
    for t in range(K):
        a = kite_actions(orc, rng)
        a[ram_envs] = kite_actions(orc, np.random.RandomState(t), ram=True)[ram_envs]
        obs, _, done, _ = env.step(torch.from_numpy(a).cuda())
        ref, _, d_ref, _ = orc.step(a.astype(np.float64))
        assert np.array_equal(done.cpu().numpy().astype(bool), d_ref), f"step {t}: terminated flags"
        got, gid = obs["lidar"].cpu().numpy(), env.lidar_ids.cpu().numpy()
        for e in range(E):
            n_ok, n_ex = _compare(got[e], gid[e], ref["lidar"][e], orc.lidar_ids[e], orc.ray_margin[e], 1e-9, 1e-6)
            excused += n_ex
        ray_cells += int(((gid >= 0).sum(axis=(1, 2)) > np.count_nonzero(orc.armed[:, 1:], axis=1)).sum())
        # an env whose agent is no publisher keeps the sphere of its last update
        if prev is not None:
            for e in np.nonzero(~orc.ray_updated)[0]:
                assert np.array_equal(got[e], prev[e]), f"step {t} env {e}: kept sphere"
                kept += 1
        prev = got
    assert ray_cells > 0, "no env ever showed more marked cells than entities: the bounding spheres never mattered"
    assert kept > 0, "the agent never died: the kept sphere was not exercised"
    assert excused < 1e-4 * E * K * 338


@pytest.mark.parametrize("name", ["exp02_vFinal", "exp02_v2_full"])
def test_teacher_forced_f32_against_the_oracle(name):
    """float32 build: every step starts from the oracle's state; cells within 1e-4 m of a decision are excused."""
    E, K, radius = 64, 60, (0.3, 0.05)
    env = _env(name, E, 21, "f32", radius, auto_reset=False)
    orc = RaycastEnvOracle(oracle_cfg(name), E, radius, seed=21, auto_reset=False)
    env.reset(); orc.reset()
    rng = np.random.RandomState(1)
    n_cmp = 0
    for t in range(K):
        env.set_state(oracle_state_dict(orc))
        a = kite_actions(orc, rng, ram=(t % 3 == 0))
        obs, _, _, _ = env.step(torch.from_numpy(a).cuda())
        orc.min_margin[:] = np.inf
        ref, _, d_ref, _ = orc.step(a.astype(np.float64))
        got, gid = obs["lidar"].cpu().numpy(), env.lidar_ids.cpu().numpy()
        for e in range(E):
            if orc.min_margin[e] > 1e-5 and orc.armed[e, 0]:          # events decided alike and the agent updated
                n_cmp += _compare(got[e], gid[e], ref["lidar"][e], orc.lidar_ids[e], orc.ray_margin[e], 1e-4, 5e-6)[0]
        done_envs = np.nonzero(d_ref)[0]
        if len(done_envs):
            mask = np.zeros(E, dtype=bool); mask[done_envs] = True
            orc.reset(mask)
            env.reset(torch.from_numpy(mask.astype(np.uint8)).cuda())
    assert n_cmp > 0.5 * E * K * 338


def _scene(radius, place):
    """One f64 env at rest whose drones `place` positions (slot -> xyz); the oracle holds the same state."""
    env = _env("exp03_vFinal", 1, 4, "f64", radius, auto_reset=False)
    orc = RaycastEnvOracle(oracle_cfg("exp03_vFinal"), 1, radius, seed=4, auto_reset=False)
    env.reset(); orc.reset()
    for d, p in place.items():
        orc.pos[0, d] = p; orc.imu["position"][0, d] = p; orc.formation[0, d] = p
        orc.armed[0, d] = True
    orc.vel[:] = 0; orc.omega[:] = 0; orc.quat[:] = [0, 0, 0, 1]; orc.imu["quaternion"][:] = [0, 0, 0, 1]
    orc.armed[0, [d for d in range(orc.D) if d not in place]] = False
    env.set_state(oracle_state_dict(orc))
    a = np.array([[0.0, 0.0, 0.0, 0.0]], dtype=np.float32)
    obs = env.step(torch.from_numpy(a).cuda())[0]
    ref = orc.step(a.astype(np.float64))[0]
    got, gid = obs["lidar"].cpu().numpy()[0], env.lidar_ids.cpu().numpy()[0]
    _compare(got, gid, ref["lidar"][0], orc.lidar_ids[0], orc.ray_margin[0], 1e-9, 1e-6)
    return got, gid, orc


def _cell_dir(ti, pj):
    th, ph = (ti + 0.5) / 13 * np.pi, -np.pi + (pj + 0.5) / 26 * 2 * np.pi
    return np.array([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)])


def test_occlusion_built_with_set_state():
    """exp03: agent (slot 0), wingman (slot 1), munitions from slot 2.  A munition straight behind the wingman along a
    cell's centre ray is hidden; with the wingman moved aside it shows again."""
    o = np.array([0.0, 0.0, 5.0])
    d = _cell_dir(6, 3)
    _, gid, _ = _scene((0.3, 0.05), {0: o, 1: o + 2.0 * d, 2: o + 5.0 * d})
    assert gid[6, 3] == 1 and (gid == 2).sum() == 0
    side = np.cross(d, [0.0, 0.0, 1.0]); side /= np.linalg.norm(side)
    _, gid, _ = _scene((0.3, 0.05), {0: o, 1: o + 2.0 * d + 1.0 * side, 2: o + 5.0 * d})
    assert gid[6, 3] == 2


def test_observer_inside_a_bounding_sphere_and_cell_borders():
    o = np.array([0.0, 0.0, 5.0])
    got, gid, _ = _scene((0.5, 0.05), {0: o, 1: o + [0.2, 0.1, 0.0], 2: o + [3.0, 0.0, 0.0]})
    assert (gid == 1).all() and (got[0] == 0).all()


def test_entity_on_a_cell_border():
    """A munition of radius 0 whose snapshot sits on the corner of four cells (theta row border 6, phi column border 20 in
    the agent's frame): only its centre claim marks the sphere, so the cell is decided by the projection at the border,
    and it is the oracle's.  The start position is corrected twice for the drones' motion during the step."""
    from oracle import dynamics as dy
    o = np.array([0.0, 0.0, 5.0])
    th, ph = 6 / 13 * np.pi, -np.pi + 20 / 26 * 2 * np.pi
    b = np.array([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)])
    p0 = o + 2.0 * b
    for it in range(3):
        _, gid, orc = _scene((0.1, 0.0), {0: o, 1: o + [0.0, -3.0, 0.0], 2: p0})
        o1, q1, p1 = orc.imu["position"][0, 0], orc.imu["quaternion"][0, 0], orc.imu["position"][0, 2]
        R = dy.rot_from_quat(q1)
        p0 = p0 + (o1 + R @ (2.0 * b) - p1)                # where the snapshot should have been
    rel = R.T @ (p1 - o1)
    t1, f1 = np.arccos(rel[2] / np.linalg.norm(rel)), np.arctan2(rel[1], rel[0])
    assert abs(t1 - th) < 1e-5 and abs(f1 - ph) < 1e-5, "the snapshot did not land on the cell corner"
    cells = np.argwhere(gid == 2)
    assert len(cells) == 1 and cells[0][0] in (5, 6) and cells[0][1] in (19, 20)
    assert np.array_equal(gid, orc.lidar_ids[0])


def test_set_ray_radii_and_create_refusals():
    """The C ABI's own checks, below the Python config's: dc_set_ray_radii on a fused sim, with a negative / NaN / infinite
    radius, after dc_reset; dc_create of DC_LIDAR_RAYCAST for stage02, for policy-driven wingmen and for eval_task."""
    import ctypes as C
    from dronechase_b200 import _lib
    L = _lib.lib()
    fused = _env("exp03_vFinal", 4, 1)
    assert L.dc_set_ray_radii(fused._sim, 0.1, 0.1) == -1 and b"DC_LIDAR_RAYCAST" in L.dc_last_error()
    ray = _env("exp03_vFinal", 4, 1, radius=(0.1, 0.1))
    for r_lw, r_lm in ((-0.1, 0.1), (0.1, -1e-6), (float("nan"), 0.1), (0.1, float("inf"))):
        assert L.dc_set_ray_radii(ray._sim, r_lw, r_lm) == -1 and b"finite and >= 0" in L.dc_last_error()
    assert L.dc_set_ray_radii(ray._sim, 0.2, 0.05) == 0
    ray.reset()
    assert L.dc_set_ray_radii(ray._sim, 0.2, 0.05) == -1 and b"once dc_reset" in L.dc_last_error()
    for field, value in (("family", 1), ("eval_task", 1), ("lw_driver", 2)):
        c = _lib.dc_config()
        C.memmove(C.byref(c), C.byref(ray._c), C.sizeof(c))
        if field == "lw_driver":
            c.lw_driver[1] = value                          # the second wingman on the behaviour tree
        else:
            setattr(c, field, value)
        sim = C.c_void_p()
        assert L.dc_create(C.byref(c), 0, C.byref(sim)) == -1 and not sim.value, field
        assert b"ray-cast LiDAR is built for the stage03 family" in L.dc_last_error(), field


def test_a_smaller_sim_keeps_a_larger_sims_shared_memory():
    """raycast_sphere_kernel's shared memory grows with the drones per env; its limit is one per process.  A float64 sim of
    204 drones per env needs more than the 48 KB default; creating a 7-drone sim afterwards must not take that away."""
    from dronechase_b200 import BatchedThreatEngageEnv, preset
    big = BatchedThreatEngageEnv(preset("swarm", n_lm=200, initial_round=200, lidar="raycast", ray_radius=(0.3, 0.3)),
                                 n_envs=8, seed=3, device=0, precision="f64", with_ids=True)
    big.reset()
    big.step(torch.zeros(8, 4, device="cuda"))
    small = _env("exp02_vFinal", 8, 3, "f64", (0.1, 0.1))
    small.reset()
    g = torch.Generator(device="cuda"); g.manual_seed(2)
    for _ in range(10):
        big.step(_actions(8, g))
        small.step(_actions(8, g))
    torch.cuda.synchronize()
    assert int((big.lidar_ids >= 0).sum(dim=(1, 2)).min()) > 0, "a sphere of the large sim was not rebuilt"


def test_lidar_ids_bound_4_byte_aligned():
    """dc_buffers.lidar_ids needs 4-byte alignment only: a row that starts 4 bytes past an 8-byte boundary gets the same ids."""
    import ctypes as C
    from dronechase_b200 import _lib
    E = 128
    ref = _env("exp03_vFinal", E, 6, "f32", (0.8, 0.5), 2)
    env = _env("exp03_vFinal", E, 6, "f32", (0.8, 0.5), 2)
    buf = torch.full((E * 338 + 1,), -1, dtype=torch.int32, device="cuda")
    env.lidar_ids = buf[1:].view(E, 13, 26)
    assert env.lidar_ids.data_ptr() % 8 == 4
    env._b.lidar_ids = env.lidar_ids.data_ptr()
    _lib.check(_lib.lib().dc_bind(env._sim, C.byref(env._b)), "dc_bind")
    ref.reset(); env.reset()
    g = torch.Generator(device="cuda"); g.manual_seed(4)
    for t in range(40):
        a = _actions(E, g)
        ref.step(a); env.step(a)
        assert torch.equal(env.lidar_ids, ref.lidar_ids), f"step {t}"
    assert int((env.lidar_ids >= 0).sum()) > E


def test_determinism_and_sub_batch_split_at_65536():
    E, K = 65536, 150
    envs = [_env("exp02_v2_full", E, 7, "f32", (0.1, 0.1), sb) for sb in (1, 2, 2)]
    for env in envs:
        env.reset()
    g = torch.Generator(device="cuda"); g.manual_seed(0)
    for t in range(K):
        a = _actions(E, g)
        outs = [env.step(a) for env in envs]
        for env, (obs, rew, done, info) in zip(envs[1:], outs[1:]):
            ref_obs, ref_rew, ref_done, ref_info = outs[0]
            for k in obs:
                assert _same_bits(obs[k], ref_obs[k]), f"step {t}: {k}"
            assert torch.equal(env.lidar_ids, envs[0].lidar_ids), f"step {t}: ids"
            assert _same_bits(rew, ref_rew) and torch.equal(done, ref_done) and torch.equal(info, ref_info), f"step {t}"
    assert int((envs[0].lidar_ids >= 0).sum()) > 0


@pytest.mark.parametrize("precision", ["3xtf32", "tf32"])
def test_fused_policy_reads_the_raycast_sphere(precision):
    """FusedPolicy takes the ray-cast sphere unchanged: it matches the torch module on the env's own observations."""
    from dronechase_b200.policy import LidarInertialActionPolicy
    TOL = {"3xtf32": 2e-5, "tf32": 5e-3}[precision]
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    env = _env("exp03_vFinal", 777, 2, "f32", (0.8, 0.5))
    obs = env.reset()
    pol = LidarInertialActionPolicy(lidar_channels=3, features_dim=256, pi=(128, 256, 512), seed=4, device="cuda")
    fused = pol.fused(precision)
    for t in range(40):
        want = pol(obs)
        got = fused(obs)
        assert float((got - want).abs().max()) < TOL, f"step {t}"
        obs = env.step(got)[0]
    assert int((obs["lidar"][:, 0] < 1).sum()) > 777
    fused.close()


def test_vec_env_hands_out_the_dense_raycast_sphere():
    from dronechase_b200 import preset
    from dronechase_b200.vec_env import DroneChaseVecEnv
    venv = DroneChaseVecEnv(preset("exp03_vFinal", lidar="raycast", ray_radius=(0.8, 0.5)), n_envs=96, seed=3, device=0,
                            pin_cores=False)
    assert not venv.sparse
    obs = venv.reset()
    rng = np.random.RandomState(0)
    for t in range(30):
        a = np.concatenate([rng.uniform(-1, 1, (96, 3)), rng.uniform(0, 1, (96, 1))], axis=1).astype(np.float32)
        obs, rew, done, infos = venv.step(a)
        torch.cuda.synchronize()
        for k in ("lidar", "inertial_data", "last_action"):
            assert np.array_equal(obs[k], venv.sim.obs[k].cpu().numpy()), f"step {t}: {k}"
    venv.close()
