"""Policy-driven wingmen served by the fused policy kernel (``FusedPolicy.serve`` / ``dc_policy_serve``, the serve
instantiation of csrc/policy_kernel.cu) on a B200:

  * bit identity with ``dc_policy_forward`` on contiguous copies of the slot, for every 3-channel network shape of
    tests/test_gpu_policy.py, both precisions, n_lw 1..3, every slot, ragged batch sizes; last_action afterwards is
    ``torch.where(present, a, last_action_before)`` bit for bit, and nothing else is written;
  * closed loops over the simulator with auto-reset on two presets with policy-driven wingmen (a level4 evaluation
    configuration with two "nn" drivers, exp05_vFinal): ``TaskDrivers`` over fused policies against ``TaskDrivers`` over
    the same kernels on contiguous copies (every output bit-identical at every step), and against the torch module.

Tolerances against the float32 module (absolute, on the clipped mean action): 2e-5 for "3xtf32", 5e-3 for "tf32"."""
import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = {"3xtf32": 2e-5, "tf32": 5e-3}
# (features_dim, pi, activation) of every 3-channel network of tests/test_gpu_policy.py
SHAPES = [(256, (128, 256, 512), "tanh"), (192, (), "tanh"), (256, (256, 256, 256), "relu"), (256, (192, 320), "tanh"),
          (192, (256, 64), "tanh"), (256, (64,) * 7 + (960,), "tanh")]


def _policy(features_dim=256, pi=(128, 256, 512), activation="tanh", seed=4, scale=1.6):
    from dronechase_b200.policy import LidarInertialActionPolicy
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False               # the module is the float32 reference
    pol = LidarInertialActionPolicy(lidar_channels=3, features_dim=features_dim, pi=pi, activation=activation, seed=seed, device="cuda")
    with torch.no_grad():
        for p in pol.parameters():
            p.mul_(scale)
    return pol


def _bits(t):
    return t.contiguous().view(torch.int32) if t.dtype == torch.float32 else t


def _same(a, b):
    return a.shape == b.shape and torch.equal(_bits(a), _bits(b))


def _slabs(E, n_lw, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    lidar = torch.rand(E, n_lw, 3, 13, 26, generator=g, device="cuda")
    lidar[lidar > 0.25] = 1.0                              # mostly empty spheres, like the simulator's
    return {"lidar": lidar, "inertial_data": torch.rand(E, n_lw, 15, generator=g, device="cuda") * 2 - 1,
            "present": torch.rand(E, n_lw, generator=g, device="cuda") < 0.6}


def _check_serve(fused, n_lw, slot, E, full, g):
    """serve on the first E rows of larger slabs: slot `slot` of lw_actions and last_action as dc_policy_forward + where."""
    lw = {k: v[:E] for k, v in full.items()}
    rows = full["lidar"].shape[0]
    last = torch.rand(rows, 4, generator=g, device="cuda")
    acts = torch.rand(rows, n_lw, 4, generator=g, device="cuda")
    last0, acts0 = last.clone(), acts.clone()
    fused.serve(lw, slot, last[:E], acts[:E])
    want = fused({"lidar": lw["lidar"][:, slot].contiguous(), "inertial_data": lw["inertial_data"][:, slot].contiguous(),
                  "last_action": last0[:E]})
    tag = f"n_lw={n_lw} slot={slot} E={E}"
    assert _same(acts[:E, slot], want), f"{tag}: lw_actions[:, slot] differs from dc_policy_forward"
    assert _same(last[:E], torch.where(lw["present"][:, slot, None], want, last0[:E])), f"{tag}: last_action"
    others = [s for s in range(n_lw) if s != slot]
    assert _same(acts[:, others], acts0[:, others]) and _same(acts[E:], acts0[E:]) and _same(last[E:], last0[E:]), \
        f"{tag}: a row or slot outside the call was written"
    return want


@pytest.mark.parametrize("precision", ["3xtf32", "tf32"])
@pytest.mark.parametrize("features_dim,pi,activation", SHAPES)
def test_serve_is_bit_identical_to_the_plain_kernel(precision, features_dim, pi, activation):
    fused = _policy(features_dim, pi, activation).fused(precision)
    g = torch.Generator(device="cuda").manual_seed(7)
    for n_lw in (1, 2, 3):
        full = _slabs(4098, n_lw, seed=n_lw)
        for slot in range(n_lw):
            for E in (1, 63, 64, 65, 4097):
                want = _check_serve(fused, n_lw, slot, E, full, g)
    p = full["present"][:4097, 2]
    assert bool(p.any()) and not bool(p.all()), "vacuous: present is constant"
    assert float(want.std()) > 0.05 and bool((want.abs() < 1).any()), "vacuous: every action clipped"
    fused.close()


def test_serve_on_an_actor_critic_policy():
    """dc_policy_serve runs on a policy made by dc_policy_create_ac as on one made by dc_policy_create."""
    from dronechase_b200.policy import LidarInertialActorCritic
    ac = LidarInertialActorCritic(seed=3, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(1)
    for precision in ("3xtf32", "tf32"):
        fused = ac.fused(precision)
        full = _slabs(1001, 2, seed=5)
        for slot in (0, 1):
            _check_serve(fused, 2, slot, 1000, full, g)
        fused.close()


def test_serve_refuses_bad_arguments():
    from dronechase_b200 import _lib
    fused = _policy(pi=(128,)).fused()
    E = 70
    lw = _slabs(E, 2, seed=0)
    last, acts = torch.zeros(E, 4, device="cuda"), torch.zeros(E, 2, 4, device="cuda")
    for slot in (2, -1):
        with pytest.raises(_lib.DroneChaseError, match=r"slot must lie in \[0, n_lw\)"):
            fused.serve(lw, slot, last, acts)
    from dronechase_b200.policy import LidarInertialActionPolicy
    two = LidarInertialActionPolicy(lidar_channels=2, features_dim=128, pi=(64,), seed=0, device="cuda").fused()
    with pytest.raises(_lib.DroneChaseError, match="lidar_channels must be 3"):
        two.serve(lw, 0, last, acts)
    strided = lw["lidar"].transpose(0, 1).contiguous().transpose(0, 1)      # [E, n_lw, ...] values, not contiguous
    assert torch.equal(strided, lw["lidar"]) and not strided.is_contiguous()
    bad = [({**lw, "lidar": strided}, last, acts), ({**lw, "inertial_data": lw["inertial_data"].double()}, last, acts),
           ({**lw, "present": lw["present"].float()}, last, acts), (lw, last.half(), acts), (lw, last, acts[:, :, :3].contiguous()),
           (lw, last[:E - 1], acts), ({**lw, "lidar": lw["lidar"][:, :, :2].contiguous()}, last, acts),
           ({k: v.cpu() for k, v in lw.items()}, last, acts)]
    for l_, la, ac in bad:
        with pytest.raises(ValueError):
            fused.serve(l_, 0, la, ac)
    torch.cuda.synchronize()
    assert not bool(last.any()) and not bool(acts.any()), "a refused call wrote"
    fused.close(); two.close()


# ------------------------------------------------------------------------------------------------ closed loops
def _wingman_env(name, E, seed):
    """eval_2nn: six munitions at once, born 3 m out, episodes of 121 steps at most."""
    from dronechase_b200 import BatchedThreatEngageEnv, preset
    from dronechase_b200.config import evaluation_preset
    if name == "eval_2nn":
        cfg = evaluation_preset({"drivers": [{"type": "nn", "name": "nn_1"}, {"type": "nn", "name": "nn_2"}], "ENEMY_BORN_RADIUS": 3,
                                 "INITIAL_ROUND": 6, "TIME_IS_LIMITED": True, "MAX_STEP": 120, "STEP_INCREMENT": 0})
    else:
        cfg = preset("exp05_vFinal")
    return BatchedThreatEngageEnv(cfg, n_envs=E, seed=seed, device=0, auto_reset=True)


def _agent_actions(E, seed):
    """exp05's agent (slot 0, the env's action): a fixed direction per env at full speed -- down into the ground, out of the
    dome: its episodes end.  The evaluation task ignores the env's action."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    d = torch.randn(E, 3, generator=g, device="cuda")
    d = d / d.norm(dim=1, keepdim=True)
    return torch.cat([d, torch.ones(E, 1, device="cuda")], dim=1).contiguous()


def _wingman_policy(seed):
    """A random network whose speed command (action[3]) is mostly clipped to 0: its wingman stays near its spawn point, where
    the munitions (which chase the nearest wingman at 0.4 of full speed) reach it -- wingmen die mid-episode."""
    pol = _policy(seed=seed)
    with torch.no_grad():
        pol.action_net.bias[3] -= 1.0
    return pol


CLOSED = [(n, p) for n in ("eval_2nn", "exp05") for p in ("3xtf32", "tf32")]


@pytest.mark.parametrize("name,precision", CLOSED, ids=[f"{n}-{p}" for n, p in CLOSED])
def test_closed_loop_serve_matches_the_kernel_on_copies(name, precision):
    """Two envs, same seed: TaskDrivers over FusedPolicy (-> serve) and over lambda obs: fused(contiguous copies) (-> the
    generic path).  Every output is bit-identical at every step of 200, with auto-reset."""
    from dronechase_b200.drivers import TaskDrivers
    E, K = 256, 200
    env_a, env_b = _wingman_env(name, E, seed=11), _wingman_env(name, E, seed=11)
    slots = env_a.cfg.policy_slots
    fused = {j: _wingman_policy(seed=20 + j).fused(precision) for j in slots}         # different weights per slot
    copies = {j: (lambda f: lambda obs: f({k: v.contiguous() for k, v in obs.items()}))(fused[j]) for j in slots}
    drv_a, drv_b = TaskDrivers(env_a, fused), TaskDrivers(env_b, copies)
    env_a.reset(); drv_a.reset(); env_b.reset(); drv_b.reset()
    chain = drv_a.last_action
    actions = _agent_actions(E, seed=3)
    resets = deaths = carried = both = 0
    seen_present = set()
    prev_present = prev_done = None
    for t in range(K):
        before = drv_a.last_action.clone()
        out_a, out_b = drv_a.step(actions), drv_b.step(actions)
        tag = f"{name} {precision} step {t}"
        obs_a, obs_b = out_a[0], out_b[0]
        for k in obs_a:
            assert _same(obs_a[k], obs_b[k]), f"{tag}: obs[{k}]"
        for i, what in ((1, "reward"), (2, "done"), (3, "info")):
            assert _same(out_a[i], out_b[i]), f"{tag}: {what}"
        for k in env_a.lw_obs:
            assert _same(env_a.lw_obs[k], env_b.lw_obs[k]), f"{tag}: lw_obs[{k}]"
        assert _same(env_a.lw_actions, env_b.lw_actions), f"{tag}: lw_actions"
        assert _same(env_a.lw_info, env_b.lw_info), f"{tag}: lw_info"
        assert _same(drv_a.last_action, drv_b.last_action), f"{tag}: last_action"
        # vacuity: episodes end, policy-driven wingmen die mid-episode, present varies, the chain carries actions
        present = env_a.lw_obs["present"][:, list(slots)]
        done = env_a.done.bool()
        resets += int(done.sum())
        seen_present |= set(present.flatten().tolist())
        if prev_present is not None:
            deaths += int((prev_present & ~present & ~prev_done[:, None]).sum())
        carried += int((before.ne(0).any(1) & present[:, 0]).sum())          # the first slot read a carried action
        if len(slots) > 1:
            both += int((present[:, 0] & present[:, 1]).sum())             # the second slot read the first one's action
        prev_present, prev_done = present, done
    assert drv_a.last_action is chain, "TaskDrivers rebound its last_action"
    print(f"{name} {precision}: resets {resets}, wingman deaths {deaths}, carried {carried}, both served {both}")
    assert resets > 0 and deaths > 0 and seen_present == {True, False} and carried > 0, (resets, deaths, seen_present, carried)
    assert len(slots) == 1 or both > 0
    for f in fused.values():
        f.close()
    env_a.close(); env_b.close()


@pytest.mark.parametrize("name,precision", CLOSED, ids=[f"{n}-{p}" for n, p in CLOSED])
def test_closed_loop_serve_against_the_module(name, precision):
    """The same loop on one env with serve; at every step the torch float32 module, evaluated on the observation each slot
    was served (its rows of the wingman slabs, the chain as that slot saw it), agrees within the precision's tolerance."""
    from dronechase_b200.drivers import TaskDrivers
    E, K = 256, 200
    env = _wingman_env(name, E, seed=13)
    slots = env.cfg.policy_slots
    mods = {j: _wingman_policy(seed=30 + j) for j in slots}
    drv = TaskDrivers(env, {j: m.fused(precision) for j, m in mods.items()})
    env.reset(); drv.reset()
    actions = _agent_actions(E, seed=5)
    worst, spread = 0.0, []
    for t in range(K):
        chain = drv.last_action.clone()
        drv.step(actions)
        lw = env.lw_obs                                    # what the policies were served this step (until the next observe)
        for j in slots:
            want = mods[j]({"lidar": lw["lidar"][:, j], "inertial_data": lw["inertial_data"][:, j], "last_action": chain})
            got = env.lw_actions[:, j]
            worst = max(worst, float((got - want).abs().max()))
            spread.append(float(want.std()))
            chain = torch.where(lw["present"][:, j, None], got, chain)
        chain.masked_fill_(env.done.bool()[:, None], 0.0)
        assert _same(chain, drv.last_action), f"step {t}: last_action"
    print(f"{name} {precision}: |serve - module| <= {worst:.3g}")
    assert worst < TOL[precision], f"{name} {precision}: |serve - float32 module| = {worst}"
    assert sum(spread) / len(spread) > 0.05, "vacuous: the policies' actions do not vary"
    env.close()
