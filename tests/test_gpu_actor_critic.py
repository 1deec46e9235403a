"""The actor-critic kernel (csrc/policy_kernel.cu policy_ac_kernel, dc_policy_act), dc_gae and PPORollout on a B200, against the
torch float32 module (LidarInertialActorCritic), the plain kernel (dc_policy_forward) and the float64 Philox / Box-Muller oracle.

Tolerances: value 2e-5 ("3xtf32") / 5e-3 ("tf32") of the float32 module, as the mean action in test_gpu_policy.py; the
normals 1e-5 of float64; log_prob 1e-4 of the float64 formula on the oracle's normals."""
import copy
import math

import numpy as np
import pytest
import torch

from tests.test_gpu_policy import _obs

pytestmark = pytest.mark.gpu

TOL = {"3xtf32": 2e-5, "tf32": 5e-3}
NETS = [(3, 256, (128, 256, 512), "tanh"), (2, 128, (64,), "tanh"), (3, 192, (), "tanh"), (3, 256, (256, 256, 256), "relu"),
        (1, 64, (256, 1024), "tanh")]
LOW, HIGH = torch.tensor([-1.0, -1, -1, 0]), torch.tensor([1.0, 1, 1, 1])


def _ac(C, features_dim, pi, activation, log_std, scale=1.6, vf=None):
    from dronechase_b200.policy import LidarInertialActorCritic
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    ac = LidarInertialActorCritic(lidar_channels=C, features_dim=features_dim, pi=pi, vf=vf, activation=activation, seed=4, device="cuda")
    with torch.no_grad():
        for p in ac.parameters():
            p.mul_(scale)
        ac.log_std.fill_(log_std)
    return ac


@pytest.mark.parametrize("log_std", [0.0, -1.0])
@pytest.mark.parametrize("precision", ["3xtf32", "tf32"])
@pytest.mark.parametrize("C,features_dim,pi,activation", NETS)
def test_act_against_the_plain_kernel_the_module_and_the_oracle(precision, C, features_dim, pi, activation, log_std):
    from oracle.policy_ac_fragment_model import policy_normals
    ac = _ac(C, features_dim, pi, activation, log_std)
    fused = ac.fused(precision)
    seed, counter, off = 0x1234_5678_9ABC, 3, 100
    sigma = math.exp(log_std)
    low, high = LOW.cuda(), HIGH.cuda()
    for E in (1, 63, 64, 65, 1000, 4133):
        obs = _obs(E, C, seed=E)
        mean_a, raw0, lp0, v0 = fused.act(obs, counter, sample=False)
        assert raw0 is None and lp0 is None
        assert torch.equal(mean_a, fused(obs)), "sample = 0: not the plain kernel's action bit for bit"
        with torch.no_grad():
            _, want_v = ac.forward_train(obs)
        err_v = float((v0 - want_v[:, 0]).abs().max())
        assert err_v < TOL[precision], f"E={E}: |value - float32 module| = {err_v}"
        env_a, raw, lp, v = fused.act(obs, counter, seed=seed, env_offset=off)
        torch.cuda.synchronize()
        assert torch.equal(v, v0)
        assert torch.equal(env_a, torch.minimum(torch.maximum(raw, low), high)), "env_action is not clip(raw)"
        eps64 = policy_normals(seed, counter, off + np.arange(E))
        # where the mean is inside the box the sample = 0 action IS the kernel's mean: recover the kernel's eps there
        m = mean_a.double().cpu().numpy()
        inside = (m > LOW.numpy()) & (m < HIGH.numpy())
        r = raw.double().cpu().numpy()
        eps = (r - m) / np.float32(sigma)
        assert inside.sum() > 0.2 * inside.size
        assert np.abs(eps - eps64)[inside].max() < 1e-5 + 1e-6 * np.abs(r[inside]).max() / sigma, "eps differs from the oracle"
        assert np.abs(r - (m + np.float32(sigma) * eps64))[inside].max() < 2e-6 * (1 + np.abs(r).max())
        lp64 = (-0.5 * eps64 ** 2 - log_std).sum(1) - 2 * math.log(2 * math.pi)
        assert np.abs(lp.double().cpu().numpy() - lp64).max() < 1e-4
        if precision == "3xtf32" and log_std == 0.0:
            with torch.no_grad():
                _, want_lp, _ = ac.evaluate_actions(obs, raw)
            assert float((lp - want_lp).abs().max()) < 5e-4
    # the same bits on every run, and for any batch a row travels in (with the batch's env_offset)
    obs = _obs(1000, C, seed=1)
    a = fused.act(obs, 7, seed=seed, env_offset=off)
    b = fused.act(obs, 7, seed=seed, env_offset=off)
    part = fused.act({k: x[640:].contiguous() for k, x in obs.items()}, 7, seed=seed, env_offset=off + 640)
    for x, y, z in zip(a, b, part):
        assert torch.equal(x, y) and torch.equal(x[640:], z)
    fused.close()


def test_sampled_noise_is_standard_normal_and_is_the_oracles():
    """action_net = 0 and log_std = 0: the raw action IS eps.  65,536 envs x 4 counters."""
    from oracle.policy_ac_fragment_model import policy_normals
    ac = _ac(3, 256, (128, 256, 512), "tanh", 0.0)
    with torch.no_grad():
        ac.action_net.weight.zero_(); ac.action_net.bias.zero_()
    fused = ac.fused()
    E = 65536
    obs = _obs(E, 3, seed=5)
    eps = []
    for c in range(4):
        raw = fused.act(obs, c, seed=99)[1].double().cpu().numpy()
        assert np.abs(raw - policy_normals(99, c, np.arange(E))).max() < 1e-5
        eps.append(raw)
    eps = np.concatenate(eps)
    assert abs(eps.mean()) < 0.01 and abs(eps.var() - 1) < 0.02
    fused.close()


def test_ppo_rollout_on_the_simulator():
    """PPORollout on exp02_v2_full: stored values and log-probs agree with evaluate_actions on minibatch rows rebuilt from the hit
    lists; dc_gae is SB3's loop; a PPO loss backpropagates; after an optimiser step and refresh() collect sees the new weights."""
    from dronechase_b200 import BatchedThreatEngageEnv
    from dronechase_b200.policy import LidarInertialActorCritic
    from dronechase_b200.rollout import PPORollout
    from tests.test_actor_critic_cpu import _sb3_gae
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    E, T = 1024, 32
    env = BatchedThreatEngageEnv("exp02_v2_full", n_envs=E, seed=3, device=0, auto_reset=True, with_hits=True)
    env.reset()
    ac = LidarInertialActorCritic(env=env, seed=0)
    fused = ac.fused()
    ro = PPORollout(env, T, seed=9)
    ro.collect(fused).compute_returns_and_advantage(0.99, 0.95)
    assert ro.counter == T and int(ro.dones.sum()) > 0
    idx = torch.randperm(T * E, device="cuda", generator=torch.Generator(device="cuda").manual_seed(0))[:4096]
    b = ro.minibatch(idx)
    obs = {k: b[k] for k in ("lidar", "inertial_data", "last_action")}
    with torch.no_grad():
        v, lp, _ = ac.evaluate_actions(obs, b["actions"])
    assert float((v[:, 0] - b["old_values"]).abs().max()) < 1e-4
    assert float((lp - b["old_log_prob"]).abs().max()) < 5e-4
    assert int((b["lidar"] < 1).sum()) > 100
    # GAE against stable-baselines3's loop
    np_ = lambda t: t.cpu().numpy()      # noqa: E731
    dn = np_(ro.dones)
    adv, ret = _sb3_gae(np_(ro.rewards), np_(ro.values), dn, np_(ro.last_values), dn[-1], 0.99, 0.95)
    scale = max(1.0, float(np.abs(adv).max()))
    assert np.allclose(np_(ro.advantages), adv, rtol=1e-5, atol=1e-5 * scale)
    assert np.allclose(np_(ro.returns), ret, rtol=1e-5, atol=1e-5 * scale)
    assert float(ro.advantages.abs().max()) > 0
    # one PPO update step
    opt = torch.optim.Adam(ac.parameters(), lr=1e-2)
    v, lp, ent = ac.evaluate_actions(obs, b["actions"])
    a = b["advantages"]
    a = (a - a.mean()) / (a.std() + 1e-8)
    ratio = torch.exp(lp - b["old_log_prob"])
    loss = (-torch.min(ratio * a, ratio.clamp(0.8, 1.2) * a).mean() + 0.5 * ((b["returns"] - v[:, 0]) ** 2).mean()
            - 0.01 * ent.mean())
    loss.backward()
    grads = [p.grad for p in ac.parameters() if p.requires_grad]
    assert all(g is not None and bool(torch.isfinite(g).all()) for g in grads)
    assert float(ac.log_std.grad.abs().sum()) > 0 and float(ac.value_net.weight.grad.abs().sum()) > 0
    before = copy.deepcopy(ac)
    opt.step()
    fused.refresh()
    obs0 = {k: x.clone() for k, x in env.obs.items()}
    ro.collect(fused, n_steps=2)
    with torch.no_grad():
        new_v, old_v = ac.predict_values(obs0)[:, 0], before.predict_values(obs0)[:, 0]
        _, new_lp, _ = ac.evaluate_actions(obs0, ro.actions[0])
    assert float((ro.values[0] - new_v).abs().max()) < 1e-4
    assert float((new_v - old_v).abs().max()) > 1e-2, "the optimiser step did not move the values: vacuous check"
    assert float((ro.log_probs[0] - new_lp).abs().max()) < 5e-4
    assert ro.counter == T + 2
    fused.close(); env.close()


def test_act_refuses_a_plain_policy():
    from dronechase_b200 import _lib
    from tests.test_gpu_policy import _module
    fused = _module(3, 256, (128,)).fused()
    obs = _obs(4, 3, seed=0)
    with pytest.raises(_lib.DroneChaseError, match="LidarInertialActorCritic"):
        fused.act(obs, 0)
    with pytest.raises(_lib.DroneChaseError, match="LidarInertialActorCritic"):
        fused.values(obs)
    fused.close()
