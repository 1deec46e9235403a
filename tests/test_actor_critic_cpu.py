"""The actor-critic side of the reference's SB3 PPO on CPU: LidarInertialActorCritic against a by-hand evaluation of an SB3 state
dict, the fragment model of the actor-critic kernel, GAE in DeviceRollout terms against SB3's own loop, and the argument
checks of dc_policy_create_ac / dc_policy_act / dc_gae."""
import ctypes as C
import io
import math
import zipfile

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from dronechase_b200.policy import LidarInertialActionPolicy, LidarInertialActorCritic
from tests.test_policy_cpu import _by_hand, _sb3_state_dict


def _shared(sd):
    """SB3 with share_features_extractor=True (PPO's default): vf_features_extractor.* alias features_extractor.*."""
    return {k: (sd["features_extractor." + k[len("vf_features_extractor."):]] if k.startswith("vf_features_extractor.") else v)
            for k, v in sd.items()}


def _obs(E, seed, dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    return {"lidar": torch.rand(E, 3, 13, 26, generator=g, dtype=dtype), "inertial_data": torch.rand(E, 15, generator=g, dtype=dtype) * 2 - 1,
            "last_action": torch.rand(E, 4, generator=g, dtype=dtype)}


def _features_by_hand(sd, obs):
    pre = "features_extractor."
    x = F.relu(F.conv2d(obs["lidar"], sd[pre + "lidar_feature_extractor.0.weight"], sd[pre + "lidar_feature_extractor.0.bias"], stride=4))
    x = F.relu(F.conv2d(x, sd[pre + "lidar_feature_extractor.2.weight"], sd[pre + "lidar_feature_extractor.2.bias"], stride=2)).flatten(1)

    def mlp(v, name):
        for j in range(3):
            v = F.relu(F.linear(v, sd[pre + f"{name}.{2 * j}.weight"], sd[pre + f"{name}.{2 * j}.bias"]))
        return v
    f = torch.cat((x, mlp(obs["inertial_data"], "inertial_feature_extractor"), mlp(obs["last_action"], "action_feature_extractor")), 1)
    return F.relu(F.linear(f, sd[pre + "final_layer.0.weight"], sd[pre + "final_layer.0.bias"]))


def test_actor_critic_matches_sb3_by_hand(tmp_path):
    sd = _shared(_sb3_state_dict())
    sd["log_std"] = torch.tensor([0.0, -1.0, 0.5, -0.3])
    obs = _obs(6, 0)
    ac = LidarInertialActorCritic(lidar_channels=3, features_dim=32, pi=(16, 24), seed=None).load_sb3_state_dict(sd)
    assert ac.vf == (16, 24)
    # every key of the archive but the aliased extractors reached the module
    got = ac.state_dict()
    for k, v in sd.items():
        if k.startswith("features_extractor."):
            assert torch.equal(got[k[len("features_extractor."):]], v)
    for i in (0, 2):
        assert torch.equal(got[f"policy_net.{i}.weight"], sd[f"mlp_extractor.policy_net.{i}.weight"])
        assert torch.equal(got[f"vf_net.{i}.weight"], sd[f"mlp_extractor.value_net.{i}.weight"])
        assert torch.equal(got[f"vf_net.{i}.bias"], sd[f"mlp_extractor.value_net.{i}.bias"])
    for k in ("action_net.weight", "action_net.bias", "value_net.weight", "value_net.bias", "log_std"):
        assert torch.equal(got[k], sd[k]), k
    # by hand: SB3's ActorCriticPolicy.evaluate_actions with a DiagGaussianDistribution
    f = _features_by_hand(sd, obs)
    h = f
    for j in range(2):
        h = torch.tanh(F.linear(h, sd[f"mlp_extractor.policy_net.{2 * j}.weight"], sd[f"mlp_extractor.policy_net.{2 * j}.bias"]))
    mean = F.linear(h, sd["action_net.weight"], sd["action_net.bias"])
    hv = f
    for j in range(2):
        hv = torch.tanh(F.linear(hv, sd[f"mlp_extractor.value_net.{2 * j}.weight"], sd[f"mlp_extractor.value_net.{2 * j}.bias"]))
    value = F.linear(hv, sd["value_net.weight"], sd["value_net.bias"])
    sigma = sd["log_std"].exp()
    actions = mean + sigma * torch.randn(6, 4, generator=torch.Generator().manual_seed(1)) * 1.3
    log_prob = (-(actions - mean) ** 2 / (2 * sigma ** 2) - sd["log_std"] - 0.5 * math.log(2 * math.pi)).sum(1)
    entropy = (0.5 + 0.5 * math.log(2 * math.pi) + sd["log_std"]).sum().expand(6)
    v, lp, ent = ac.evaluate_actions(obs, actions)
    assert v.shape == (6, 1) and lp.shape == (6,) and ent.shape == (6,)
    assert torch.allclose(v, value, atol=1e-6) and torch.allclose(lp, log_prob, atol=1e-5) and torch.allclose(ent, entropy, atol=1e-6)
    m2, v2 = ac.forward_train(obs)
    assert torch.allclose(m2, mean, atol=1e-6) and torch.allclose(v2, value, atol=1e-6)
    assert torch.allclose(ac.predict_values(obs), value, atol=1e-6)
    assert torch.allclose(ac(obs), _by_hand(sd, obs, "features_extractor.", 2), atol=1e-6)      # forward: the clipped mean
    assert v.requires_grad and lp.requires_grad                                                   # differentiable for the update
    # from an archive: pi, vf, features_dim inferred; a separate vf extractor is refused
    path = tmp_path / "model.zip"
    buf = io.BytesIO(); torch.save(sd, buf)
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("policy.pth", buf.getvalue())
    ac2 = LidarInertialActorCritic.from_sb3_zip(str(path))
    assert ac2.pi == (16, 24) and ac2.vf == (16, 24) and ac2.features_dim == 32
    assert torch.allclose(ac2.predict_values(obs), value, atol=1e-6)
    with pytest.raises(ValueError, match="vf_features_extractor"):
        LidarInertialActorCritic(lidar_channels=3, features_dim=32, pi=(16, 24), seed=None).load_sb3_state_dict(_sb3_state_dict())


def test_actor_critic_leaves_the_actor_alone():
    """Seeded construction gives the plain policy's actor; the plain class keeps its parameters and describe()."""
    ac = LidarInertialActorCritic(lidar_channels=3, features_dim=64, pi=(64, 128), vf=(128,), seed=5)
    pol = LidarInertialActionPolicy(lidar_channels=3, features_dim=64, pi=(64, 128), seed=5)
    sd = ac.state_dict()
    for k, v in pol.state_dict().items():
        assert torch.equal(sd[k], v), k
    assert set(sd) - set(pol.state_dict()) == {"vf_net.0.weight", "vf_net.0.bias", "value_net.weight", "value_net.bias", "log_std"}
    assert "actor-critic" not in pol.describe() and "vf [128]" in ac.describe()
    obs = _obs(3, 2)
    assert torch.equal(ac(obs), pol(obs))


@pytest.mark.parametrize("features_dim,pi,vf,E", [(256, (128, 256, 512), (128, 256, 512), 37), (128, (64,), (256, 128), 64),
                                                  (192, (), (64,), 5), (64, (128,), (), 20), (128, (), (), 9)])
def test_fragment_model_of_the_actor_critic_kernel_matches_the_module(features_dim, pi, vf, E):
    """oracle/policy_ac_fragment_model.forward_ac restates the actor-critic kernel: the feature stash (row stride 260), the vf layers
    in place in it, the streamed 1-wide value head, value_net on the features when vf == () and the second final_layer when
    pi == ().  It must give the module's mean and value."""
    from oracle.policy_ac_fragment_model import forward_ac
    ac = LidarInertialActorCritic(lidar_channels=3, features_dim=features_dim, pi=pi, vf=vf, seed=11).double()
    with torch.no_grad():
        for p_ in ac.parameters():
            p_.mul_(1.7)
    obs = _obs(E, E, torch.float64)
    obs["lidar"][obs["lidar"] > 0.3] = 1.0
    with torch.no_grad():
        mean, value = ac.forward_train(obs)
    w = {k: ([t.detach().numpy() for t in v] if isinstance(v, list) else v.detach().numpy()) for k, v in ac.weight_arrays().items()}
    lin = [m for m in ac.vf_net if isinstance(m, torch.nn.Linear)]
    vw = {"vf_w": [m.weight.detach().numpy() for m in lin], "vf_b": [m.bias.detach().numpy() for m in lin],
          "value_w": ac.value_net.weight.detach().numpy(), "value_b": ac.value_net.bias.detach().numpy()}
    got_mean, got_value = forward_ac(w, vw, obs["lidar"].numpy(), obs["inertial_data"].numpy(), obs["last_action"].numpy(), activation=2)
    assert np.abs(got_mean - mean.numpy()).max() < 1e-12
    assert np.abs(got_value - value[:, 0].numpy()).max() < 1e-12
    assert value.std() > 1e-3, "vacuous comparison: constant value"


def test_policy_normals_are_standard_normal():
    from oracle.policy_ac_fragment_model import policy_normals
    eps = np.concatenate([policy_normals(7, c, np.arange(50000)) for c in range(4)])
    assert eps.shape == (200000, 4) and np.isfinite(eps).all()
    assert abs(eps.mean()) < 0.01 and abs(eps.var() - 1) < 0.02
    assert not np.array_equal(policy_normals(7, 0, np.arange(8)), policy_normals(7, 1, np.arange(8)))
    assert not np.array_equal(policy_normals(7, 0, np.arange(8)), policy_normals(8, 0, np.arange(8)))


def _sb3_gae(rewards, values, dones_after, last_values, last_dones, gamma, lam):
    """stable-baselines3 RolloutBuffer.compute_returns_and_advantage, literally: episode_starts[t] = done before step t."""
    T = rewards.shape[0]
    episode_starts = np.zeros_like(rewards)
    episode_starts[1:] = dones_after[:-1]
    adv = np.zeros_like(rewards)
    last_gae_lam = 0
    for step in reversed(range(T)):
        if step == T - 1:
            next_non_terminal = 1.0 - last_dones.astype(np.float32)
            next_values = last_values
        else:
            next_non_terminal = 1.0 - episode_starts[step + 1]
            next_values = values[step + 1]
        delta = rewards[step] + gamma * next_values * next_non_terminal - values[step]
        last_gae_lam = delta + gamma * lam * next_non_terminal * last_gae_lam
        adv[step] = last_gae_lam
    return adv, adv + values


def gae_formula(rewards, values, dones, last_values, gamma, lam):
    """The recurrence of dc_gae: dones[t] = the done after step t."""
    T = rewards.shape[0]
    adv = np.zeros_like(rewards)
    a, next_v = np.zeros_like(last_values), last_values
    for t in reversed(range(T)):
        nt = 1.0 - dones[t].astype(np.float32)
        a = rewards[t] + gamma * next_v * nt - values[t] + gamma * lam * nt * a
        adv[t] = a
        next_v = values[t]
    return adv, adv + values


def test_gae_in_rollout_terms_is_sb3s():
    rng = np.random.default_rng(0)
    T, E = 33, 57
    rewards = rng.normal(size=(T, E)).astype(np.float32)
    values = rng.normal(size=(T, E)).astype(np.float32)
    dones = (rng.random((T, E)) < 0.1).astype(np.uint8)
    last_values = rng.normal(size=E).astype(np.float32)
    a1, r1 = _sb3_gae(rewards, values, dones, last_values, dones[-1], 0.99, 0.95)
    a2, r2 = gae_formula(rewards, values, dones, last_values, 0.99, 0.95)
    assert np.allclose(a1, a2, rtol=1e-5, atol=1e-5) and np.allclose(r1, r2, rtol=1e-5, atol=1e-5)
    assert dones.sum() > 50


def test_new_c_entry_points_check_arguments_and_refuse_without_a_device():
    from dronechase_b200 import _lib
    L = _lib.lib()
    h = C.c_void_p()
    w, v = _lib.dc_policy_weights(), _lib.dc_value_weights()
    assert L.dc_policy_create_ac(C.byref(w), None, 0, C.byref(h)) == -1 and b"null argument" in L.dc_last_error()
    assert L.dc_policy_create_ac(C.byref(w), C.byref(v), 0, C.byref(h)) == -1 and b"lidar_channels" in L.dc_last_error()
    w.lidar_channels, w.features_dim, w.n_pi, w.activation = 3, 256, 1, 2
    w.pi[0] = 128
    buf = (C.c_float * 4)()
    p = C.cast(buf, C.POINTER(C.c_float))
    for name, _ in _lib.dc_policy_weights._fields_:
        if name.endswith(("_w", "_b")):
            f = getattr(w, name)
            if isinstance(f, C.Array):
                for i in range(len(f)):
                    f[i] = p
            else:
                setattr(w, name, p)
    v.n_vf = 9
    assert L.dc_policy_create_ac(C.byref(w), C.byref(v), 0, C.byref(h)) == -1 and b"n_vf" in L.dc_last_error()
    v.n_vf, v.vf[0], v.vf[1] = 2, 128, 96
    assert L.dc_policy_create_ac(C.byref(w), C.byref(v), 0, C.byref(h)) == -1 and b"multiples of 64" in L.dc_last_error()
    v.vf[1] = 1024
    assert L.dc_policy_create_ac(C.byref(w), C.byref(v), 0, C.byref(h)) == -1 and b"null vf weight" in L.dc_last_error()
    for i in range(8):
        v.vf_w[i] = v.vf_b[i] = p
    assert L.dc_policy_create_ac(C.byref(w), C.byref(v), 0, C.byref(h)) == -1 and b"value_net" in L.dc_last_error()
    v.value_w = v.value_b = v.log_std = p
    x = C.c_void_p(1)
    assert L.dc_policy_act(None, x, x, x, 4, 0, 0, 0, 1, x, x, x, x, 0, None) == -1 and b"bad argument" in L.dc_last_error()
    assert L.dc_gae(None, x, x, x, 4, 4, 0.99, 0.95, x, x, None) == -1 and b"bad argument" in L.dc_last_error()
    assert L.dc_gae(x, x, x, x, 4, 4, 1.5, 0.95, x, x, None) == -1 and b"gamma" in L.dc_last_error()
    if not torch.cuda.is_available():
        assert L.dc_policy_create_ac(C.byref(w), C.byref(v), 0, C.byref(h)) == -4 and b"no CPU fallback" in L.dc_last_error()
        assert L.dc_gae(x, x, x, x, 4, 4, 0.99, 0.95, x, x, None) == -4 and b"no CPU fallback" in L.dc_last_error()
        from dronechase_b200.rollout import PPORollout                                       # noqa: F401 -- importable
        with pytest.raises(_lib.DroneChaseError, match="no CPU fallback"):
            LidarInertialActorCritic(lidar_channels=3, seed=0).fused()
