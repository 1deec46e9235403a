"""The fused policy kernel (csrc/policy_kernel.cu, dc_policy_forward) against the torch float32 module of
dronechase_b200/policy.py -- the network of ppo_policies.py:234-342 -- through the C ABI on a B200.

Tolerances (absolute, on the clipped mean action, |a| <= 1): 2e-5 for precision "3xtf32" (every product as three TF32 MMAs),
5e-3 for "tf32" (10-bit mantissa operands, float32 accumulate)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = {"3xtf32": 2e-5, "tf32": 5e-3}


def _obs(E, C, seed, dev="cuda"):
    g = torch.Generator(device=dev); g.manual_seed(seed)
    lidar = torch.rand(E, C, 13, 26, generator=g, device=dev)
    lidar[lidar > 0.25] = 1.0                              # mostly empty spheres, like the simulator's
    return {"lidar": lidar.contiguous(), "inertial_data": torch.rand(E, 15, generator=g, device=dev) * 2 - 1,
            "last_action": torch.rand(E, 4, generator=g, device=dev)}


def _module(C, features_dim, pi, activation="tanh", scale=1.6):
    from dronechase_b200.policy import LidarInertialActionPolicy
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False               # the reference of this test is float32 arithmetic
    pol = LidarInertialActionPolicy(lidar_channels=C, features_dim=features_dim, pi=pi, activation=activation, seed=4, device="cuda")
    with torch.no_grad():
        for p in pol.parameters():
            p.mul_(scale)
    return pol


def _check_against_the_module(pol, fused, precision, E, C):
    obs = _obs(E, C, seed=E)
    want = pol(obs)
    got = fused(obs)
    torch.cuda.synchronize()
    err = float((got - want).abs().max())
    assert got.shape == (E, 4) and err < TOL[precision], f"E={E}: |fused - float32 module| = {err}"
    assert float(got[:, 3].min()) >= 0 and float(got.abs().max()) <= 1
    assert float(want.std()) > 0.05 and bool((want.abs() < 1).any()), "vacuous comparison: every action clipped"


# the last five: an intermediate layer of 192 columns (idle column warps of the 32 x 32 tiles), last layers of 320 and 960
# columns (the last 256-column pass of head_layer partly filled), pi = () on 64 features, one layer narrower than the
# features, and the deepest net the kernel holds (8 pi layers: 15 of its 16 layers)
@pytest.mark.parametrize("precision", ["3xtf32", "tf32"])
@pytest.mark.parametrize("C,features_dim,pi,activation", [(3, 256, (128, 256, 512), "tanh"), (2, 128, (64,), "tanh"),
                                                          (3, 192, (), "tanh"), (3, 256, (256, 256, 256), "relu"),
                                                          (1, 64, (256, 1024), "tanh"), (3, 256, (192, 320), "tanh"),
                                                          (2, 64, (), "relu"), (1, 128, (64,), "tanh"),
                                                          (3, 192, (256, 64), "tanh"), (3, 256, (64,) * 7 + (960,), "tanh")])
def test_fused_policy_matches_the_float32_module(precision, C, features_dim, pi, activation):
    pol = _module(C, features_dim, pi, activation)
    fused = pol.fused(precision)
    for E in (1, 63, 64, 65, 127, 128, 1000, 4133):       # ragged last block, single env, whole blocks, several blocks
        _check_against_the_module(pol, fused, precision, E, C)
    # the same bits on every run, and for any batch a row travels in
    obs = _obs(1000, C, seed=1)
    a, b = fused(obs), fused(obs)
    part = fused({k: v[640:].contiguous() for k, v in obs.items()})
    assert torch.equal(a, b) and torch.equal(a[640:], part)
    fused.close()


def test_fused_policy_on_a_ragged_batch_of_65537():
    """1,025 blocks, the last with one env: grid-sized row indices."""
    pol = _module(3, 256, (128, 256, 512))
    fused = pol.fused("3xtf32")
    _check_against_the_module(pol, fused, "3xtf32", 65537, 3)
    fused.close()


def test_fused_policy_on_the_simulator_observations_and_sb3_weights(tmp_path):
    """Closed loop: the fused kernel reads the simulator's own observation tensors and its actions drive dc_step; the torch
    module evaluated on the same observations agrees at every step.  Weights come from an SB3-style archive."""
    import io, zipfile
    from dronechase_b200 import BatchedThreatEngageEnv
    from dronechase_b200.policy import LidarInertialActionPolicy
    from tests.test_policy_cpu import _sb3_state_dict
    sd = _sb3_state_dict(pi=(128, 256, 512), features_dim=256)
    path = tmp_path / "model.zip"
    buf = io.BytesIO(); torch.save(sd, buf)
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("policy.pth", buf.getvalue())
    env = BatchedThreatEngageEnv("exp02_v2_full", n_envs=777, seed=2, device=0, auto_reset=True)
    env.reset()
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    pol = LidarInertialActionPolicy.from_sb3_zip(str(path), env=env)
    fused = pol.fused()
    import copy
    pol64 = copy.deepcopy(pol).double()                   # these weights are larger than a trained net's (randn * 0.2): float32
    worst = worst32 = 0.0                                 # rounding itself is ~1e-4 here, so both are measured against float64
    for t in range(120):
        a = fused(env.obs)
        want = pol64({k: v.double() for k, v in env.obs.items()})
        worst = max(worst, float((a.double() - want).abs().max()))
        worst32 = max(worst32, float((pol(env.obs).double() - want).abs().max()))
        env.step(a)
    print(f"fused vs float64 {worst:.3g}, torch float32 vs float64 {worst32:.3g}")
    # three TF32 MMAs keep 21-22 mantissa bits of a product (the tail operand is truncated to TF32, tail x tail is dropped)
    # against float32's 24: a few times torch's own float32 rounding on these large weights
    assert worst < max(2e-5, 8.0 * worst32), f"fused vs float64 {worst}, torch float32 vs float64 {worst32}"
    assert int((env.obs["lidar"] < 1).sum()) > 100        # the spheres were not empty: the convolution saw entities
    fused.close(); env.close()


def test_fused_policy_refuses_shapes_it_does_not_hold():
    from dronechase_b200 import _lib
    pol = _module(3, 256, (128, 320, 512))
    with pytest.raises(_lib.DroneChaseError, match="multiples of 64"):
        pol.fused()
    ok = _module(3, 256, (128,)).fused()
    with pytest.raises(ValueError):
        ok({"lidar": torch.zeros(4, 2, 13, 26, device="cuda"), "inertial_data": torch.zeros(4, 15, device="cuda"),
            "last_action": torch.zeros(4, 4, device="cuda")})
    ok.close()
