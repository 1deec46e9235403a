"""The fused policy kernel (csrc/policy_kernel.cu: policy_kernel behind dc_policy_forward, policy_ac_kernel behind dc_policy_act),
dc_gae (csrc/gae.cu) and PPORollout (rollout.py) on a B200, at the edges of what they accept, each against a float64 evaluation:
``copy.deepcopy(module).double()`` on ``obs.double()``, ``policy_normals`` (the float64 Philox / Box-Muller oracle of the
sampling epilogue) and the GAE recurrence of tests/test_actor_critic_cpu.py in float64.

- mean action and V(s) of both kernels in both precisions on random inputs and on inputs at the edges of the observation
  space, and in TF32 with the last tanh layer driven into saturation: error <= max(2e-5 (3xtf32) / 5e-3 (tf32), 8 x torch
  float32's own error against float64 on the same inputs), the bound of the SB3 closed loop in test_gpu_policy.py; the
  value's relative to max(1, |V|);
- a log_std per component and an asymmetric action box: clipping, noise, log-probability;
- the Philox key and counter at their top bits and the last env window dc_policy_act accepts;
- rows that move to another position inside their 64-row block when the batch is split;
- dc_gae over ragged shapes, gamma / lambda at 0 and 1, done patterns and partial calls, with an error bound derived from
  float32 rounding;
- PPORollout over an env window (env_offset) and across collect calls."""
import copy
import ctypes as C
import math

import numpy as np
import pytest
import torch
from torch import nn

from tests.test_gpu_actor_critic import NET_IDS, NETS, _ac
from tests.test_gpu_policy import _obs

pytestmark = pytest.mark.gpu

TOL = {"3xtf32": 2e-5, "tf32": 5e-3}
U32 = 2.0 ** -24                                   # float32 unit roundoff: |fl(x) - x| <= U32 |x|
SPREAD = 3.0                                       # standard deviation of the pre-activations of a saturated tanh layer


def _f64(obs):
    return {k: v.double() for k, v in obs.items()}


def _edge_obs(C, E=200, dev="cuda"):
    """Rows at the edges of the observation space: all-1.0 spheres (nothing seen), all-0.0 spheres (everything at zero
    distance) and mostly-empty ones in turn, every inertial entry exactly -1 or +1, last actions at the 16 corners of the
    default action box."""
    g = torch.Generator(device=dev)
    g.manual_seed(17)
    lidar = torch.rand(E, C, 13, 26, generator=g, device=dev)
    lidar[lidar > 0.25] = 1.0
    lidar[0::3] = 1.0
    lidar[1::3] = 0.0
    inertial = torch.where(torch.rand(E, 15, generator=g, device=dev) < 0.5, -1.0, 1.0)
    corners = torch.tensor([[x, y, z, w] for x in (-1.0, 1.0) for y in (-1.0, 1.0) for z in (-1.0, 1.0) for w in (0.0, 1.0)],
                           device=dev)
    return {"lidar": lidar.contiguous(), "inertial_data": inertial.contiguous(),
            "last_action": corners[torch.arange(E, device=dev) % 16].contiguous()}


def _last_hidden(ac, obs):
    """The last hidden layers of pi and vf (the ones streamed into action_net / value_net) and their inputs."""
    out = []
    with torch.no_grad():
        f = ac.features(obs)
        for seq in (ac.policy_net, ac.vf_net):
            if len(seq):
                out.append((seq[-2], seq[:-2](f)))
    return out


def _saturate(ac, obs):
    """Scale the last hidden layer of pi and of vf (weights and bias) so that its pre-activations spread over the batch with
    standard deviation SPREAD: a third of its tanh outputs lie beyond |h| = 0.995, where tanh.approx flattens, and go straight
    into the head.  Scaling every layer instead would compound TF32's operand rounding layer after layer."""
    with torch.no_grad():
        for layer, x in _last_hidden(ac, obs):
            s = SPREAD / float(layer(x).std())
            layer.weight.mul_(s)
            layer.bias.mul_(s)


# saturated: nets with a hidden tanh layer, in TF32, whose tanh.approx it is there for.  In 3xTF32 (tanhf) the saturating weights
# measure the operand split instead: the tensor core truncates the tail operands and drops tail x tail, about 21 bits per
# product, and V(s) came to 2.3e-5 / 3.3e-5 of float64 on the default and the deepest net (1,000 envs, B200), 12x / 15x
# torch float32's own error -- past the 8x of the bound, with nothing wrong in the kernel.
CASES = [pytest.param(net, inp, prec, id=f"{nid}-{inp}-{prec}") for net, nid in zip(NETS, NET_IDS)
         for inp in ("random", "edges", "saturated") for prec in ("3xtf32", "tf32")
         if inp != "saturated" or (prec == "tf32" and net[4] == "tanh" and (net[2] or net[3]))]


@pytest.mark.parametrize("net,inputs,precision", CASES)
def test_mean_action_and_value_against_float64(net, inputs, precision):
    C, features_dim, pi, vf, activation = net
    ac = _ac(C, features_dim, pi, activation, 0.0, vf=vf)
    obs = _edge_obs(C) if inputs == "edges" else _obs(1000, C, seed=11)
    if inputs == "saturated":
        _saturate(ac, obs)
    ac64, obs64 = copy.deepcopy(ac).double(), _f64(obs)
    with torch.no_grad():
        want_a, want_v = ac64(obs64), ac64.predict_values(obs64)[:, 0]
        a32, v32 = ac(obs).double(), ac.predict_values(obs)[:, 0].double()
        if inputs == "saturated":
            h = torch.cat([torch.tanh(layer(x)).flatten() for layer, x in _last_hidden(ac64, obs64)])
            assert float((h.abs() > 0.995).double().mean()) > 0.25, "the weights do not saturate tanh"
    vscale = want_v.abs().clamp(min=1.0)
    bound_a = max(TOL[precision], 8.0 * float((a32 - want_a).abs().max()))
    bound_v = max(TOL[precision], 8.0 * float(((v32 - want_v).abs() / vscale).max()))
    low, high = ac64.low, ac64.high
    assert float(((want_a > low) & (want_a < high)).double().mean()) > 0.2, "vacuous comparison: most actions clipped"
    assert float(want_v.std()) > 1e-3, "vacuous comparison: constant value"

    fused = ac.fused(precision)
    plain = fused(obs)                                                 # dc_policy_forward
    mean_ac, _, _, value = fused.act(obs, 0, sample=False)            # dc_policy_act
    values = fused.values(obs)
    torch.cuda.synchronize()
    for name, got in (("dc_policy_forward", plain), ("dc_policy_act", mean_ac)):
        err = float((got.double() - want_a).abs().max())
        assert err <= bound_a, f"{name}: |mean action - float64| = {err:.3g} > {bound_a:.3g}"
    err_v = float(((value.double() - want_v).abs() / vscale).max())
    assert err_v <= bound_v, f"|V - float64| / max(1, |V|) = {err_v:.3g} > {bound_v:.3g}"
    assert torch.equal(values, value)
    fused.close()


# ---------------------------------------------------------------------------------------------- log_std per component, box
LOG_STD = [0.3, -1.2, -0.1, -2.5]
BOX_LOW, BOX_HIGH = [-0.5, -2.0, -1.0, 0.25], [0.5, 2.0, 0.1, 0.75]
MEDIAN = [0.45, 0.0, 0.1, 0.5]       # action_net's bias moves the median of the mean there: k = 0, 2 at a box edge, 3 mid-box


@pytest.mark.parametrize("precision", ["3xtf32", "tf32"])
@pytest.mark.parametrize("net", [NETS[0], NETS[6], NETS[7]], ids=[NET_IDS[0], NET_IDS[6], NET_IDS[7]])
def test_per_component_log_std_and_an_asymmetric_box(net, precision):
    from oracle.policy_ac_fragment_model import policy_normals
    C, features_dim, pi, vf, activation = net
    ac = _ac(C, features_dim, pi, activation, 0.0, vf=vf)
    seed, counter, off, E = 0x0BAD_CAFE_1234, 11, 4096, 4133
    obs = _obs(E, C, seed=21)
    with torch.no_grad():
        ac.action_net.bias.add_(torch.tensor(MEDIAN, device="cuda") - ac.forward_train(obs)[0].median(0).values)
        ac.log_std.copy_(torch.tensor(LOG_STD))
        ac.low.copy_(torch.tensor(BOX_LOW))
        ac.high.copy_(torch.tensor(BOX_HIGH))
    # the same weights with an unbounded box: its clipped mean is the kernel's unclipped mean
    wide = copy.deepcopy(ac)
    with torch.no_grad():
        wide.low.fill_(-math.inf)
        wide.high.fill_(math.inf)
    fused, fused_wide = ac.fused(precision), wide.fused(precision)
    low, high = ac.low, ac.high
    sigma = np.exp(np.float32(LOG_STD)).astype(np.float64)            # what expf gives, to an ulp
    ac64, obs64 = copy.deepcopy(ac).double(), _f64(obs)
    with torch.no_grad():
        mean64 = ac64.forward_train(obs64)[0]
        bound_m = max(TOL[precision], 8.0 * float((ac.forward_train(obs)[0].double() - mean64).abs().max()))

    plain = fused(obs)
    mean_c, _, _, v0 = fused.act(obs, counter, sample=False)
    mean_u = fused_wide.act(obs, counter, sample=False)[0]
    assert torch.equal(mean_c, plain), "sample = 0: not dc_policy_forward's action bit for bit"
    # both kernels clip to the module's box
    assert torch.equal(plain, torch.minimum(torch.maximum(mean_u, low), high)), "the mean is not clipped to the module's box"
    outside = (mean_u < low) | (mean_u > high)
    assert int(outside.sum()) > 0.02 * outside.numel() and float(outside.double().mean()) < 0.8, "the box clips nothing / everything"
    err_m = float((mean_u.double() - mean64).abs().max())
    assert err_m <= bound_m, f"|unclipped mean - float64| = {err_m:.3g} > {bound_m:.3g}"

    env_a, raw, lp, v = fused.act(obs, counter, seed=seed, env_offset=off)
    torch.cuda.synchronize()
    assert torch.equal(v, v0)
    assert torch.equal(env_a, torch.minimum(torch.maximum(raw, low), high)), "env_action is not clip(raw) under the module's box"
    assert int(((raw < low) | (raw > high)).sum()) > 0.05 * raw.numel(), "vacuous: the samples stay inside the box"
    eps64 = policy_normals(seed, counter, off + np.arange(E))
    r, m = raw.double().cpu().numpy(), mean_c.double().cpu().numpy()
    inside = (m > np.float32(BOX_LOW)) & (m < np.float32(BOX_HIGH))
    for k in range(4):
        sel = inside[:, k]
        assert sel.sum() > 0.1 * E, f"component {k}: the mean is inside the box for too few rows"
        eps = (r[sel, k] - m[sel, k]) / sigma[k]
        tol = 1e-5 + 1e-6 * np.abs(r[sel, k]).max() / sigma[k]
        assert np.abs(eps - eps64[sel, k]).max() < tol, f"component {k}: eps differs from the oracle"
    # the log-probability: the float64 formula on the oracle's normals, and float64 evaluate_actions on the returned raw actions
    lp_k = lp.double().cpu().numpy()
    lp64 = (-0.5 * eps64 ** 2 - np.float32(LOG_STD).astype(np.float64)).sum(1) - 2 * math.log(2 * math.pi)
    assert np.abs(lp_k - lp64).max() < 1e-4, "log_prob differs from the float64 formula"
    with torch.no_grad():
        _, lp_eval, _ = ac64.evaluate_actions(obs64, raw.double())
    # the kernel's mean differs from float64 by dm: the log-probability of the same raw action moves by
    # sum_k (dm_k eps_k / sigma_k + dm_k^2 / (2 sigma_k^2))
    dm = (mean_u.double() - mean64).abs().cpu().numpy()
    allow = 1e-4 + 1.01 * (dm * np.abs(eps64) / sigma + dm ** 2 / (2 * sigma ** 2)).sum(1)
    assert (np.abs(lp_k - lp_eval.cpu().numpy()) <= allow).all(), "log_prob differs from float64 evaluate_actions"
    fused.close(); fused_wide.close()


# ------------------------------------------------------------------------------------------------------------- Philox edges
@pytest.mark.parametrize("precision", ["3xtf32", "tf32"])
def test_philox_key_counter_and_env_index_at_their_top_bits(precision):
    """action_net = 0 and log_std = 0: the raw action IS eps.  Key 0xFEDCBA9876543210 (top bit of k1 set), counter 2^32 - 1,
    the last window of E envs below 2^32; one env more is refused."""
    from dronechase_b200 import _lib
    from oracle.policy_ac_fragment_model import policy_normals
    ac = _ac(3, 256, (128, 256, 512), "tanh", 0.0)
    with torch.no_grad():
        ac.action_net.weight.zero_(); ac.action_net.bias.zero_()
    fused = ac.fused(precision)
    E, seed, counter = 1000, 0xFEDC_BA98_7654_3210, 0xFFFF_FFFF
    off = 2 ** 32 - E
    obs = _obs(E, 3, seed=2)
    raw = fused.act(obs, counter, seed=seed, env_offset=off)[1]
    eps64 = policy_normals(seed, counter, off + np.arange(E))
    assert np.abs(raw.double().cpu().numpy() - eps64).max() < 1e-5, "eps differs from the oracle at the top of the key space"
    with pytest.raises(_lib.DroneChaseError, match="env_offset"):
        fused.act(obs, counter, seed=seed, env_offset=off + 1)
    for other in (seed & 0xFFFF_FFFF, seed ^ (1 << 63), seed ^ (1 << 32)):          # only the high 32 bits differ
        raw2 = fused.act(obs, counter, seed=other, env_offset=off)[1]
        assert bool((raw2 != raw).any(dim=1).all()), f"seed {other:#x}: the high word of the key does not reach the noise"
    fused.close()


# ----------------------------------------------------------------------------------------------- batch splits, unaligned rows
@pytest.mark.parametrize("precision", ["3xtf32", "tf32"])
@pytest.mark.parametrize("net", [NETS[0], NETS[7]], ids=[NET_IDS[0], NET_IDS[7]])
def test_rows_that_move_inside_their_block_keep_their_bits(net, precision):
    """Rows [641:] and [1:] of a batch: every row lands at another position of its 64-row block (641 = 10 x 64 + 1)."""
    C, features_dim, pi, vf, activation = net
    ac = _ac(C, features_dim, pi, activation, -0.5, vf=vf)
    fused = ac.fused(precision)
    seed, counter, off = 0x5EED_0000_0001, 9, 300
    obs = _obs(1000, C, seed=4)
    full_call, full_act, full_v = fused(obs), fused.act(obs, counter, seed=seed, env_offset=off), fused.values(obs)
    for start in (641, 1):
        part = {k: x[start:].contiguous() for k, x in obs.items()}
        assert torch.equal(fused(part), full_call[start:]), f"[{start}:]: dc_policy_forward"
        got = fused.act(part, counter, seed=seed, env_offset=off + start)
        for name, x, y in zip(("env_actions", "raw_actions", "log_prob", "value"), got, full_act):
            assert torch.equal(x, y[start:]), f"[{start}:]: act {name}"
        assert torch.equal(fused.values(part), full_v[start:]), f"[{start}:]: values"
    fused.close()


# ------------------------------------------------------------------------------------------------------------------ dc_gae
def _gae_reference(rewards, values, dones, last_values, gamma, lam):
    """(advantages, returns) in float64 -- gae_formula of test_actor_critic_cpu on float64 arrays, with the float32
    coefficients dc_gae receives -- and their error bounds for a float32 evaluation.

    A step of the recurrence rounds at most five quantities, once each: gamma V_{t+1}, r_t + gamma V_{t+1} nt_t, delta_t,
    gl nt_t A_{t+1} and A_t (nt = 1 - done, gl = gamma lambda; dc_gae's FMAs skip some of these roundings, a plain float32
    loop makes all five).  Round to nearest leaves an error uniform within +-ulp(x)/2, standard deviation <= U32 |x| / sqrt(3).
    An error made at step s reaches A_t multiplied by prod_{j=t}^{s-1} gl nt_j, so as independent zero-mean errors the error of
    A_t has standard deviation <= U32 sigma_t / sqrt(3), with sigma_t^2 = q_t + (gl nt_t)^2 sigma_{t+1}^2 and q_t the sum of the
    squares of the five quantities; R_t = A_t + V_t adds R_t^2.  Of n such errors none exceeds z times its standard deviation
    but with probability < 1e-6 for z = sqrt(2 ln(2n / 1e-6)).  dc_gae also forms gl = float32(gamma lambda): that error dgl
    enters every step with the same sign and is added in full, lin_t = |dgl| |nt_t A_{t+1}| + gl nt_t lin_{t+1}."""
    from tests.test_actor_critic_cpu import gae_formula
    g32, l32 = float(np.float32(gamma)), float(np.float32(lam))
    r, v, lv = rewards.astype(np.float64), values.astype(np.float64), last_values.astype(np.float64)
    adv, ret = gae_formula(r, v, dones, lv, g32, l32)
    gl = g32 * l32                                                     # exact in float64
    dgl = abs(float(np.float32(gl)) - gl)
    T = r.shape[0]
    s2, lin = np.zeros_like(lv), np.zeros_like(lv)
    sig_a, lin_a = np.zeros_like(r), np.zeros_like(r)
    for t in reversed(range(T)):
        nt = 1.0 - dones[t].astype(np.float64)
        nv = v[t + 1] if t + 1 < T else lv
        na = adv[t + 1] if t + 1 < T else np.zeros_like(lv)
        gv = g32 * nv
        delta = r[t] + gv * nt - v[t]
        q = gv ** 2 + (r[t] + gv * nt) ** 2 + delta ** 2 + (gl * nt * na) ** 2 + adv[t] ** 2
        s2 = q + (gl * nt) ** 2 * s2
        lin = dgl * np.abs(nt * na) + gl * nt * lin
        sig_a[t], lin_a[t] = np.sqrt(s2), lin
    z = math.sqrt(2 * math.log(2 * r.size / 1e-6))
    bound_a = z * U32 * sig_a / math.sqrt(3) + lin_a
    bound_r = z * U32 * np.sqrt(sig_a ** 2 + ret ** 2) / math.sqrt(3) + lin_a
    return adv, ret, bound_a, bound_r


def _dc_gae(rewards, dones, values, last_values, T, gamma, lam, adv, ret):
    from dronechase_b200 import _lib
    p = lambda t: C.c_void_p(t.data_ptr())                            # noqa: E731
    _lib.check(_lib.lib().dc_gae(p(rewards), p(dones), p(values), p(last_values), T, rewards.shape[1], float(gamma), float(lam),
                                 p(adv), p(ret), C.c_void_p(torch.cuda.current_stream().cuda_stream)), "dc_gae")


def _dones(pattern, T, E, rng):
    d = np.zeros((T, E), np.uint8)
    if pattern == "10%":
        d[:] = rng.random((T, E)) < 0.1
    elif pattern == "all":
        d[:] = 1
    elif pattern == "last":
        d[T - 1] = 1
    elif pattern == "first":
        d[0] = 1
    return d


GAMMA_LAMBDA = [(0.99, 0.95), (1.0, 1.0), (0.0, 0.95), (0.99, 0.0), (1.0, 0.0)]
DONES = ["10%", "none", "all", "last", "first"]


@pytest.mark.parametrize("T,E", [(1, 1), (1, 257), (7, 255), (128, 256), (33, 65537), (1024, 300)])
def test_dc_gae_against_the_float64_recurrence(T, E):
    """Every (gamma, lambda) x done pattern on this shape, called with T rows of a buffer of T + 2: the rows past T (NaN in
    and out) must be neither read nor written.  dc_gae and a float32 numpy loop of the same recurrence both stay within the
    bound of _gae_reference; on the large shapes the numpy loop reaches a quarter of it somewhere (the bound is not vacuous)."""
    from tests.test_actor_critic_cpu import gae_formula
    rng = np.random.default_rng(T * 100003 + E)
    rows = T + 2
    worst_kernel = worst_loop = 0.0
    for gamma, lam in GAMMA_LAMBDA:
        for pattern in DONES:
            rewards = rng.normal(size=(rows, E)).astype(np.float32)
            values = (rng.normal(size=(rows, E)) * 3 + 1).astype(np.float32)
            last_values = (rng.normal(size=E) * 3 + 1).astype(np.float32)
            dones = np.ones((rows, E), np.uint8)
            dones[:T] = _dones(pattern, T, E, rng)
            rewards[T:] = np.nan
            values[T:] = np.nan
            adv64, ret64, bound_a, bound_r = _gae_reference(rewards[:T], values[:T], dones[:T], last_values, gamma, lam)
            # the plain float32 loop, coefficients as float32
            g32, l32 = float(np.float32(gamma)), float(np.float32(lam))
            adv32, ret32 = gae_formula(rewards[:T], values[:T], dones[:T], last_values, g32, l32)
            assert adv32.dtype == np.float32
            loop = max(float((np.abs(adv32 - adv64) / bound_a).max()), float((np.abs(ret32 - ret64) / bound_r).max()))
            assert loop <= 1.0, f"gamma={gamma} lambda={lam} dones={pattern}: the float32 loop exceeds the bound ({loop:.3g})"
            dev = {k: torch.from_numpy(x).cuda() for k, x in (("r", rewards), ("v", values), ("lv", last_values), ("d", dones))}
            adv = torch.full((rows, E), math.nan, device="cuda")
            ret = torch.full((rows, E), math.nan, device="cuda")
            _dc_gae(dev["r"], dev["d"], dev["v"], dev["lv"], T, gamma, lam, adv, ret)
            a, rr = adv.cpu().numpy(), ret.cpu().numpy()
            tag = f"gamma={gamma} lambda={lam} dones={pattern}"
            assert np.isnan(a[T:]).all() and np.isnan(rr[T:]).all(), f"{tag}: rows past T were written"
            assert np.isfinite(a[:T]).all() and np.isfinite(rr[:T]).all(), f"{tag}: rows below T not written, or rows past T read"
            ka = float((np.abs(a[:T] - adv64) / bound_a).max())
            kr = float((np.abs(rr[:T] - ret64) / bound_r).max())
            assert ka <= 1.0 and kr <= 1.0, f"{tag}: dc_gae exceeds the float32 bound (advantages {ka:.3g}, returns {kr:.3g} of it)"
            worst_kernel, worst_loop = max(worst_kernel, ka, kr), max(worst_loop, loop)
    print(f"T={T} E={E}: largest error / bound: dc_gae {worst_kernel:.3g}, float32 loop {worst_loop:.3g}")
    if T * E >= 30000:
        assert worst_loop >= 0.25, f"the bound is more than 4x the float32 loop's largest error ({worst_loop:.3g})"


# ------------------------------------------------------------------------------------------------------------- PPORollout
def _env(E, env_offset):
    from dronechase_b200 import BatchedThreatEngageEnv
    env = BatchedThreatEngageEnv("exp02_v2_full", n_envs=E, seed=3, device=0, env_offset=env_offset, auto_reset=True,
                                 with_hits=True)
    env.reset()
    return env


def test_ppo_rollout_of_an_env_window_is_the_same_rows_of_the_whole_batch():
    """Envs [512, 768) collected as a batch of their own (env_offset = 512) and inside a batch of 1024: the same env seed,
    rollout seed and weights give the same bits for everything the rollout stores."""
    from dronechase_b200.policy import LidarInertialActorCritic
    from dronechase_b200.rollout import PPORollout
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    T, lo, hi = 16, 512, 768
    big, small = _env(1024, 0), _env(hi - lo, lo)
    assert small.env_offset == lo
    ac = LidarInertialActorCritic(env=big, seed=0)
    with torch.no_grad():
        ac.log_std.copy_(torch.tensor(LOG_STD))
    fused = ac.fused()
    out = []
    for env in (big, small):
        ro = PPORollout(env, T, seed=0xFEDC_BA98_7654_3210)
        ro.collect(fused).compute_returns_and_advantage(0.99, 0.95)
        out.append(ro)
    a, b = out
    assert int(a.dones[:, lo:hi].sum()) > 0, "no episode ended in the window: resets were not exercised"
    for name in ("actions", "log_probs", "values", "rewards", "dones", "advantages", "returns"):
        x, y = getattr(a, name), getattr(b, name)
        assert torch.equal(x[:, lo:hi], y), f"{name}: the window differs from the same rows of the whole batch"
    assert torch.equal(a.last_values[lo:hi], b.last_values)
    assert torch.equal(a.env_actions[lo:hi], b.env_actions)
    fused.close(); big.close(); small.close()


def test_ppo_rollout_counter_carries_across_collects_and_a_partial_collect_bootstraps_gae():
    """collect(3) then collect(2): the counter is 5 and step t of the second collect draws policy_normals(seed, 3 + t,
    env_offset + e) (action_net = 0, log_std = 0: the stored raw action IS eps); the GAE of the partial collect is the float64
    recurrence over its two steps, bootstrapped from V(s_2), and leaves the other rows alone."""
    from dronechase_b200.policy import LidarInertialActorCritic
    from dronechase_b200.rollout import PPORollout
    from oracle.policy_ac_fragment_model import policy_normals
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    E, off, seed = 200, 700, 0xFEDC_BA98_7654_3210
    env = _env(E, off)
    ac = LidarInertialActorCritic(env=env, seed=1)
    with torch.no_grad():
        ac.action_net.weight.zero_(); ac.action_net.bias.zero_()
    fused = ac.fused()
    ro = PPORollout(env, 8, seed=seed)
    ro.collect(fused, n_steps=3)
    assert ro.counter == 3 and ro.pos == 3
    first = ro.actions[:3].double().cpu().numpy()
    for t in range(3):
        assert np.abs(first[t] - policy_normals(seed, t, off + np.arange(E))).max() < 1e-5, f"first collect, step {t}"
    ro.advantages.fill_(math.nan); ro.returns.fill_(math.nan)
    obs_before = {k: x.clone() for k, x in env.obs.items()}
    ro.collect(fused, n_steps=2)
    assert ro.counter == 5 and ro.pos == 2
    for t in range(2):
        eps = ro.actions[t].double().cpu().numpy()
        assert np.abs(eps - policy_normals(seed, 3 + t, off + np.arange(E))).max() < 1e-5, f"second collect, step {t}"
    assert np.array_equal(ro.actions[2].double().cpu().numpy(), first[2]), "the second collect wrote past its two steps"
    with torch.no_grad():
        v_before = fused.values(obs_before)
    assert torch.equal(ro.values[0], v_before)
    ro.compute_returns_and_advantage(0.99, 0.95)
    np_ = lambda x: x.cpu().numpy()                                  # noqa: E731
    adv64, ret64, bound_a, bound_r = _gae_reference(np_(ro.rewards[:2]), np_(ro.values[:2]), np_(ro.dones[:2]),
                                                    np_(ro.last_values), 0.99, 0.95)
    assert (np.abs(np_(ro.advantages[:2]) - adv64) <= bound_a).all()
    assert (np.abs(np_(ro.returns[:2]) - ret64) <= bound_r).all()
    assert bool(ro.advantages[2:].isnan().all()) and bool(ro.returns[2:].isnan().all()), "GAE ran past the collected steps"
    assert float(ro.advantages[:2].abs().max()) > 0
    fused.close(); env.close()
