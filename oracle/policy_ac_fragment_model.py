"""TEST INFRASTRUCTURE (never imported by the product): a lane-by-lane numpy model of the actor-critic instantiation of
dronechase_b200/csrc/policy_kernel.cu (policy_ac_kernel, dc_policy_act), built on the trunk, dense layer, head, fragment
layout, packed weight order and MMA model of oracle/policy_fragment_model.py.

It restates what the actor-critic kernel adds, in float64, on the same flat shared-memory array act | red | stash: the
features copied into the stash (row stride SV) after final_layer, the vf layers in place in the stash, the last one streamed
into the 1-wide value head with its partial sums in red, value_net on the stash when vf == (), the second final_layer into the
stash when pi == (), and ``policy_normals``, the Box-Muller noise of the sampling epilogue.  tests/test_actor_critic_cpu.py
compares it with the torch module; tests/test_gpu_actor_critic.py uses ``policy_normals`` as the float64 reference of the
kernel's noise.
"""
from __future__ import annotations

import numpy as np

from oracle.philox import philox4x32
from oracle.policy_fragment_model import BM, FINAL_LAYER, RED, STASH, S, SV, _dense, _head, _trunk

STREAM_POLICY = 5


def policy_normals(seed: int, counter: int, env) -> np.ndarray:
    """The four standard normals of the sampling epilogue for global env indices ``env``, float64: Philox4x32-10 with key seed
    and counter (counter, STREAM_POLICY, env, 0); k = 0, 1 from words (0, 1), k = 2, 3 from words (2, 3)."""
    x = philox4x32(np.uint32(counter & 0xFFFFFFFF), np.uint32(STREAM_POLICY), np.asarray(env, dtype=np.uint32), 0,
                   seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    out = []
    for a, b in ((x[0], x[1]), (x[2], x[3])):
        r = np.sqrt(-2.0 * np.log(((a >> np.uint32(8)).astype(np.float64) + 1.0) / 16777216.0))
        ang = np.pi * (b >> np.uint32(8)).astype(np.float64) / 8388608.0
        out += [r * np.cos(ang), r * np.sin(ang)]
    return np.stack(out, axis=-1)


def forward_ac(weights: dict, value: dict, lidar, inertial, last_action, activation=2):
    """The actor-critic kernel over one block of <= 64 envs: (mean action, unclipped [E][4]; value [E]).  weights: as
    policy_fragment_model.forward; value: vf_w / vf_b lists (mlp_extractor.value_net), value_w [1][N], value_b [1]."""
    E = lidar.shape[0]
    smem, layers, inputs = _trunk(weights, lidar, inertial, last_action, activation, stash=True)
    red, stash = smem[RED:STASH], smem[STASH:]
    # ---- last layer + head
    W, b, in_off, _, a_fn, _ = layers[-1]
    mean = (weights["head_b"][None, :] + _head(smem, S, W, b, in_off, a_fn, weights["head_w"], red))[:E]
    # ---- value branch: red is free again
    red[:] = np.nan
    if len(layers) == FINAL_LAYER + 1:                         # pi == (): final_layer once more, into the stash
        _dense(smem, S, stash, SV, *layers[FINAL_LAYER], inputs)
    vf = list(zip(value["vf_w"], value["vf_b"]))
    for W, b in vf[:-1]:
        _dense(stash, SV, stash, SV, W, b, 0, 0, activation, 0, inputs)
    if vf:
        W, b = vf[-1]
        v = value["value_b"][0] + _head(stash, SV, W, b, 0, activation, value["value_w"], red)[:, 0]
    else:
        F = layers[FINAL_LAYER][0].shape[0]
        v = value["value_b"][0] + stash.reshape(BM, SV)[:, :F] @ value["value_w"][0]
    return mean, v[:E]
