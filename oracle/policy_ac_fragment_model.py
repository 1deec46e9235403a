"""TEST INFRASTRUCTURE (never imported by the product): a lane-by-lane numpy model of the actor-critic instantiation of
dronechase_b200/csrc/policy_kernel.cu (policy_ac_kernel, dc_policy_act), built on the fragment layout, packed weight order and
MMA model of oracle/policy_fragment_model.py.

It restates what the actor-critic kernel adds, in float64: act, red and the feature stash as ONE flat shared-memory array (so
that a wrong row stride or base shows up), the features copied into the stash (row stride SV) after final_layer, the vf layers
in place in the stash, the last one streamed into the 1-wide value head with its partial sums in red, value_net on the stash
when vf == (), the second final_layer into the stash when pi == (), and ``policy_normals``, the Box-Muller noise of the sampling
epilogue.  The trunk (conv1, conv2, the input MLPs) is the same arithmetic as policy_fragment_model.forward, restated here on
the flat array.  tests/test_actor_critic_cpu.py compares it with the torch module; tests/test_gpu_actor_critic.py uses
``policy_normals`` as the float64 reference of the kernel's noise.
"""
from __future__ import annotations

import numpy as np

from oracle.philox import philox4x32
from oracle.policy_fragment_model import BM, G, LANE, S, T, WARPS, _act, mma, mma_block, pack

SV, MAX_UNITS, STREAM_POLICY = 260, 32, 5


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


def _dense(src, ldi, dst, ldo, W, b, in_off, out_off, a_fn, sel, inputs, E):
    """dense_layer<.., LDI, LDO>: rows of `src` / `dst` (flat shared-memory arrays) at stride ldi / ldo."""
    N, K = W.shape
    KS, w = (K + 7) // 8, pack(W)
    MT, NT = (1, 4) if N in (128, 64) else (2, 4)              # DCP_WIDE = 1: 32 x 32 warp tiles for the wide layers
    RG = BM // (16 * MT)
    results = {}
    for warp in range(WARPS):
        rg, cc = warp % RG, warp // RG
        row0, nt0 = rg * 16 * MT, cc * NT
        if nt0 * 8 >= N:
            continue

        def aload(mt, ks, row0=row0):
            ra, rb = row0 + mt * 16 + G, row0 + mt * 16 + G + 8
            k0, k1 = ks * 8 + T, ks * 8 + T + 4
            if sel == 0:
                return np.stack([src[ra * ldi + in_off + k0], src[rb * ldi + in_off + k0], src[ra * ldi + in_off + k1],
                                 src[rb * ldi + in_off + k1]], axis=1)
            x = inputs[sel]
            a = np.zeros((32, 4))
            for i, (rows, k) in enumerate(((ra, k0), (rb, k0), (ra, k1), (rb, k1))):
                ok = (rows < E) & (k < K)
                a[ok, i] = x[rows[ok], k[ok]]
            return a
        results[warp] = (mma_block(MT, NT, aload, KS, w, nt0), row0, nt0)
    for warp, (acc, row0, nt0) in results.items():            # after the barrier
        for mt in range(MT):
            for j in range(NT):
                col = (nt0 + j) * 8 + 2 * T
                r = row0 + mt * 16 + G
                dst[r * ldo + out_off + col] = _act(acc[mt, j][:, 0] + b[col], a_fn)
                dst[r * ldo + out_off + col + 1] = _act(acc[mt, j][:, 1] + b[col + 1], a_fn)
                dst[(r + 8) * ldo + out_off + col] = _act(acc[mt, j][:, 2] + b[col], a_fn)
                dst[(r + 8) * ldo + out_off + col + 1] = _act(acc[mt, j][:, 3] + b[col + 1], a_fn)


def _head(src, ld, W, b, in_off, a_fn, hw, red):
    """head_layer<2, 4, X3, NH, LD>: the last hidden layer streamed into the NH = len(hw) outputs; partial sums into
    red[unit][row][k] (a flat view of the kernel's red array).  Returns the number of units."""
    N, K = W.shape
    NH = hw.shape[0]
    KS, w = (K + 7) // 8, pack(W)
    MT, NT, RG = 2, 4, 2                                       # units of 32 columns, 8 per pass
    CP = WARPS // RG
    n_units = N // (NT * 8)
    for p4 in range((n_units + CP - 1) // CP):
        for warp in range(WARPS):
            rg, cc = warp % RG, warp // RG
            unit, row0 = p4 * CP + cc, rg * 16 * MT
            if unit >= n_units:
                continue

            def aload(mt, ks, row0=row0):
                ra = row0 + mt * 16 + G
                k0 = in_off + ks * 8 + T
                return np.stack([src[ra * ld + k0], src[(ra + 8) * ld + k0], src[ra * ld + k0 + 4], src[(ra + 8) * ld + k0 + 4]], axis=1)
            acc = mma_block(MT, NT, aload, KS, w, unit * NT)
            for mt in range(MT):
                part = np.zeros((2, 32, NH))
                for j in range(NT):
                    col = (unit * NT + j) * 8 + 2 * T
                    h = [_act(acc[mt, j][:, 0] + b[col], a_fn), _act(acc[mt, j][:, 1] + b[col + 1], a_fn),
                         _act(acc[mt, j][:, 2] + b[col], a_fn), _act(acc[mt, j][:, 3] + b[col + 1], a_fn)]
                    for k in range(NH):
                        part[0, :, k] += h[0] * hw[k, col] + h[1] * hw[k, col + 1]
                        part[1, :, k] += h[2] * hw[k, col] + h[3] * hw[k, col + 1]
                for hh in range(2):
                    quad = part[hh].reshape(8, 4, NH).sum(axis=1)           # the two shfl_xor steps: sum over t
                    rows = row0 + mt * 16 + hh * 8 + np.arange(8)
                    for k in range(NH):
                        red[(unit * BM + rows) * NH + k] = quad[:, k]
    return n_units


def forward_ac(weights: dict, value: dict, lidar, inertial, last_action, activation=2):
    """The actor-critic kernel over one block of <= 64 envs: (mean action, unclipped [E][4]; value [E]).  weights: as
    policy_fragment_model.forward; value: vf_w / vf_b lists (mlp_extractor.value_net), value_w [1][N], value_b [1]."""
    E, C = lidar.shape[0], lidar.shape[1]
    lid = lidar.reshape(E, -1)
    smem = np.full(BM * S + MAX_UNITS * BM * 4 + BM * SV, np.nan)       # act | red | stash
    act_flat, red = smem[:BM * S], smem[BM * S:BM * S + MAX_UNITS * BM * 4]
    stash = smem[BM * S + MAX_UNITS * BM * 4:]
    act = act_flat.reshape(BM, S)
    act[:] = 0.0
    # ---- conv1
    w1, KS1 = pack(weights["conv1_w"], ntg=4), 2 * C
    for warp in range(WARPS):
        for p3 in range(3):
            mti = warp * 3 + p3
            patch = mti >> 2; py, px = patch // 6, patch % 6
            el = (mti & 3) * 16 + G
            acc = np.zeros((4, 32, 4))
            for ks in range(KS1):
                off = ((ks >> 1) * 13 + 4 * py + (ks & 1) * 2) * 26 + 4 * px + T
                a = np.zeros((32, 4))
                for i, (rows, o) in enumerate(((el, off), (el + 8, off), (el, off + 26), (el + 8, off + 26))):
                    ok = rows < E
                    a[ok, i] = lid[rows[ok], o[ok]]
                for j in range(4):
                    mma(acc[j], a, w1[(ks * 4 + j) * 32 + LANE])
            for j in range(4):
                col = j * 8 + 2 * T
                b0, b1 = weights["conv1_b"][col], weights["conv1_b"][col + 1]
                act[el, patch * 32 + col] = np.maximum(acc[j][:, 0] + b0, 0); act[el, patch * 32 + col + 1] = np.maximum(acc[j][:, 1] + b1, 0)
                act[el + 8, patch * 32 + col] = np.maximum(acc[j][:, 2] + b0, 0); act[el + 8, patch * 32 + col + 1] = np.maximum(acc[j][:, 3] + b1, 0)
    # ---- conv2
    w2 = pack(weights["conv2_w"], kmap=1, ntg=4)
    outs = []
    for warp in range(WARPS):
        qn, mg = warp & 3, warp >> 2

        def aload(mt, ks, mg=mg):
            mtile = mg * 3 + mt; wpos, el = mtile >> 2, (mtile & 3) * 16 + G
            q = ks >> 2; ky, kx, c = q >> 1, q & 1, (ks & 3) * 8 + T
            col = (ky * 6 + 2 * wpos + kx) * 32 + c
            return np.stack([act[el, col], act[el + 8, col], act[el, col + 4], act[el + 8, col + 4]], axis=1)
        outs.append(mma_block(3, 2, aload, 16, w2, qn * 2, NTG=4))
    for warp in range(WARPS):                                   # after the barrier
        qn, mg = warp & 3, warp >> 2
        for mt in range(3):
            mtile = mg * 3 + mt; wpos, el = mtile >> 2, (mtile & 3) * 16 + G
            for j in range(2):
                n = (qn * 2 + j) * 8 + 2 * T
                b0, b1 = weights["conv2_b"][n], weights["conv2_b"][n + 1]
                a = outs[warp][mt, j]
                act[el, n * 3 + wpos] = np.maximum(a[:, 0] + b0, 0); act[el, (n + 1) * 3 + wpos] = np.maximum(a[:, 1] + b1, 0)
                act[el + 8, n * 3 + wpos] = np.maximum(a[:, 2] + b0, 0); act[el + 8, (n + 1) * 3 + wpos] = np.maximum(a[:, 3] + b1, 0)
    # ---- dense layers
    layers = []
    for i in range(3):
        layers.append((weights["inertial_w"][i], weights["inertial_b"][i], 0 if i == 0 else 192, 192, 1, 1 if i == 0 else 0))
    for i in range(3):
        layers.append((weights["action_w"][i], weights["action_b"][i], 0 if i == 0 else 320, 320, 1, 2 if i == 0 else 0))
    layers.append((weights["final_w"], weights["final_b"], 0, 0, 1, 0))
    for W, b in zip(weights["pi_w"], weights["pi_b"]):
        layers.append((W, b, 0, 0, activation, 0))
    inputs = {1: inertial, 2: last_action}
    FINAL = 6
    for li, (W, b, in_off, out_off, a_fn, src) in enumerate(layers[:-1]):
        _dense(act_flat, S, act_flat, S, W, b, in_off, out_off, a_fn, src, inputs, E)
        if li == FINAL:                                        # the features -> the stash
            F = W.shape[0]
            for r in range(BM):
                stash[r * SV:r * SV + F] = act_flat[r * S:r * S + F]
    # ---- last layer + head
    W, b, in_off, _, a_fn, _ = layers[-1]
    n_units = _head(act_flat, S, W, b, in_off, a_fn, weights["head_w"], red)
    mean = (weights["head_b"][None, :] + red[:n_units * BM * 4].reshape(n_units, BM, 4).sum(axis=0))[:E]
    # ---- value branch: red is free again
    red[:] = np.nan
    if len(layers) == FINAL + 1:                               # pi == (): final_layer once more, into the stash
        W, b, in_off, out_off, a_fn, src = layers[FINAL]
        _dense(act_flat, S, stash, SV, W, b, in_off, out_off, a_fn, src, inputs, E)
    vf = list(zip(value["vf_w"], value["vf_b"]))
    for W, b in vf[:-1]:
        _dense(stash, SV, stash, SV, W, b, 0, 0, activation, 0, inputs, E)
    if vf:
        W, b = vf[-1]
        n_units = _head(stash, SV, W, b, 0, activation, value["value_w"], red)
        v = value["value_b"][0] + red[:n_units * BM].reshape(n_units, BM).sum(axis=0)
    else:
        F = layers[FINAL][0].shape[0]
        v = value["value_b"][0] + stash.reshape(BM, SV)[:, :F] @ value["value_w"][0]
    return mean, v[:E]
