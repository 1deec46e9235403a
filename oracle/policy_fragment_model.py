"""TEST INFRASTRUCTURE (never imported by the product): a lane-by-lane numpy model of dronechase_b200/csrc/policy_kernel.cu.

It restates the kernel's INDEX ARITHMETIC -- the packed B-fragment order of pack_kernel, the A-fragment addresses of every
layer (conv1 patches read from the sphere, conv2's (ky, kx, channel) ordering over h1, the in-place dense layers, the
streamed last layer + action head) and the PTX fragment layout of mma.sync.m16n8k8 (row.col, tf32):

    A (16x8):  a0 = (g, t)   a1 = (g+8, t)   a2 = (g, t+4)   a3 = (g+8, t+4)
    B (8x8):   b0 = (k = t, n = g)           b1 = (k = t+4, n = g)
    C (16x8):  c0 = (g, 2t)  c1 = (g, 2t+1)  c2 = (g+8, 2t)  c3 = (g+8, 2t+1)        g = lane >> 2, t = lane & 3

in float64, so that a wrong offset shows up on the CPU (tests/test_policy_cpu.py compares it with the torch module of
dronechase_b200/policy.py, i.e. with ppo_policies.py:234-342) before any GPU time is spent.  Products are exact here: the
TF32 head/tail split of the kernel is not modelled.
"""
from __future__ import annotations

import numpy as np

BM, WARPS, S = 64, 16, 452
SV, MAX_UNITS, FINAL_LAYER = 260, 32, 6                      # stash row stride, head partial sums, layers[6] = final_layer
RED, STASH = BM * S, BM * S + MAX_UNITS * BM * 4            # offsets of red and the stash in the flat shared memory
LANE = np.arange(32)
G, T = LANE >> 2, LANE & 3


def pack(W: np.ndarray, kmap: int = 0, ntg: int = 8) -> np.ndarray:
    """[N][K] -> [(N/8) * KS * 32][2] in the order pack_kernel writes: [group of ntg n-tiles][k-step][n-tile in group][lane]."""
    N, K = W.shape
    KS = (K + 7) // 8
    out = np.zeros(((N // 8) * KS * 32, 2))
    for idx in range(out.shape[0]):
        lane, j, ks = idx & 31, (idx >> 5) % ntg, ((idx >> 5) // ntg) % KS
        nt = ((idx >> 5) // (ntg * KS)) * ntg + j
        g, t, n = lane >> 2, lane & 3, nt * 8 + (lane >> 2)
        for i in range(2):
            k = ks * 8 + t + 4 * i
            if kmap == 1:
                out[idx, i] = W[n, (k & 31) * 4 + (k >> 5)]
            else:
                out[idx, i] = W[n, k] if k < K else 0.0
    return out


def mma(acc, a, b):
    """acc [32][4] += fragments a [32][4] x b [32][2] of one warp (the PTX layout in the module docstring)."""
    A = np.zeros((16, 8)); B = np.zeros((8, 8))
    A[G, T] = a[:, 0]; A[G + 8, T] = a[:, 1]; A[G, T + 4] = a[:, 2]; A[G + 8, T + 4] = a[:, 3]
    B[T, G] = b[:, 0]; B[T + 4, G] = b[:, 1]
    C = A @ B
    acc[:, 0] += C[G, 2 * T]; acc[:, 1] += C[G, 2 * T + 1]; acc[:, 2] += C[G + 8, 2 * T]; acc[:, 3] += C[G + 8, 2 * T + 1]


def mma_block(MT, NT, aload, KS, w, nt0, NTG=8):
    """A warp consumes NT n-tiles (from nt0) of a packed group of NTG."""
    acc = np.zeros((MT, NT, 32, 4))
    for ks in range(KS):
        a = [aload(mt, ks) for mt in range(MT)]
        for j in range(NT):
            b = w[(((nt0 // NTG) * KS + ks) * NTG + (nt0 % NTG) + j) * 32 + LANE]
            for mt in range(MT):
                mma(acc[mt, j], a[mt], b)
    return acc


def _act(x, act):
    return np.maximum(x, 0) if act == 1 else np.tanh(x) if act == 2 else x


def _dense(src, ldi, dst, ldo, W, b, in_off, out_off, a_fn, sel, inputs):
    """dense_layer<MT, NT, X3, LDI, LDO> as hidden_layer picks the tile: rows of `src` / `dst` (flat shared-memory arrays) at
    stride ldi / ldo; sel 1 / 2 reads the rows of inputs[sel] (inertial vector / last action) instead."""
    N, K = W.shape
    KS, w = (K + 7) // 8, pack(W)
    MT, NT = (1, 4) if N in (128, 64) else (2, 4)              # 16 x 32 warp tiles for 64 and 128 columns, 32 x 32 otherwise
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
                ok = (rows < len(x)) & (k < K)
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
    """head_layer<2, 4, X3, NH, LD> + head_sum<NH>: the last hidden layer streamed into the NH = len(hw) outputs, partial sums
    into red[unit][row][k] (a flat view of the kernel's red array), then added over the units.  Returns [BM][NH], no bias."""
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
    return red[:n_units * BM * NH].reshape(n_units, BM, NH).sum(axis=0)


def _trunk(weights: dict, lidar, inertial, last_action, activation=2, stash=False):
    """conv1, conv2 and every dense layer but the last hidden one, in place in act, over one block of <= 64 envs.  The
    shared memory is ONE flat array act | red | stash (the actor-critic kernel's layout; the plain kernel stops after red),
    filled with NaN so that a read at a wrong row stride or base shows up.  stash: copy the features (final_layer's output)
    into the stash at row stride SV, as the actor-critic kernel does.  Returns (smem, layers, inputs): layers are
    (W, b, in_off, out_off, activation, source) of every dense layer, the last one included; inputs the arrays of sources 1, 2."""
    E, C = lidar.shape[0], lidar.shape[1]
    lid = lidar.reshape(E, -1)
    smem = np.full(STASH + BM * SV, np.nan)
    act = smem[:RED].reshape(BM, S)
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
    for li, layer in enumerate(layers[:-1]):
        _dense(smem, S, smem, S, *layer, inputs)
        if stash and li == FINAL_LAYER:                        # the features -> the stash
            F = layer[0].shape[0]
            for r in range(BM):
                smem[STASH + r * SV:STASH + r * SV + F] = smem[r * S:r * S + F]
    return smem, layers, inputs


def forward(weights: dict, lidar, inertial, last_action, low, high, activation=2):
    """weights: conv1_w [32][C*16], conv1_b, conv2_w [64][128], conv2_b, inertial_w/b[3], action_w/b[3], final_w/b, pi_w/b lists,
    head_w [4][N], head_b (float64 arrays in torch layout, convs flattened).  One block of <= 64 envs."""
    smem, layers, _ = _trunk(weights, lidar, inertial, last_action, activation)
    W, b, in_off, _, a_fn, _ = layers[-1]
    out = weights["head_b"][None, :] + _head(smem, S, W, b, in_off, a_fn, weights["head_w"], smem[RED:STASH])
    return np.clip(out, low, high)[:lidar.shape[0]]
