"""CPU oracle of the ray-cast LiDAR as the agent's sensor of a stage03 env (``TaskConfig(lidar="raycast")``).

TEST INFRASTRUCTURE, not the product.  The reference has no ray cast (SURVEY.md section 8(f) rank 4), so this sensor's
parity is unpinned by it; it is property-pinned:
  * with zero radii the sphere and the ids are ``env_oracle.lidar_project``'s fused ones (the projection pinned by
    tests/golden);
  * for an observer outside every bounding sphere and away from ties it agrees with ``oracle.lidar_raycast``, the ray-cast
    definition of the stand-alone ``dc_lidar_raycast`` (tests/test_raycast_env_cpu.py checks both).
Where that definition leaves the env sensor open, this module fixes it -- and ``raycast_sphere_kernel`` follows it:
  * the rays and the centre claims are taken from the snapshot the fused flavour projects from (float32 IMU positions and
    attitude of the agent, the entities alive after the engagement);
  * an observer inside (or on) a bounding sphere sees that entity at distance 0 in every cell;
  * a radius of 0 casts no ray: the entity only claims the cell of its centre;
  * a cell's candidates are the entities in slot order, each with the smaller of its ray hit and its centre claim, and the
    winner is picked by FusedLIDAR.add_features' rule (strict '<' of the float64 value against the float32 value the cell
    holds) -- nearest first, the fused flavour's tie rule after;
  * the radii are float32, as ``dc_set_ray_radii`` takes them.
"""
from __future__ import annotations

import numpy as np

from . import dynamics as dy
from .env_oracle import LM_TYPE, LW_TYPE, N_PHI, N_THETA, EnvOracle

_TI, _PJ = np.meshgrid(np.arange(N_THETA), np.arange(N_PHI), indexing="ij")
_TH = (_TI.ravel() + 0.5) / N_THETA * np.pi
_PH = -np.pi + (_PJ.ravel() + 0.5) / N_PHI * 2 * np.pi
CELL_RAYS = np.stack([np.sin(_TH) * np.cos(_PH), np.sin(_TH) * np.sin(_PH), np.cos(_TH)], axis=1)   # body frame, [338, 3]


def centre_claim(own_p32, own_q32, p):
    """(cell, r_n float64 before the [0, 1] clip) of one entity: the fused flavour of env_oracle.lidar_project."""
    nsq = np.dot(own_q32, own_q32)
    qinv = np.array([-own_q32[0], -own_q32[1], -own_q32[2], own_q32[3]], dtype=np.float32) / nsq
    rel = dy.rot_from_quat(qinv.astype(np.float64)) @ (np.asarray(p, dtype=np.float32).astype(np.float64) - own_p32.astype(np.float64))
    x, y, z = rel
    r = np.sqrt(x * x + y * y + z * z)
    theta, phi = (0.0, 0.0) if r == 0 else (np.arccos(np.clip(z / r, -1.0, 1.0)), np.arctan2(y, x))
    ti = int(np.clip(int(theta / np.pi * N_THETA), 0, N_THETA - 1))
    pj = int(np.clip(int((phi + np.pi) / (2 * np.pi) * N_PHI), 0, N_PHI - 1))
    return ti * N_PHI + pj, r


def lidar_raycast_env(own_pos, own_quat, ent_pos, ent_type, ent_id, ent_radius, max_range):
    """Returns (sphere f32 (3,13,26), ids i32 (13,26), margin f64 (13,26)).

    margin (metres) = how far the cell is from changing its content: the smallest |miss distance - radius| of a ray that
    passes in front of the observer, |distance - radius| of a sphere the observer is inside or near, and the gap between
    the two best candidates of the cell.  A float32 build may legitimately differ where it is tiny."""
    own_p32 = np.asarray(own_pos).astype(np.float32)
    own_q32 = np.asarray(own_quat).astype(np.float32)
    # the offsets are taken into the frame of R(q) (R^T (e - o)) and met with the body-frame rays: rel . (R b) = (R^T rel) . b,
    # and the miss vector is formed where the rays are unit, whatever the float32 quaternion's norm
    R = dy.rot_from_quat(own_q32.astype(np.float64))
    cur = np.ones(N_THETA * N_PHI, dtype=np.float32)
    ids = np.full(N_THETA * N_PHI, -1, dtype=np.int32)
    margin = np.full(N_THETA * N_PHI, np.inf)
    vals = []
    for p, etype, eid, rad in zip(ent_pos, ent_type, ent_id, ent_radius):
        cell, rc = centre_claim(own_p32, own_q32, p)
        rn = min(max(rc / max_range, 0.0), 1.0)
        r = float(np.float32(rad))
        v = np.full(N_THETA * N_PHI, 2.0)
        if r > 0:
            rel = np.asarray(p, dtype=np.float32).astype(np.float64) - own_p32.astype(np.float64)
            rel2 = float(rel @ rel)
            margin = np.minimum(margin, abs(np.sqrt(rel2) - r))
            if rel2 <= r * r:
                v[:] = 0.0
            else:
                rel_b = R.T @ rel
                tca = CELL_RAYS @ rel_b
                d2 = ((rel_b[None, :] - tca[:, None] * CELL_RAYS) ** 2).sum(axis=1)        # squared miss distance
                front = tca > 0
                margin[front] = np.minimum(margin[front], np.abs(np.sqrt(np.maximum(d2[front], 0.0)) - r))
                hit = front & (d2 <= r * r)
                v[hit] = np.clip((tca[hit] - np.sqrt(r * r - d2[hit])) / max_range, 0.0, 1.0)
        v[cell] = min(v[cell], rn)
        vals.append(v)
        take = v < cur.astype(np.float64)
        cur[take] = v[take].astype(np.float32)
        ids[take] = eid
    if len(vals) >= 2:
        s = np.sort(np.stack(vals), axis=0)
        near = s[0] < 1.0
        margin[near] = np.minimum(margin[near], (s[1][near] - s[0][near]) * max_range)
    types = {int(i): t for i, t in zip(ent_id, ent_type)}
    sphere = np.ones((3, N_THETA * N_PHI), dtype=np.float32)
    held = ids >= 0
    sphere[0] = cur
    sphere[1, held] = [types[int(i)] / 5 for i in ids[held]]
    sphere[2, held] = 0.1
    return sphere.reshape(3, N_THETA, N_PHI), ids.reshape(N_THETA, N_PHI), margin.reshape(N_THETA, N_PHI)


class RaycastEnvOracle(EnvOracle):
    """EnvOracle whose agent senses with the ray-cast LiDAR; ``ray_margin[e]`` is the margin of env e's last observation
    (inf where the sphere was kept), ``ray_updated[e]`` whether that observation rebuilt the sphere."""

    def __init__(self, cfg, n_envs, ray_radius, **kw):
        self.ray_radius = (float(np.float32(ray_radius[0])), float(np.float32(ray_radius[1])))
        self.ray_margin = np.full((n_envs, N_THETA, N_PHI), np.inf)
        self.ray_updated = np.zeros(n_envs, dtype=bool)       # the agent's sphere was rebuilt at the last observation
        super().__init__(cfg, n_envs, **kw)

    def _lidar(self, e, obs_slot):
        self.ray_updated[e] = self.armed[e, obs_slot]
        if not self.armed[e, obs_slot]:
            self.ray_margin[e] = np.inf
            return super()._lidar(e, obs_slot)
        c = self.cfg
        others = [d for d in range(self.D) if d != obs_slot and self.armed[e, d]]
        types = [LW_TYPE if d < c.n_lw else LM_TYPE for d in others]
        radii = [self.ray_radius[0] if d < c.n_lw else self.ray_radius[1] for d in others]
        sphere, ids, self.ray_margin[e] = lidar_raycast_env(self.imu["position"][e, obs_slot], self.imu["quaternion"][e, obs_slot],
                                                            self.imu["position"][e, others], types, others, radii,
                                                            2 * c.dome_radius)
        return sphere, ids
