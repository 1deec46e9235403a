"""Device-resident rollout storage (SURVEY.md section 8(f), rank 1).

The reference collects rollouts through SB3's ``RolloutBuffer``: every env step the observation dict crosses to the
host as numpy, is copied into the buffer, and goes back to the device for the policy update
(src/core/rl_framework/utils/pipeline.py:214-241, stable-baselines3 ``OnPolicyAlgorithm.collect_rollouts``).  Here the
rollout stays in HBM.  The (3,13,26) sphere -- 4 KB per env step, 99 % of it 1.0 -- is stored as the hit list the
simulator already maintains (``dc_buffers.lidar_hits``: 8 B per drone slot) and rebuilt by ``dc_scatter_hits`` for the
time steps or the minibatch rows that are asked for: 128 steps x 65,536 envs take 1.1 GB instead of 35 GB.

    env = BatchedThreatEngageEnv("exp02_vFinal", n_envs=65536, with_hits=True)
    ro = DeviceRollout(env, n_steps=128)
    ro.collect(policy)                      # policy: obs dict of CUDA tensors -> actions [E,4] CUDA tensor
    batch = ro.minibatch(torch.randperm(ro.n_steps * env.n_envs, device="cuda")[:4096])

level5 (threatsense): the stacked observation (6,3,13,26) -- 24 KB per env step -- is stored as ITS hit list (at most
8 * (5 D + 1) bytes, -1 terminated; ``dc_scatter_stack`` rebuilds it) with the 6-byte validity mask beside it; the batch
key is ``stacked_spheres`` + ``validity_mask`` instead of ``lidar``.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Dict, Optional

import torch

from . import _lib
from .sim import BatchedThreatEngageEnv


class DeviceRollout:
    def __init__(self, env: BatchedThreatEngageEnv, n_steps: int):
        if env.cfg.lidar == "raycast":
            raise _lib.DroneChaseError("the rollout stores the sphere as its hit list, one (cell, r_n) per drone slot, which "
                                       "cannot describe a ray-cast sphere (lidar='raycast'); hit-list storage of ray-cast "
                                       "spheres is not built")
        if env.lidar_hits is None:
            raise _lib.DroneChaseError("create the env with with_hits=True: the rollout stores the sphere as its hit list")
        self.env, self.n_steps = env, int(n_steps)
        T, E, D, dev = self.n_steps, env.n_envs, env.cfg.n_drones, env.device
        self.channels = env.cfg.lidar_channels
        self.level5 = env.cfg.family == "level5"
        f32 = dict(dtype=torch.float32, device=dev)
        # observation BEFORE the action of step t, as its hit list
        self.hits = torch.empty(T, E, 5 * D + 1 if self.level5 else D, 2, dtype=torch.int32, device=dev)
        self.mask = torch.empty(T, E, _lib.DC_LIDAR_STACK, dtype=torch.bool, device=dev) if self.level5 else None
        self.inertial = torch.empty(T, E, 15, **f32)
        self.last_action = torch.empty(T, E, 4, **f32)
        self.actions = torch.empty(T, E, 4, **f32)
        self.rewards = torch.empty(T, E, **f32)
        self.dones = torch.empty(T, E, dtype=torch.uint8, device=dev)
        self.pos = 0

    @property
    def bytes(self) -> int:
        return sum(t.numel() * t.element_size() for t in (self.hits, self.inertial, self.last_action, self.actions,
                                                          self.rewards, self.dones, self.mask) if t is not None)

    def _store_obs(self, t: int):
        e = self.env
        self.hits[t].copy_(e.lidar_hits, non_blocking=True)
        if self.level5:
            self.mask[t].copy_(e.obs["validity_mask"], non_blocking=True)
        self.inertial[t].copy_(e.obs["inertial_data"], non_blocking=True)
        self.last_action[t].copy_(e.obs["last_action"], non_blocking=True)

    def _step(self, t: int, env_actions: torch.Tensor):
        e = self.env
        e.step(env_actions)                                       # zero copy: the kernel reads the slab
        self.rewards[t].copy_(e.reward, non_blocking=True)
        self.dones[t].copy_(e.done, non_blocking=True)
        self.pos += 1

    def add(self, actions: torch.Tensor):
        """Store the env's CURRENT observation with `actions`, step the env, store reward and done (SB3 order)."""
        t = self.pos
        self._store_obs(t)
        if actions.data_ptr() != self.actions[t].data_ptr():      # a policy may have written the slab itself (FusedPolicy, out=)
            self.actions[t].copy_(actions, non_blocking=True)
        self._step(t, self.actions[t])

    def collect(self, policy: Callable[[Dict[str, torch.Tensor]], torch.Tensor], n_steps: Optional[int] = None):
        """Fill the buffer from position 0: actions = policy(env.obs) on the device, nothing touches the host."""
        self.pos = 0
        direct = hasattr(policy, "precision") and hasattr(policy, "refresh")      # policy.FusedPolicy: one kernel, writes the slab
        for _ in range(n_steps or self.n_steps):
            self.add(policy(self.env.obs, out=self.actions[self.pos]) if direct else policy(self.env.obs))
        return self

    def _scatter(self, hits: torch.Tensor, index: Optional[torch.Tensor], n_rows: int) -> torch.Tensor:
        e = self.env
        ip = C.c_void_p(index.data_ptr()) if index is not None else None
        if self.level5:
            out = torch.empty(n_rows, _lib.DC_LIDAR_STACK, 3, _lib.N_THETA, _lib.N_PHI, dtype=torch.float32, device=e.device)
            with torch.cuda.device(e.device):
                _lib.check(_lib.lib().dc_scatter_stack(C.c_void_p(hits.data_ptr()), ip, n_rows, e.cfg.n_drones, C.c_void_p(out.data_ptr()),
                                                       C.c_void_p(torch.cuda.current_stream(e.device).cuda_stream)), "dc_scatter_stack")
            return out
        out = torch.empty(n_rows, self.channels, _lib.N_THETA, _lib.N_PHI, dtype=torch.float32, device=e.device)
        with torch.cuda.device(e.device):
            _lib.check(_lib.lib().dc_scatter_hits(C.c_void_p(hits.data_ptr()), C.c_void_p(index.data_ptr()) if index is not None else None,
                                                  n_rows, e.cfg.n_drones, e.cfg.n_lw, self.channels, C.c_void_p(out.data_ptr()),
                                                  C.c_void_p(torch.cuda.current_stream(e.device).cuda_stream)), "dc_scatter_hits")
        return out

    def lidar(self, t: int) -> torch.Tensor:
        """Dense [E, C, 13, 26] (level5: [E, 6, 3, 13, 26]) observation of time step t."""
        return self._scatter(self.hits[t], None, self.env.n_envs)

    def minibatch(self, flat_index: torch.Tensor) -> Dict[str, torch.Tensor]:
        """Rows ``flat_index`` (int64 CUDA tensor over the flattened [T * E] axis) as a training batch."""
        idx = flat_index.to(device=self.env.device, dtype=torch.int64).contiguous()
        T, E = self.n_steps, self.env.n_envs
        lidar = self._scatter(self.hits, idx, idx.numel())
        obs = ({"stacked_spheres": lidar, "validity_mask": self.mask.view(T * E, -1)[idx]} if self.level5 else {"lidar": lidar})
        return {**obs,
                "inertial_data": self.inertial.view(T * E, 15)[idx], "last_action": self.last_action.view(T * E, 4)[idx],
                "actions": self.actions.view(T * E, 4)[idx], "rewards": self.rewards.view(T * E)[idx],
                "dones": self.dones.view(T * E)[idx]}


class PPORollout(DeviceRollout):
    """The device rollout of SB3's ``collect_rollouts`` for PPO: per step ONE actor-critic kernel launch
    (``FusedPolicy.act`` of a ``LidarInertialActorCritic``) samples the action, its log-probability and V(s); ``actions``
    keeps the unclipped sample, as SB3's buffer does, and the env steps on the clipped copy.  After the loop V(s_T) goes to
    ``last_values`` and ``compute_returns_and_advantage`` runs GAE in one kernel (``dc_gae``).

        env = BatchedThreatEngageEnv("exp02_v2_full", n_envs=65536, with_hits=True)
        ro = PPORollout(env, n_steps=128, seed=1)
        fused = LidarInertialActorCritic(env=env).fused()
        ro.collect(fused).compute_returns_and_advantage(gamma=0.99, gae_lambda=0.95)
        batch = ro.minibatch(torch.randperm(ro.n_steps * env.n_envs, device="cuda")[:4096])

    The noise of env e at a step is a pure function of (seed, counter, env.env_offset + e); the counter counts the steps
    this rollout has collected, across ``collect`` calls.  level5 is not supported: its stacked observation is not what
    the fused kernel reads."""

    def __init__(self, env: BatchedThreatEngageEnv, n_steps: int, seed: int = 0):
        if env.cfg.family == "level5":
            raise _lib.DroneChaseError("PPORollout: level5's stacked observation is not what the fused policy kernel reads")
        super().__init__(env, n_steps)
        T, E = self.n_steps, env.n_envs
        f32 = dict(dtype=torch.float32, device=env.device)
        self.values = torch.empty(T, E, **f32)
        self.log_probs = torch.empty(T, E, **f32)
        self.advantages = torch.zeros(T, E, **f32)
        self.returns = torch.zeros(T, E, **f32)
        self.last_values = torch.zeros(E, **f32)
        self.env_actions = torch.empty(E, 4, **f32)              # the clipped actions env.step reads in place
        assert self.env_actions.data_ptr() % 16 == 0
        self.seed, self.counter = int(seed), 0

    @property
    def bytes(self) -> int:
        return super().bytes + sum(t.numel() * t.element_size() for t in (self.values, self.log_probs, self.advantages,
                                                                          self.returns, self.last_values, self.env_actions))

    def collect(self, fused, n_steps: Optional[int] = None):
        """Fill the buffer from position 0 with ``fused`` (a FusedPolicy of a LidarInertialActorCritic); nothing touches the
        host.  Then last_values = V(observation after the last step)."""
        if not hasattr(fused, "act"):
            raise TypeError("PPORollout.collect needs a FusedPolicy of a LidarInertialActorCritic")
        e = self.env
        self.pos = 0
        for _ in range(n_steps or self.n_steps):
            t = self.pos
            self._store_obs(t)
            fused.act(e.obs, self.counter, seed=self.seed, env_offset=e.env_offset, env_actions=self.env_actions,
                      raw_actions=self.actions[t], log_prob=self.log_probs[t], value=self.values[t])
            self.counter += 1
            self._step(t, self.env_actions)
        fused.values(e.obs, out=self.last_values)
        return self

    def compute_returns_and_advantage(self, gamma: float = 0.99, gae_lambda: float = 0.95):
        """SB3's RolloutBuffer.compute_returns_and_advantage over the collected steps, in one kernel (dc_gae)."""
        e, T = self.env, self.pos
        p = lambda t: C.c_void_p(t.data_ptr())      # noqa: E731
        with torch.cuda.device(e.device):
            _lib.check(_lib.lib().dc_gae(p(self.rewards), p(self.dones), p(self.values), p(self.last_values), T, e.n_envs,
                                         float(gamma), float(gae_lambda), p(self.advantages), p(self.returns),
                                         C.c_void_p(torch.cuda.current_stream(e.device).cuda_stream)), "dc_gae")
        return self

    def minibatch(self, flat_index: torch.Tensor) -> Dict[str, torch.Tensor]:
        """The parent's batch (``actions`` = the unclipped samples) + ``old_values``, ``old_log_prob``, ``advantages``,
        ``returns``."""
        b = super().minibatch(flat_index)
        idx = flat_index.to(device=self.env.device, dtype=torch.int64)
        n = self.n_steps * self.env.n_envs
        return {**b, "old_values": self.values.view(n)[idx], "old_log_prob": self.log_probs.view(n)[idx],
                "advantages": self.advantages.view(n)[idx], "returns": self.returns.view(n)[idx]}
