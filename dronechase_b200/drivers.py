"""Host side of the tasks that fly wingmen with policies of their own: ``Evaluation_Task.drive_lw``
(src/threatengage/environments/level4/components/tasks_management/tasks/evaluation_task.py:257-277) and
``Exp05_vFinal_Task.drive_lw_rl_agent`` (exp05_vFinal_task.py:252-260).

The reference serves the armed wingmen one after the other: ``observation = compute_lw_observation(pursuer)``,
``action = driver.predict(observation, deterministic=True)``, ``self.last_action = action``, ``pursuer.drive(action)`` --
``last_action`` is ONE variable of the task, so a wingman sees the action of whichever wingman was served before it (in
this step, or in the previous one), and ``init_globals`` zeroes it at a reset (:141).  ``TaskDrivers`` does that loop for the
whole batch on the device: per policy slot one batched policy call over all envs, the shared ``last_action`` advanced only in
the envs where that wingman was served.  A slot whose policy is a ``policy.FusedPolicy`` is served by ``FusedPolicy.serve``: one
kernel launch that reads the slot's rows of the wingman slabs in place, writes ``env.lw_actions[:, slot]`` and advances
``last_action`` in the same launch, with the same bits as the generic path.
"""
from __future__ import annotations

from typing import Callable, Dict, Optional, Sequence

import torch

Policy = Callable[[Dict[str, torch.Tensor]], torch.Tensor]      # obs dict of [B, ...] CUDA tensors -> [B, 4] float32 actions


def sb3_policy(model) -> Policy:
    """Wrap an object with SB3's ``predict(observation, deterministic=True)`` (numpy in / numpy out, batched over the
    leading axis) as a device policy -- one PCIe round trip per call; prefer dronechase_b200.policy for throughput."""
    def call(obs):
        import numpy as np
        a, _ = model.predict({k: v.detach().cpu().numpy() for k, v in obs.items()}, deterministic=True)
        return torch.as_tensor(np.asarray(a, dtype=np.float32), device=next(iter(obs.values())).device)
    return call


class TaskDrivers:
    def __init__(self, env, policies: Dict[int, Policy] | Sequence[Optional[Policy]]):
        """``policies``: wingman slot -> policy for every slot in ``env.cfg.policy_slots``."""
        self.env = env
        self.policies = dict(policies) if isinstance(policies, dict) else {j: p for j, p in enumerate(policies) if p is not None}
        missing = [j for j in env.cfg.policy_slots if j not in self.policies]
        if missing:
            raise ValueError(f"no policy for the policy-driven wingman slots {missing}")
        # the task's shared variable: ONE tensor, only ever updated in place (FusedPolicy.serve writes it from its kernel)
        self.last_action = torch.zeros(env.n_envs, 4, dtype=torch.float32, device=env.device)

    def reset(self, mask: Optional[torch.Tensor] = None):
        """Task.init_globals at Env.reset: last_action = zeros."""
        if mask is None:
            self.last_action.zero_()
        else:
            self.last_action[mask.to(self.last_action.device).bool()] = 0

    def serve(self) -> torch.Tensor:
        """on_step_start: observe, run every policy, fill ``env.lw_actions``.  Returns ``env.lw_actions``."""
        env = self.env
        lw = env.lw_observe()
        for j in env.cfg.policy_slots:                    # pursuers are served in slot order
            policy = self.policies[j]
            if hasattr(policy, "precision") and hasattr(policy, "refresh"):       # policy.FusedPolicy: one launch, in place
                policy.serve(lw, j, self.last_action, env.lw_actions)
                continue
            present = lw["present"][:, j]
            obs = {"lidar": lw["lidar"][:, j], "inertial_data": lw["inertial_data"][:, j], "last_action": self.last_action}
            a = policy(obs).to(torch.float32)
            env.lw_actions[:, j] = a
            self.last_action.copy_(torch.where(present[:, None], a, self.last_action))
        return env.lw_actions

    def step(self, actions: Optional[torch.Tensor] = None):
        """One env step: on_step_start (policies) + dc_step; with auto-reset the shared last_action of the envs that
        finished is zeroed like the reference's reset does."""
        self.serve()
        out = self.env.step(actions)
        if self.env._c.auto_reset:
            self.last_action.masked_fill_(self.env.done.bool()[:, None], 0.0)
        return out
