"""Policy-driven wingmen served by the fused policy kernel, checked without a GPU: the C ABI of ``dc_policy_serve`` (v10) refuses
bad arguments before it touches a device, and ``drivers.TaskDrivers`` hands a ``FusedPolicy`` slot to ``serve`` while keeping
the task's shared ``last_action`` one tensor, updated in place, with the values of the generic per-slot path."""
import ctypes as C
from types import SimpleNamespace

import pytest
import torch

from dronechase_b200 import _lib
from dronechase_b200.drivers import TaskDrivers


def test_abi_version_10_exports_dc_policy_serve():
    L = _lib.lib()
    assert _lib.DC_ABI_VERSION == 10 and L.dc_abi_info(0) == 10
    assert "dc_policy_serve" in _lib.EXPORTS and hasattr(L, "dc_policy_serve")


def test_dc_policy_serve_argument_checks():
    L = _lib.lib()
    buf = (C.c_float * 64)()
    base = C.addressof(buf)                                # float-aligned host memory: never dereferenced by a refused call
    assert base % 4 == 0
    ok = C.c_void_p(base)

    def serve(policy=None, lidar=ok, inertial=ok, present=ok, n_lw=2, slot=0, n_envs=4, last=ok, acts=ok, precision=0):
        return L.dc_policy_serve(policy, lidar, inertial, present, n_lw, slot, n_envs, last, acts, precision, None)

    for kw in (dict(slot=2), dict(slot=-1), dict(n_lw=0, slot=0), dict(n_lw=3, slot=7)):
        assert serve(**kw) == -1 and b"slot must lie in [0, n_lw)" in L.dc_last_error(), kw
    for kw in (dict(lidar=None), dict(inertial=None), dict(present=None), dict(last=None), dict(acts=None), dict(n_envs=-1)):
        assert serve(**kw) == -1 and b"bad argument" in L.dc_last_error(), kw
    assert serve(precision=2) == -1 and b"precision" in L.dc_last_error()
    odd = C.c_void_p(base + 2)
    for kw in (dict(lidar=odd), dict(inertial=odd), dict(last=odd), dict(acts=odd)):
        assert serve(**kw) == -1 and b"4-byte aligned" in L.dc_last_error(), kw
    assert serve(present=odd) == -1 and b"null policy" in L.dc_last_error()     # bytes: any address
    assert serve() == -1 and b"null policy" in L.dc_last_error()


class _Env:
    """What TaskDrivers reads of a BatchedThreatEngageEnv, on the CPU: the wingman slabs of lw_observe, lw_actions, done."""

    def __init__(self, E=40, n_lw=3, slots=(0, 2), seed=0):
        self.n_envs, self.device = E, torch.device("cpu")
        self.cfg = SimpleNamespace(policy_slots=tuple(slots))
        self._c = SimpleNamespace(auto_reset=1)
        self.g = torch.Generator().manual_seed(seed)
        self.lw_actions = torch.zeros(E, n_lw, 4)
        self.done = torch.zeros(E, dtype=torch.uint8)
        self.n_lw = n_lw
        self.lw_obs = None

    def lw_observe(self):
        E, L, g = self.n_envs, self.n_lw, self.g
        self.lw_obs = {"lidar": torch.rand(E, L, 3, 13, 26, generator=g), "inertial_data": torch.rand(E, L, 15, generator=g) * 2 - 1,
                       "present": torch.rand(E, L, generator=g) < 0.6}
        return self.lw_obs

    def step(self, actions=None):
        self.done = (torch.rand(self.n_envs, generator=self.g) < 0.2).to(torch.uint8)
        return None, None, self.done, None


def _net(salt):
    def call(obs):
        return torch.tanh(obs["inertial_data"][:, :4] + 0.5 * obs["last_action"] + obs["lidar"][:, 0, 0, :4] * salt)
    return call


class _FusedLike:
    """Stands in for policy.FusedPolicy (precision, refresh, serve): serve does what dc_policy_serve does, in torch."""
    precision = "3xtf32"

    def __init__(self, salt):
        self.f, self.calls = _net(salt), []

    def refresh(self):
        return self

    def __call__(self, obs):
        raise AssertionError("TaskDrivers must hand a FusedPolicy slot to serve")

    def serve(self, lw, slot, last_action, lw_actions):
        self.calls.append((lw, slot, last_action, lw_actions))
        a = self.f({"lidar": lw["lidar"][:, slot], "inertial_data": lw["inertial_data"][:, slot], "last_action": last_action})
        lw_actions[:, slot] = a
        last_action[lw["present"][:, slot]] = a[lw["present"][:, slot]]
        return lw_actions


@pytest.mark.parametrize("fused_slots", [(), (0,), (2,), (0, 2)])
def test_task_drivers_serve_step_reset_keep_last_action_in_place(fused_slots):
    """Any mix of fused and generic slots gives what the generic chain gives (torch.where per slot, rebinding, zeroing of the
    finished envs); the shared last_action stays the tensor it was created as."""
    env = _Env()
    pols = {j: (_FusedLike(0.3 * j) if j in fused_slots else _net(0.3 * j)) for j in env.cfg.policy_slots}
    drv = TaskDrivers(env, pols)
    chain = drv.last_action
    ref = torch.zeros(env.n_envs, 4)
    for t in range(12):
        drv.step(None)
        lw = env.lw_obs
        want_acts = torch.zeros_like(env.lw_actions)
        for j in env.cfg.policy_slots:                    # the formulation TaskDrivers had before serve existed
            a = _net(0.3 * j)({"lidar": lw["lidar"][:, j], "inertial_data": lw["inertial_data"][:, j], "last_action": ref})
            want_acts[:, j] = a
            ref = torch.where(lw["present"][:, j][:, None], a, ref)
        ref = torch.where(env.done.bool()[:, None], torch.zeros_like(ref), ref)
        assert drv.last_action is chain
        assert torch.equal(drv.last_action, ref), f"step {t}"
        for j in env.cfg.policy_slots:
            assert torch.equal(env.lw_actions[:, j], want_acts[:, j]), f"step {t} slot {j}"
        if t == 5:
            drv.reset(torch.arange(env.n_envs) % 3 == 0)
            ref[torch.arange(env.n_envs) % 3 == 0] = 0
            assert drv.last_action is chain and torch.equal(drv.last_action, ref)
    assert bool(ref.any()) and bool((ref == 0).all(1).any())        # the chain carried actions and was zeroed somewhere
    for j in fused_slots:
        calls = pols[j].calls
        assert len(calls) == 12 and all(c[1] == j and c[2] is chain and c[3] is env.lw_actions for c in calls)
    drv.reset()
    assert drv.last_action is chain and not bool(chain.any())
