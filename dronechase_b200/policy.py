"""Device-resident policy inference (SURVEY.md section 8(f), rank 1, second half).

The reference drives the agent with an SB3 PPO whose feature extractor is ``LidarInertialActionExtractor``
(src/core/rl_framework/agents/policies/ppo_policies.py:234-342): Conv2d(C,32,k4,s4)-ReLU-Conv2d(32,64,k2,s2)-ReLU-Flatten
over the (C,13,26) sphere, two 3 x 128 MLPs over ``inertial_data`` and ``last_action``, Linear(448, features_dim)-ReLU; SB3 then
applies ``mlp_extractor.policy_net`` (``net_arch["pi"]``, Tanh by default -- ``create_policy_kwargs`` :150-156 passes
``net_arch=dict(pi=hiddens, vf=hiddens)``) and ``action_net``; ``predict(deterministic=True)`` returns the Gaussian mean
clipped to the action box.  Through SubprocVecEnv every step of that costs an observation round trip host -> device ->
host.  ``LidarInertialActionPolicy`` is the same network as a plain ``torch.nn.Module`` that reads the simulator's
observation tensors where they are (HBM) and writes the action tensor ``dc_step`` consumes: with ``DeviceRollout`` nothing
crosses PCIe during collection.  ``from_sb3_zip`` loads the weights of a model the reference trained (the ``policy.pth``
inside an SB3 ``.zip``) without needing stable-baselines3.
"""
from __future__ import annotations

import io
import zipfile
from typing import Dict, Optional, Sequence

import torch
from torch import nn


def _mlp3(n_in: int) -> nn.Sequential:
    return nn.Sequential(nn.Linear(n_in, 128), nn.ReLU(), nn.Linear(128, 128), nn.ReLU(), nn.Linear(128, 128), nn.ReLU())


class LidarInertialActionPolicy(nn.Module):
    def __init__(self, env=None, lidar_channels: int = 3, features_dim: int = 256, pi: Sequence[int] = (128, 256, 512),
                 activation: str = "tanh", seed: Optional[int] = 0, device=None):
        super().__init__()
        if env is not None:
            lidar_channels, device = env.cfg.lidar_channels, env.device
        if seed is not None:
            torch.manual_seed(int(seed))
        self.lidar_feature_extractor = nn.Sequential(nn.Conv2d(lidar_channels, 32, kernel_size=4, stride=4), nn.ReLU(),
                                                     nn.Conv2d(32, 64, kernel_size=2, stride=2), nn.ReLU(), nn.Flatten())
        self.inertial_feature_extractor = _mlp3(15)
        self.action_feature_extractor = _mlp3(4)
        n_lidar = 64 * ((13 // 4) // 2) * ((26 // 4) // 2)                 # (32,3,6) -> (64,1,3) = 192
        self.final_layer = nn.Sequential(nn.Linear(n_lidar + 128 + 128, features_dim), nn.ReLU())
        act = {"tanh": nn.Tanh, "relu": nn.ReLU}[activation]
        self.activation = activation
        layers, n = [], features_dim
        for h in pi:
            layers += [nn.Linear(n, int(h)), act()]
            n = int(h)
        self.policy_net = nn.Sequential(*layers)
        self.action_net = nn.Linear(n, 4)
        self.register_buffer("low", torch.tensor([-1.0, -1.0, -1.0, 0.0]))
        self.register_buffer("high", torch.tensor([1.0, 1.0, 1.0, 1.0]))
        self.pi, self.features_dim = tuple(int(h) for h in pi), int(features_dim)
        if device is not None:
            self.to(device)
        self.eval()

    def features(self, obs: Dict[str, torch.Tensor]) -> torch.Tensor:
        f = torch.cat((self.lidar_feature_extractor(obs["lidar"]), self.inertial_feature_extractor(obs["inertial_data"].flatten(1)),
                       self.action_feature_extractor(obs["last_action"])), dim=1)
        return self.final_layer(f)

    @torch.no_grad()
    def forward(self, obs: Dict[str, torch.Tensor]) -> torch.Tensor:
        """``model.predict(obs, deterministic=True)``: the mean action, clipped to Box([-1,-1,-1,0],[1,1,1,1])."""
        a = self.action_net(self.policy_net(self.features(obs)))
        return torch.maximum(torch.minimum(a, self.high), self.low).contiguous()

    def fused(self, precision: str = "3xtf32") -> "FusedPolicy":
        """The same network as ONE hand-written kernel (csrc/policy_kernel.cu, dc_policy_forward): see FusedPolicy."""
        return FusedPolicy(self, precision)

    def weight_arrays(self) -> Dict[str, object]:
        """The tensors dc_policy_weights names (torch layout, convolutions flattened to [out][in*kh*kw])."""
        lf, fi, fa = self.lidar_feature_extractor, self.inertial_feature_extractor, self.action_feature_extractor
        lin = [m for m in self.policy_net if isinstance(m, nn.Linear)]
        return {"conv1_w": lf[0].weight.flatten(1), "conv1_b": lf[0].bias, "conv2_w": lf[2].weight.flatten(1), "conv2_b": lf[2].bias,
                "inertial_w": [fi[j].weight for j in (0, 2, 4)], "inertial_b": [fi[j].bias for j in (0, 2, 4)],
                "action_w": [fa[j].weight for j in (0, 2, 4)], "action_b": [fa[j].bias for j in (0, 2, 4)],
                "final_w": self.final_layer[0].weight, "final_b": self.final_layer[0].bias,
                "pi_w": [m.weight for m in lin], "pi_b": [m.bias for m in lin],
                "head_w": self.action_net.weight, "head_b": self.action_net.bias}

    def describe(self) -> str:
        n = sum(p.numel() for p in self.parameters())
        return (f"LidarInertialActionExtractor (ppo_policies.py:234-342) + pi {list(self.pi)} + action_net, {n} parameters, float32, "
                "deterministic mean action")

    # ------------------------------------------------------------------ weights of a reference-trained SB3 model
    # (SB3 key prefix, own prefix) of everything but the features extractor
    _SB3_KEYS = (("mlp_extractor.policy_net.", "policy_net."), ("action_net.", "action_net."))

    def load_sb3_state_dict(self, sd: Dict[str, torch.Tensor]) -> "LidarInertialActionPolicy":
        """``sd`` = ``model.policy.state_dict()`` of an SB3 PPO (keys ``features_extractor.*`` or ``pi_features_extractor.*``,
        ``mlp_extractor.policy_net.*``, ``action_net.*``); value-function and log_std entries are ignored."""
        fx = "pi_features_extractor." if any(k.startswith("pi_features_extractor.") for k in sd) else "features_extractor."
        mine = {}
        for k, v in sd.items():
            if k.startswith(fx):
                mine[k[len(fx):]] = v
            for theirs, ours in self._SB3_KEYS:
                if k.startswith(theirs):
                    mine[ours + k[len(theirs):]] = v
        want = {k for k in self.state_dict() if k not in ("low", "high")}
        missing = want - set(mine)
        if missing:
            raise KeyError(f"SB3 state dict lacks {sorted(missing)[:4]} ...: not a LidarInertialActionExtractor PPO with pi={list(self.pi)}")
        self.load_state_dict({**{k: mine[k] for k in want}, "low": self.low, "high": self.high})
        return self

    @staticmethod
    def _sb3_widths(sd: Dict[str, torch.Tensor], net: str):
        out, i = [], 0
        while f"mlp_extractor.{net}.{i}.weight" in sd:
            out.append(sd[f"mlp_extractor.{net}.{i}.weight"].shape[0])
            i += 2
        return out

    @classmethod
    def _sb3_sizes(cls, sd: Dict[str, torch.Tensor]) -> Dict[str, object]:
        return {"pi": cls._sb3_widths(sd, "policy_net")}

    @classmethod
    def from_sb3_zip(cls, path: str, env=None, **kw) -> "LidarInertialActionPolicy":
        """Build from an SB3 ``model.save`` archive: reads ``policy.pth``, infers pi sizes and features_dim from the shapes."""
        with zipfile.ZipFile(path) as z:
            sd = torch.load(io.BytesIO(z.read("policy.pth")), map_location="cpu", weights_only=True)
        fx = "pi_features_extractor." if any(k.startswith("pi_features_extractor.") for k in sd) else "features_extractor."
        kw.setdefault("features_dim", sd[fx + "final_layer.0.weight"].shape[0])
        kw.setdefault("lidar_channels", sd[fx + "lidar_feature_extractor.0.weight"].shape[1])
        return cls(env=env, seed=None, **cls._sb3_sizes(sd), **kw).load_sb3_state_dict(sd)


class LidarInertialActorCritic(LidarInertialActionPolicy):
    """The whole SB3 ``ActorCriticPolicy`` of the reference's PPO (shared features extractor, ``net_arch = dict(pi=h, vf=h)``,
    ``DiagGaussianDistribution`` with ``log_std_init = 0``): the actor of ``LidarInertialActionPolicy`` plus ``vf_net``
    (= ``mlp_extractor.value_net``: hidden layers over the features, the activation of pi), ``value_net`` and ``log_std``.
    The value-branch parameters are created after the actor's, so a seeded actor is initialised as in the parent class.
    ``forward`` stays the clipped mean action; ``forward_train``, ``evaluate_actions`` and ``predict_values`` are
    differentiable, for the PPO update.  ``fused()`` gives the one-kernel rollout policy (``FusedPolicy.act`` / ``values``)."""

    _SB3_KEYS = LidarInertialActionPolicy._SB3_KEYS + (("mlp_extractor.value_net.", "vf_net."), ("value_net.", "value_net."),
                                                       ("log_std", "log_std"))

    def __init__(self, env=None, lidar_channels: int = 3, features_dim: int = 256, pi: Sequence[int] = (128, 256, 512),
                 vf: Optional[Sequence[int]] = None, activation: str = "tanh", seed: Optional[int] = 0, device=None):
        super().__init__(env, lidar_channels, features_dim, pi, activation, seed, device)
        device = env.device if env is not None else device
        act = {"tanh": nn.Tanh, "relu": nn.ReLU}[activation]
        vf = tuple(int(h) for h in (pi if vf is None else vf))
        layers, n = [], int(features_dim)
        for h in vf:
            layers += [nn.Linear(n, h), act()]
            n = h
        self.vf_net = nn.Sequential(*layers)
        self.value_net = nn.Linear(n, 1)
        self.log_std = nn.Parameter(torch.zeros(4))
        self.vf = vf
        if device is not None:
            self.to(device)
        self.eval()

    def forward_train(self, obs: Dict[str, torch.Tensor]):
        """(mean action, unclipped [N, 4]; value [N, 1]) from one evaluation of the features."""
        f = self.features(obs)
        return self.action_net(self.policy_net(f)), self.value_net(self.vf_net(f))

    def predict_values(self, obs: Dict[str, torch.Tensor]) -> torch.Tensor:
        """SB3 ``predict_values``: [N, 1]."""
        return self.value_net(self.vf_net(self.features(obs)))

    def evaluate_actions(self, obs: Dict[str, torch.Tensor], actions: torch.Tensor):
        """SB3 ``evaluate_actions``: (value [N, 1], log_prob [N], entropy [N]) of the UNCLIPPED ``actions`` under the diagonal
        Gaussian N(mean, exp(log_std)^2)."""
        mean, value = self.forward_train(obs)
        dist = torch.distributions.Normal(mean, torch.ones_like(mean) * self.log_std.exp())
        return value, dist.log_prob(actions).sum(dim=-1), dist.entropy().sum(dim=-1)

    def describe(self) -> str:
        n = sum(p.numel() for p in self.parameters())
        return (f"LidarInertialActionExtractor (ppo_policies.py:234-342) + pi {list(self.pi)} + action_net, vf {list(self.vf)} + "
                f"value_net, log_std; {n} parameters, float32, diagonal Gaussian actor-critic")

    def load_sb3_state_dict(self, sd: Dict[str, torch.Tensor]) -> "LidarInertialActorCritic":
        """As the parent's, and ``mlp_extractor.value_net.*``, ``value_net.*`` and ``log_std`` too.  The value branch must read the
        actor's features: an archive trained with ``share_features_extractor=False`` (its ``vf_features_extractor.*`` differ from
        the actor's extractor) raises ``ValueError``."""
        fx = "pi_features_extractor." if any(k.startswith("pi_features_extractor.") for k in sd) else "features_extractor."
        for k, v in sd.items():
            if k.startswith("vf_features_extractor."):
                mine = sd.get(fx + k[len("vf_features_extractor."):])
                if mine is None or mine.shape != v.shape or not torch.equal(mine, v):
                    raise ValueError("this SB3 policy has a separate vf_features_extractor (share_features_extractor=False): "
                                     "LidarInertialActorCritic evaluates the value branch on the actor's features")
        return super().load_sb3_state_dict(sd)

    @classmethod
    def _sb3_sizes(cls, sd: Dict[str, torch.Tensor]) -> Dict[str, object]:
        return {"pi": cls._sb3_widths(sd, "policy_net"), "vf": cls._sb3_widths(sd, "value_net")}


class FusedPolicy:
    """``LidarInertialActionPolicy`` evaluated by ONE kernel launch (``dc_policy_forward``, csrc/policy_kernel.cu): the twelve
    layers from the sphere to the clipped mean action run over 64 envs per block with every activation in shared memory and
    the products on the tensor cores.  ``precision="3xtf32"`` (default): every product as three TF32 MMAs, float32-grade --
    within 2e-5 of the torch float32 module; ``"tf32"``: plain TF32 operands, within 5e-3, three times fewer MMAs.
    The weights are re-laid out once, here; call ``refresh()`` after the module's parameters changed (PPO update).
    Shapes the kernel holds: features_dim and the hidden widths of ``pi`` multiples of 64 up to 256, the last one up to 1024
    (the defaults and ``net_arch`` of the reference's apps); anything else raises, use the module itself.  There is no
    fallback: without the CUDA library or a device this class raises.

    Built from a ``LidarInertialActorCritic`` (``dc_policy_create_ac``), it also runs the actor-critic kernel
    (``dc_policy_act``): ``act`` samples actions for PPO rollout collection, ``values`` gives V(s).  Precision matters more
    there: the log-probability error is about ``|eps| * (mean error) / sigma``.  With ``"tf32"`` (5e-3 on the mean) that is
    about 1e-2 in log-probability, a 1 % bias in PPO's first-epoch probability ratio; the default ``"3xtf32"`` keeps it near
    1e-4.

    ``serve`` runs the same network for one policy-driven wingman slot of a level4 task (``drivers.TaskDrivers``): it reads
    the wingman slabs of ``env.lw_observe()`` in place and advances the task's shared ``last_action`` in the same launch."""

    PRECISIONS = {"3xtf32": 0, "tf32": 1}

    def __init__(self, module: LidarInertialActionPolicy, precision: str = "3xtf32"):
        import ctypes as C
        from . import _lib
        self._C, self._lib = C, _lib
        self.module, self.precision = module, precision
        self._prec = self.PRECISIONS[precision]
        self._handle = None
        self.refresh()

    def refresh(self) -> "FusedPolicy":
        C, _lib, m = self._C, self._lib, self.module
        dev = next(m.parameters()).device
        if dev.type != "cuda":
            raise _lib.DroneChaseError("FusedPolicy needs the module on a CUDA device: there is no CPU fallback")
        wa = m.weight_arrays()
        keep = []

        def ptr(t):
            t = t.detach().to(torch.float32).contiguous()
            keep.append(t)
            return C.cast(C.c_void_p(t.data_ptr()), C.POINTER(C.c_float))
        w = _lib.dc_policy_weights()
        w.lidar_channels = m.lidar_feature_extractor[0].in_channels
        w.features_dim, w.n_pi = m.features_dim, len(m.pi)
        if len(m.pi) > 8:
            raise ValueError("FusedPolicy: at most 8 hidden layers in pi")
        for i, h in enumerate(m.pi):
            w.pi[i] = h
        w.activation = {"relu": 1, "tanh": 2}[m.activation]
        w.conv1_w, w.conv1_b, w.conv2_w, w.conv2_b = ptr(wa["conv1_w"]), ptr(wa["conv1_b"]), ptr(wa["conv2_w"]), ptr(wa["conv2_b"])
        for i in range(3):
            w.inertial_w[i], w.inertial_b[i] = ptr(wa["inertial_w"][i]), ptr(wa["inertial_b"][i])
            w.action_w[i], w.action_b[i] = ptr(wa["action_w"][i]), ptr(wa["action_b"][i])
        w.final_w, w.final_b = ptr(wa["final_w"]), ptr(wa["final_b"])
        for i in range(len(m.pi)):
            w.pi_w[i], w.pi_b[i] = ptr(wa["pi_w"][i]), ptr(wa["pi_b"][i])
        w.head_w, w.head_b = ptr(wa["head_w"]), ptr(wa["head_b"])
        for k in range(4):
            w.low[k], w.high[k] = float(m.low[k]), float(m.high[k])
        h = C.c_void_p()
        if isinstance(m, LidarInertialActorCritic):
            if len(m.vf) > 8:
                raise ValueError("FusedPolicy: at most 8 hidden layers in vf")
            v = _lib.dc_value_weights()
            v.n_vf = len(m.vf)
            vl = [x for x in m.vf_net if isinstance(x, nn.Linear)]
            for i, h_ in enumerate(m.vf):
                v.vf[i], v.vf_w[i], v.vf_b[i] = h_, ptr(vl[i].weight), ptr(vl[i].bias)
            v.value_w, v.value_b, v.log_std = ptr(m.value_net.weight), ptr(m.value_net.bias), ptr(m.log_std)
            torch.cuda.synchronize(dev)
            _lib.check(_lib.lib().dc_policy_create_ac(C.byref(w), C.byref(v), dev.index or 0, C.byref(h)), "dc_policy_create_ac")
        else:
            torch.cuda.synchronize(dev)
            _lib.check(_lib.lib().dc_policy_create(C.byref(w), dev.index or 0, C.byref(h)), "dc_policy_create")
        self.close()
        self._handle, self.device = h, dev
        return self

    def _is_f32(self, *ts: torch.Tensor) -> bool:
        """Every tensor is contiguous float32 on the policy's device: what the kernels read and write."""
        return all(t.dtype == torch.float32 and t.is_contiguous() and t.device == self.device for t in ts)

    def _call(self, fn: str, *args):
        """``fn(handle, *args, precision, stream)`` of the C library on the current stream of the policy's device; tensors in
        ``args`` are passed as their data pointers."""
        C = self._C
        args = [C.c_void_p(a.data_ptr()) if isinstance(a, torch.Tensor) else a for a in args]
        with torch.cuda.device(self.device):
            self._lib.check(getattr(self._lib.lib(), fn)(self._handle, *args, self._prec,
                                                          C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)), fn)

    def _check_obs(self, obs: Dict[str, torch.Tensor]):
        lidar, inertial, last = obs["lidar"], obs["inertial_data"], obs["last_action"]
        E = lidar.shape[0]
        if not self._is_f32(lidar, inertial, last):
            raise ValueError("FusedPolicy: observations must be contiguous float32 tensors on the policy's device")
        if tuple(lidar.shape[1:]) != (self.module.lidar_feature_extractor[0].in_channels, 13, 26) or inertial.numel() != E * 15 \
                or last.numel() != E * 4:
            raise ValueError("FusedPolicy: observation shapes must be lidar [E,C,13,26], inertial_data [E,15], last_action [E,4]")
        return lidar, inertial, last, E

    def __call__(self, obs: Dict[str, torch.Tensor], out: Optional[torch.Tensor] = None) -> torch.Tensor:
        lidar, inertial, last, E = self._check_obs(obs)
        if out is None:
            out = torch.empty(E, 4, dtype=torch.float32, device=self.device)
        self._call("dc_policy_forward", lidar, inertial, last, E, out)
        return out

    def serve(self, lw: Dict[str, torch.Tensor], slot: int, last_action: torch.Tensor, lw_actions: torch.Tensor) -> torch.Tensor:
        """Serve policy-driven wingman ``slot`` of a level4 task in one launch (``dc_policy_serve``).  ``lw`` is the dict
        ``env.lw_observe()`` returns (``lidar`` [E,n_lw,3,13,26], ``inertial_data`` [E,n_lw,15], ``present`` [E,n_lw]); the
        kernel reads the slot's rows in place.  ``lw_actions[:, slot]`` ([E,n_lw,4]) receives the clipped mean action of every
        env, and ``last_action`` ([E,4], the task's shared chain, which is also the policy's input) is overwritten with it
        where ``present[:, slot]``.  Bit for bit ``self`` on contiguous copies of the slot followed by ``torch.where``.
        Needs a 3-channel policy.  Returns ``lw_actions``."""
        lidar, inertial, present = lw["lidar"], lw["inertial_data"], lw["present"]
        if not self._is_f32(lidar, inertial, last_action, lw_actions):
            raise ValueError("FusedPolicy.serve: the wingman slabs, last_action and lw_actions must be contiguous float32 "
                             "tensors on the policy's device")
        if present.dtype not in (torch.bool, torch.uint8) or not present.is_contiguous() or present.device != self.device:
            raise ValueError("FusedPolicy.serve: present must be a contiguous bool or uint8 tensor on the policy's device")
        E, n_lw = lidar.shape[:2] if lidar.dim() == 5 else (-1, -1)
        if (tuple(lidar.shape) != (E, n_lw, 3, 13, 26) or tuple(inertial.shape) != (E, n_lw, 15) or tuple(present.shape) != (E, n_lw)
                or tuple(last_action.shape) != (E, 4) or tuple(lw_actions.shape) != (E, n_lw, 4)):
            raise ValueError("FusedPolicy.serve: shapes must be lidar [E,n_lw,3,13,26], inertial_data [E,n_lw,15], present [E,n_lw], "
                             "last_action [E,4], lw_actions [E,n_lw,4]")
        self._call("dc_policy_serve", lidar, inertial, present, n_lw, int(slot), E, last_action, lw_actions)
        return lw_actions

    def _run_act(self, obs, counter: int, seed: int, env_offset: int, sample: int, env_actions, raw_actions, log_prob, value):
        if not isinstance(self.module, LidarInertialActorCritic):
            raise self._lib.DroneChaseError("FusedPolicy.act / values need a LidarInertialActorCritic module (value branch, log_std)")
        lidar, inertial, last, E = self._check_obs(obs)

        def buf(t, shape):
            if t is None:
                return torch.empty(shape, dtype=torch.float32, device=self.device)
            if not self._is_f32(t) or tuple(t.shape) != shape:
                raise ValueError(f"FusedPolicy: outputs must be contiguous float32 tensors of shape {shape} on the policy's device")
            return t
        env_actions, value = buf(env_actions, (E, 4)), buf(value, (E,))
        if sample:
            raw_actions, log_prob = buf(raw_actions, (E, 4)), buf(log_prob, (E,))
        self._call("dc_policy_act", lidar, inertial, last, E, int(seed) & 0xFFFFFFFFFFFFFFFF, int(env_offset), int(counter) & 0xFFFFFFFF,
                   sample, env_actions, raw_actions if sample else None, log_prob if sample else None, value)
        return env_actions, raw_actions, log_prob, value

    def act(self, obs: Dict[str, torch.Tensor], counter: int, *, seed: int = 0, env_offset: int = 0,
            env_actions: Optional[torch.Tensor] = None, raw_actions: Optional[torch.Tensor] = None,
            log_prob: Optional[torch.Tensor] = None, value: Optional[torch.Tensor] = None, sample: bool = True):
        """One PPO collection step in one launch: (env_actions [E,4] clipped to the action box, raw_actions [E,4] the unclipped
        Gaussian sample that goes into the rollout buffer, log_prob [E], value [E]).  The noise of row e is a pure function of
        (seed, counter, env_offset + e): Philox4x32-10 stream 5 of the simulator's counter-based generator.  Outputs given as
        arguments are written in place.  ``sample=False``: env_actions = the clipped mean action, bit for bit what ``__call__``
        returns, and raw_actions / log_prob are None."""
        return self._run_act(obs, counter, seed, env_offset, int(bool(sample)), env_actions, raw_actions, log_prob, value)

    def values(self, obs: Dict[str, torch.Tensor], out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """V(s) [E] (the actor-critic kernel without sampling: ``predict_values`` for the bootstrap of the last step)."""
        return self._run_act(obs, 0, 0, 0, 0, None, None, None, out)[3]

    def describe(self) -> str:
        return self.module.describe().replace("float32", "one fused kernel, " + ("3 x TF32 (float32-grade)" if self._prec == 0 else "TF32"))

    def close(self):
        if getattr(self, "_handle", None) is not None:
            self._lib.lib().dc_policy_destroy(self._handle)
            self._handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:                                 # noqa: BLE001 -- interpreter shutdown
            pass
