"""SB3 ``VecEnv`` adapter and single-env ``gymnasium.Env`` view over the batched simulator.

Boundary being replaced: ``ReinforcementLearningPipeline.create_vectorized_environment``
(src/core/rl_framework/utils/pipeline.py:32-61) returns ``VecMonitor(SubprocVecEnv([...]))`` of
``Exp02vFinalEnvironment``-style envs; ``DroneChaseVecEnv`` offers the same numpy-facing contract
(``reset() -> obs``, ``step_async/step_wait -> (obs, rewards, dones, infos)`` with SB3's auto-reset
and ``infos[i]["terminal_observation"]``) backed by ONE device-resident batch.  stable-baselines3 and
gymnasium are optional here: when importable the classes subclass them, otherwise they duck-type
the documented interface.
"""
from __future__ import annotations

from typing import Any, Dict, List, Optional, Sequence

import numpy as np
import torch

from .config import TaskConfig, preset
from .sim import BatchedThreatEngageEnv, INFO_KEYS

try:  # pragma: no cover - depends on the host image
    from stable_baselines3.common.vec_env import VecEnv as _VecEnvBase
except Exception:  # noqa: BLE001
    _VecEnvBase = object
try:  # pragma: no cover
    import gymnasium as _gym
    from gymnasium import spaces as _spaces
except Exception:  # noqa: BLE001
    _gym = None
    _spaces = None


class Box:
    """Minimal stand-in for gymnasium.spaces.Box (used only when gymnasium is absent)."""

    def __init__(self, low, high, shape=None, dtype=np.float32):
        self.dtype = np.dtype(dtype)
        self.shape = tuple(shape) if shape is not None else np.shape(low)
        self.low = np.broadcast_to(np.asarray(low, dtype=self.dtype), self.shape).copy()
        self.high = np.broadcast_to(np.asarray(high, dtype=self.dtype), self.shape).copy()

    def sample(self):
        return np.random.uniform(self.low, self.high).astype(self.dtype)

    def contains(self, x):
        x = np.asarray(x)
        return x.shape == self.shape and bool(np.all(x >= self.low) and np.all(x <= self.high))


class MultiBinary:
    """Minimal stand-in for gymnasium.spaces.MultiBinary."""

    def __init__(self, n):
        self.n, self.shape, self.dtype = n, (n,), np.dtype(np.int8)


class DictSpace:
    def __init__(self, spaces):
        self.spaces = dict(spaces)

    def __getitem__(self, k):
        return self.spaces[k]

    def keys(self):
        return self.spaces.keys()


def make_spaces(cfg: TaskConfig):
    """_action_space / _observation_space of exp02_vFinal_environment.py:197-204,236-284."""
    B = _spaces.Box if _spaces is not None else Box
    D = _spaces.Dict if _spaces is not None else DictSpace
    action = B(low=np.array([-1, -1, -1, 0], dtype=np.float32), high=np.array([1, 1, 1, 1], dtype=np.float32),
               shape=(4,), dtype=np.float32)
    if cfg.family == "level5":      # level5_c1_fusion_environment.py:59-104
        MB = _spaces.MultiBinary if _spaces is not None else MultiBinary
        lidar = {"stacked_spheres": B(0, 1, shape=(6, 3, 13, 26), dtype=np.float32), "validity_mask": MB(6)}
    else:
        lidar = {"lidar": B(0, 1, shape=(cfg.lidar_channels, 13, 26), dtype=np.float32)}
    obs = D({
        **lidar,
        "inertial_data": B(-np.ones(15, dtype=np.float32), np.ones(15, dtype=np.float32), shape=(15,), dtype=np.float32),
        "last_action": B(np.array([-1, -1, -1, 0], dtype=np.float32), np.array([1, 1, 1, 1], dtype=np.float32),
                         shape=(4,), dtype=np.float32),
    })
    return action, obs


class _TerminalInfo(dict):
    """Info dict of an env that finished: ``terminal_observation`` is materialised (its arrays copied) when first asked
    for.  SB3 reads it only to bootstrap time-limit truncations, which never happen here (truncated is always False,
    exp02_vFinal_environment.py:172), and VecMonitor only copies the dict and adds ``episode``: hundreds of envs finish per
    step at 65,536 envs and most of their terminal observations are never looked at.  Like the observation arrays of the
    step it belongs to, it must be read before the second next step recycles them."""
    _KEY = "terminal_observation"

    def __init__(self, base, thunk):
        super().__init__(base)
        self._thunk = thunk

    def _fill(self):
        if self._thunk is not None:
            thunk, self._thunk = self._thunk, None
            dict.__setitem__(self, self._KEY, thunk())

    def __getitem__(self, k):
        if k == self._KEY:
            self._fill()
        return dict.__getitem__(self, k)

    def get(self, k, default=None):
        if k == self._KEY:
            self._fill()
        return dict.get(self, k, default)

    def __contains__(self, k):
        return (k == self._KEY and self._thunk is not None) or dict.__contains__(self, k)

    def copy(self):
        c = _TerminalInfo(dict(dict.items(self)), self._thunk)
        return c

    def __len__(self):
        return dict.__len__(self) + (1 if self._thunk is not None else 0)

    def _all(self):
        self._fill()
        return self

    def keys(self):
        return dict.keys(self._all())

    def items(self):
        return dict.items(self._all())

    def values(self):
        return dict.values(self._all())

    def __iter__(self):
        return dict.__iter__(self._all())

    def __repr__(self):
        return dict.__repr__(self._all())

    def __eq__(self, other):
        return dict.__eq__(self._all(), other)

    __hash__ = None


class InfoList:
    """Sequence of per-env info dicts built on demand from the batched counters.

    SB3 (VecMonitor, on-policy rollouts) only indexes the infos of envs that finished, so materialising
    65,536 dicts per step would be pure overhead; ``list(infos)`` still gives ordinary dicts.  The terminal observations
    of the finished envs arrive as stacked rows (``terminal`` = (env indices, {key: [n_done, ...] array}, obs dict of the
    step, extra keys)) and become per-env dicts -- with their own copy of the sphere -- when an info is first read."""

    def __init__(self, info_np: np.ndarray, terminal=None):
        self._info, self._cache = info_np, {}
        self._rows_map = {}
        if isinstance(terminal, dict):                    # already per-env dicts
            self._cache = {int(k): v for k, v in terminal.items()}
            terminal = None
        self._terminal = terminal
        self._rows_built = terminal is None

    @property
    def _rows(self):
        """env index -> row of the stacked terminal observations; built when an info is first read (a step that nobody
        asks about does not pay ~0.1 ms for a thousand-entry dict)."""
        if not self._rows_built:
            self._rows_map = {int(e): j for j, e in enumerate(self._terminal[0])}
            self._rows_built = True
        return self._rows_map

    def __len__(self):
        return self._info.shape[0]

    def _terminal_obs(self, i):
        if i not in self._cache:
            _, rows, obs, extra = self._terminal            # rows: [n_done, ...] host arrays, one row per finished env
            j = self._rows[i]
            d = {k: obs[k][i].copy() for k in obs if k not in rows}
            d.update({k: v[j].copy() for k, v in rows.items()})
            d.update(extra)
            self._cache[i] = d
        return self._cache[i]

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(len(self)))]
        if i < 0:
            i += len(self)
        r = self._info[i]
        d = {"agent_kills": int(r[0]), "allies_kills": int(r[1]), "deads": int(r[2]), "current_wave": int(r[3]),
             "TimeLimit.truncated": False}
        if i in self._rows or i in self._cache:
            d["episode_steps"] = int(r[7])
            return _TerminalInfo(d, lambda i=i: self._terminal_obs(i))
        return d

    def __iter__(self):
        return (self[i] for i in range(len(self)))


def _huge_zeros(shape, dtype):
    """Zero-filled host tensor on an anonymous mapping advised MADV_HUGEPAGE (falls back to a plain tensor)."""
    import mmap
    n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
    try:
        n_map = (n + (1 << 21) - 1) & ~((1 << 21) - 1)
        mm = mmap.mmap(-1, n_map)
        if hasattr(mm, "madvise") and hasattr(mmap, "MADV_HUGEPAGE"):
            mm.madvise(mmap.MADV_HUGEPAGE)
        arr = np.frombuffer(mm, dtype=np.uint8, count=n)
        t = torch.from_numpy(arr).view(dtype).view(*shape)
        t._dc_mmap = mm                       # keeps the mapping alive with the tensor
        return t
    except (OSError, ValueError, AttributeError, RuntimeError):
        return torch.zeros(shape, dtype=dtype)


def _pin_to_rank_cores():
    """Several ranks on one box (torchrun sets LOCAL_RANK / LOCAL_WORLD_SIZE): give each its own contiguous slice of the
    cores the process may run on.  Threads created afterwards (the host scatter pool, torch's copy threads) inherit it."""
    import os
    if not hasattr(os, "sched_setaffinity"):
        return
    n, r = int(os.environ.get("LOCAL_WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    if n <= 1 or os.environ.get("DRONECHASE_B200_NO_PIN"):
        return
    cores = sorted(os.sched_getaffinity(0))
    per = len(cores) // n
    if per < 1:
        return
    try:
        os.sched_setaffinity(0, cores[r * per:(r + 1) * per])
    except OSError:
        pass


class DroneChaseVecEnv(_VecEnvBase):
    """``num_envs`` reference envs as one GPU batch behind the SB3 VecEnv interface."""

    def __init__(self, cfg: TaskConfig | str = "exp02_vFinal", n_envs: int = 8, seed: int = 0, device=0,
                 env_offset: int = 0, terminal_observation: bool = True, sparse_lidar: bool = True,
                 host_threads: Optional[int] = None, mapped_lidar: Optional[bool] = None, pin_cores: bool = True,
                 pairs_lidar: Optional[bool] = None, transfer_graphs: bool = True):
        """``sparse_lidar``: move the sphere observation over PCIe as its hit list (8 B per entity slot instead of 4 KB per
        env) and rebuild the dense (C,13,26) arrays in host memory (dc_host_scatter_sphere); the arrays handed out are
        bit-identical to a dense copy (level5: the stacked spheres travel as one hit list per env, dc_host_scatter_stack).
        ``pairs_lidar`` (the default of the level4/3/2 families when ``sparse_lidar``): the update as a LIST -- a kernel
        (dc_diff_hits) writes the (index, value) pairs that changed into a device buffer, the copy engines bring them to pinned
        memory and a few host threads store them into the dense arrays (dc_host_apply_pairs): 0.71 ms per 65,536-env step
        against 0.98 ms for the mapped mirror (profiles/r2ah_e2e_ab.txt).
        ``mapped_lidar``: the dense host arrays are page-locked and mapped into the device address space, and a kernel
        (dc_mirror_hits) writes the few words that changed straight into them over PCIe -- no copy, no host core busy, but
        posted 4-byte writes run at ~0.3 G/s (0.42 ms per 65,536 envs).
        ``transfer_graphs`` (with ``pairs_lidar``): everything step_wait enqueues -- the change-list kernel, a dozen device-to-host
        copies, the gather of the finished envs' terminal rows -- is captured once per landing zone into two CUDA graphs and
        replayed: the host side of a step is then two graph launches instead of ~20 torch dispatches.
        ``pin_cores``: with several ranks on a box (LOCAL_WORLD_SIZE > 1) restrict this process to its own slice of the
        host cores, so that the ranks' scatter / copy threads do not migrate over each other."""
        if isinstance(cfg, str):
            cfg = preset(cfg)
        self.cfg = cfg
        if getattr(cfg, "level5_multi_obs", 0):
            raise ValueError("the multi-observer / evaluation level5 envs return no per-env observation dict: use "
                             "BatchedThreatEngageEnv(...).multi_obs / dronechase_b200.io_data.collect_data_multiobs, or the "
                             "single-env facades Level5DumbMultiObs / Level52BTEvaluationEnvironment")
        if cfg.lidar == "raycast":
            # a ray-cast sphere has no per-slot hit list: it crosses PCIe dense (4 KB per env)
            if pairs_lidar or mapped_lidar:
                raise ValueError("lidar='raycast' moves the sphere dense: pairs_lidar / mapped_lidar need the per-slot hit "
                                 "list, which cannot describe a ray-cast sphere")
            sparse_lidar, pairs_lidar, mapped_lidar = False, False, False
        self.sparse = bool(sparse_lidar)
        self._lidar_key = "stacked_spheres" if cfg.family == "level5" else "lidar"
        # level4/3/2 families: "pairs" (default) | "mapped" | "scatter" (hit list + host scatter, also the level5 way);
        # DRONECHASE_B200_LIDAR_TRANSFER overrides the default when neither keyword is given
        if pairs_lidar is None and mapped_lidar is None:
            import os
            want = os.environ.get("DRONECHASE_B200_LIDAR_TRANSFER", "pairs").lower()
            pairs_lidar, mapped_lidar = want == "pairs", (True if want == "mapped" else (None if want == "pairs" else False))
        self.pairs = self.sparse and cfg.family != "level5" and bool(pairs_lidar) and not mapped_lidar
        self.mapped = self.sparse and cfg.family != "level5" and not self.pairs and (mapped_lidar is None or bool(mapped_lidar))
        if pin_cores:
            _pin_to_rank_cores()
        self.sim = BatchedThreatEngageEnv(cfg, n_envs=n_envs, seed=seed, device=device, env_offset=env_offset,
                                          auto_reset=True, with_terminal_obs=terminal_observation, with_hits=self.sparse)
        self.action_space, self.observation_space = make_spaces(cfg)
        if _VecEnvBase is not object:
            super().__init__(n_envs, self.observation_space, self.action_space)
        self.num_envs = n_envs
        self.render_mode = None
        E = n_envs
        pin = dict(pin_memory=True)
        self._h_actions = torch.zeros(E, 4, dtype=torch.float32, **pin)
        self._h_actions_np = self._h_actions.numpy()
        # two pinned landing zones: the arrays returned by step t stay valid while step t+1 is produced
        # (with the sparse transfer the dense sphere is never a DMA target: it lives in ordinary memory on huge pages,
        # the host scatter touches ~1e6 random lines of it per step and 4 KB pages made that a TLB-miss benchmark)
        # (the small outputs -- inertial vector, last action, reward, info, done -- mirror the simulator's `out_arena`: one
        # pinned allocation per landing zone, filled by ONE copy)
        from .sim import carve_outputs
        self._h = []
        for _ in range(2):
            arena, views = carve_outputs(E, None, pin=True)
            self._h.append({"obs": {k: (_huge_zeros(v.shape, v.dtype) if self.sparse and k == self._lidar_key
                                        else views[k] if k in views else torch.zeros(v.shape, dtype=v.dtype, **pin))
                                    for k, v in self.sim.obs.items()},
                            "reward": views["reward"], "done": views["done"], "info": views["info"], "arena": arena})
        self._flip = 0
        self._hits_ready = torch.cuda.Event()
        if self.sparse:
            import os
            # host threads of the scatter helper: the cores this process may use, shared with the other ranks of the box
            cpus = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
            ranks = 1 if pin_cores else max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
            # (the helper hands out small env chunks dynamically, so a descheduled core of a shared box costs one chunk)
            self._threads = int(host_threads or max(1, min(16, cpus // ranks)))
            for h in self._h:
                h["obs"][self._lidar_key].fill_(1.0)
        if self.mapped:
            # the two dense landing zones, mapped into the device address space + what each of them shows (device side)
            import ctypes as C
            from . import _lib
            self._dense_dev, self._registered = [], []
            try:
                for h in self._h:
                    t = h["obs"][self._lidar_key]
                    dp = C.c_void_p()
                    _lib.check(_lib.lib().dc_host_register(C.c_void_p(t.data_ptr()), t.numel() * 4, C.byref(dp)), "dc_host_register")
                    self._registered.append(t.data_ptr())
                    self._dense_dev.append(dp.value)
                self._shown = [torch.full(tuple(self.sim.lidar_hits.shape), -1, dtype=torch.int32, device=self.sim.device)
                               for _ in range(2)]
            except _lib.DroneChaseError:
                if mapped_lidar:                      # asked for explicitly: fail loudly
                    raise
                self._unregister()
                self.mapped = False
        if self.pairs:
            # what each landing zone shows (device side), the change list of a step on the device and in pinned memory:
            # [count, pad, (index, value) ...]; the first `_pairs_fast` pairs travel with the count in one copy
            D = self.sim.lidar_hits.shape[1]
            self._shown = [torch.full(tuple(self.sim.lidar_hits.shape), -1, dtype=torch.int32, device=self.sim.device)
                           for _ in range(2)]
            self._pairs_dev = torch.zeros(2 * (1 + 6 * E * D), dtype=torch.int32, device=self.sim.device)
            self._pairs_h = torch.zeros(2 * (1 + 6 * E * D), dtype=torch.int32, **pin)
            self._pairs_fast = min(6 * E * D, max(4096, 4 * E))
        if self.sparse and not self.mapped and not self.pairs:
            # hits the dense array of each landing zone currently shows + one incoming buffer (swapped, never copied)
            self._hits = [torch.full(tuple(self.sim.lidar_hits.shape), -1, dtype=torch.int32, **pin) for _ in range(3)]
        # terminal observations: only the rows of the envs that finished cross PCIe -- torch.nonzero_static gathers up to
        # `cap` of them on the device without a host sync (more than `cap` in one step: a second, full copy) -- into one of
        # two landing zones; the per-env dicts are built on the host when an info dict asks for them
        self._term_cap = min(E, max(1024, E // 8))
        self._h_term = ([{**{k: torch.zeros((self._term_cap,) + tuple(v.shape[1:]), dtype=torch.float32, **pin)
                             for k, v in self.sim.terminal_obs.items()},
                          "_idx": torch.zeros(self._term_cap, dtype=torch.int64, **pin)}
                         for _ in range(2)] if terminal_observation else None)
        self._np_views = [{"obs": {k: v.numpy() for k, v in h["obs"].items()}, "reward": h["reward"].numpy(),
                           "done": h["done"].numpy().view(np.bool_), "info": h["info"].numpy(),
                           "term": ({k: v.numpy() for k, v in self._h_term[f].items()} if self._h_term is not None else None)}
                          for f, h in enumerate(self._h)]
        self._dev_actions = torch.zeros(E, 4, dtype=torch.float32, device=self.sim.device)
        self.h2d_bytes_per_step = self._h_actions.numel() * 4
        obs_bytes = sum(v.numel() * v.element_size() for k, v in self._h[0]["obs"].items() if not (self.sparse and k == self._lidar_key))
        if self.sparse and not self.mapped and not self.pairs:
            obs_bytes += self._hits[0].numel() * 4
        if self.pairs:
            obs_bytes += 8 * (1 + self._pairs_fast)       # what every step copies; a longer list costs a second copy
        # mapped: the sphere crosses PCIe as the words that changed (a few per env, data dependent): not counted here
        self.d2h_bytes_per_step = obs_bytes + E * 4 + E + self._h[0]["info"].numel() * 4
        if terminal_observation:
            self.d2h_bytes_per_step += sum(v.numel() * v.element_size() for v in self._h_term[0].values())
        self._graphs = None
        self._use_graphs = bool(transfer_graphs) and self.pairs
        self._side = torch.cuda.Stream(device=self.sim.device) if self.mapped else None
        self._step_done = torch.cuda.Event()
        self._mirror_done = torch.cuda.Event()

    # -- VecEnv interface ---------------------------------------------------------------------
    def _unregister(self):
        from . import _lib
        import ctypes as C
        for ptr in getattr(self, "_registered", []):
            _lib.lib().dc_host_unregister(C.c_void_p(ptr))
        self._registered = []

    def _enqueue_obs(self, h):
        # the hit list goes first and gets its own event: the host scatter starts as soon as it has landed, while the
        # rest of the step's outputs are still crossing PCIe
        if self.mapped:
            # the mirror kernel's PCIe writes (0.5 ms at 65,536 envs) run on a side stream while the copy engines move the
            # rest of the step's outputs
            import ctypes as C
            from . import _lib
            f = self._flip
            main = torch.cuda.current_stream(self.sim.device)
            self._step_done.record(main)
            self._side.wait_event(self._step_done)
            with torch.cuda.device(self.sim.device):
                _lib.check(_lib.lib().dc_mirror_hits(C.c_void_p(self._shown[f].data_ptr()), C.c_void_p(self.sim.lidar_hits.data_ptr()),
                                                     self.num_envs, self.cfg.n_drones, self.cfg.n_lw, self.cfg.lidar_channels,
                                                     C.c_void_p(self._dense_dev[f]), C.c_void_p(self._side.cuda_stream)), "dc_mirror_hits")
            self._mirror_done.record(self._side)
        elif self.pairs:
            self._enqueue_pairs(self._flip)
            self._hits_ready.record(torch.cuda.current_stream(self.sim.device))
        elif self.sparse:
            self._hits[2].copy_(self.sim.lidar_hits, non_blocking=True)
            self._hits_ready.record(torch.cuda.current_stream(self.sim.device))
        for k, v in self.sim.obs.items():
            if not (self.sparse and k == self._lidar_key):
                h["obs"][k].copy_(v, non_blocking=True)

    def _enqueue_pairs(self, f):
        """The sphere update of landing zone f as a change list: dc_diff_hits + the copy of its head to pinned memory."""
        import ctypes as C
        from . import _lib
        main = torch.cuda.current_stream(self.sim.device)
        with torch.cuda.device(self.sim.device):
            _lib.check(_lib.lib().dc_diff_hits(C.c_void_p(self._shown[f].data_ptr()), C.c_void_p(self.sim.lidar_hits.data_ptr()),
                                               self.num_envs, self.cfg.n_drones, self.cfg.n_lw, self.cfg.lidar_channels,
                                               C.c_void_p(self._pairs_dev.data_ptr()), C.c_void_p(main.cuda_stream)), "dc_diff_hits")
        k = 2 * (1 + self._pairs_fast)
        self._pairs_h[:k].copy_(self._pairs_dev[:k], non_blocking=True)

    def _enqueue_rest(self, f):
        """Everything else a step hands out, into landing zone f: the other observation tensors, reward, done, info and the
        terminal rows of (up to _term_cap of) the envs that finished."""
        s, h = self.sim, self._h[f]
        h["arena"].copy_(s.out_arena, non_blocking=True)          # inertial vector, last action, reward, info, done
        for k, v in s.obs.items():
            if not (self.sparse and k == self._lidar_key) and k not in ("inertial_data", "last_action"):
                h["obs"][k].copy_(v, non_blocking=True)
        if self._h_term is not None:
            ht = self._h_term[f]
            didx = torch.nonzero_static(s.done, size=self._term_cap, fill_value=-1).view(-1)
            ht["_idx"].copy_(didx, non_blocking=True)
            sel = didx.clamp(min=0)
            for k, v in s.terminal_obs.items():
                ht[k].copy_(v.index_select(0, sel), non_blocking=True)

    def _capture_graphs(self):
        """Two graphs per landing zone (the change list first, so that the host can start storing it while the rest is still
        crossing PCIe).  Any failure leaves the eager path in charge."""
        self._use_graphs = False
        dev = self.sim.device
        try:
            torch.cuda.synchronize(dev)
            side = torch.cuda.Stream(device=dev)
            graphs = []
            for f in (0, 1):
                g_pairs, g_rest = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
                with torch.cuda.graph(g_pairs, stream=side):
                    self._enqueue_pairs(f)
                with torch.cuda.graph(g_rest, stream=side):
                    self._enqueue_rest(f)
                graphs.append((g_pairs, g_rest))
            torch.cuda.synchronize(dev)
            self._graphs = graphs
        except Exception:                                 # noqa: BLE001 -- capture is an optimisation, never a requirement
            self._graphs = None
            torch.cuda.synchronize(dev)

    def _wait_and_densify(self, h):
        if self.mapped:      # joined AFTER the copies were enqueued, so that they run under the mirror kernel
            torch.cuda.current_stream(self.sim.device).wait_event(self._mirror_done)
        if self.pairs:
            import ctypes as C
            from . import _lib
            self._hits_ready.synchronize()
            n = int(self._pairs_h[0])
            if n > self._pairs_fast:                      # a longer list than the first copy holds (e.g. right after a reset)
                k0, k1 = 2 * (1 + self._pairs_fast), 2 * (1 + n)
                self._pairs_h[k0:k1].copy_(self._pairs_dev[k0:k1], non_blocking=True)
                torch.cuda.current_stream(self.sim.device).synchronize()
            _lib.check(_lib.lib().dc_host_apply_pairs(C.c_void_p(h["obs"][self._lidar_key].data_ptr()),
                                                      C.c_void_p(self._pairs_h.data_ptr() + 8), n, self._threads), "dc_host_apply_pairs")
        elif self.sparse and not self.mapped:
            self._hits_ready.synchronize()
            self._densify(h)
        torch.cuda.current_stream(self.sim.device).synchronize()

    def _densify(self, h):
        """After the stream is synchronised: bring this landing zone's dense sphere from the hits it shows to the new ones."""
        if not self.sparse or self.mapped or self.pairs:
            return
        f = self._flip
        from . import _lib
        dense = h["obs"][self._lidar_key]
        if self.cfg.family == "level5":
            _lib.check(_lib.lib().dc_host_scatter_stack(dense.data_ptr(), self._hits[f].data_ptr(), self._hits[2].data_ptr(),
                                                        self.num_envs, self.cfg.n_drones, self._threads), "dc_host_scatter_stack")
        else:
            _lib.check(_lib.lib().dc_host_scatter_sphere(dense.data_ptr(), self._hits[f].data_ptr(), self._hits[2].data_ptr(),
                                                         self.num_envs, self.cfg.n_drones, self.cfg.n_lw, dense.shape[1],
                                                         self._threads), "dc_host_scatter_sphere")
        self._hits[f], self._hits[2] = self._hits[2], self._hits[f]

    def _fetch_obs(self) -> Dict[str, np.ndarray]:
        h = self._h[self._flip]
        self._enqueue_obs(h)
        self._wait_and_densify(h)
        return {k: v.numpy() for k, v in h["obs"].items()}

    def reset(self):
        self.sim.reset()
        return self._fetch_obs()

    def step_async(self, actions: np.ndarray) -> None:
        # plain memcpy into the pinned buffer: torch's copy_ wakes its intra-op thread pool for this 1 MB, which cost
        # 2 ms per step whenever the pool had gone to sleep behind a long host scatter (level5, profiles/l5_async_probe.py)
        np.copyto(self._h_actions_np, np.asarray(actions, dtype=np.float32).reshape(self.num_envs, 4))
        self._dev_actions.copy_(self._h_actions, non_blocking=True)
        self.sim.step(self._dev_actions)

    def step_wait(self):
        s = self.sim
        self._flip ^= 1
        h = self._h[self._flip]
        if self._use_graphs and self._graphs is None:
            self._capture_graphs()
        if self._graphs is not None:
            g_pairs, g_rest = self._graphs[self._flip]
            g_pairs.replay()
            self._hits_ready.record(torch.cuda.current_stream(s.device))
            g_rest.replay()
        else:
            self._enqueue_obs(h)
            h["reward"].copy_(s.reward, non_blocking=True)
            h["done"].copy_(s.done, non_blocking=True)
            h["info"].copy_(s.info, non_blocking=True)
            if self._h_term is not None:
                ht = self._h_term[self._flip]
                didx = torch.nonzero_static(s.done, size=self._term_cap, fill_value=-1).view(-1)
                ht["_idx"].copy_(didx, non_blocking=True)
                sel = didx.clamp(min=0)
                for k, v in s.terminal_obs.items():
                    ht[k].copy_(v.index_select(0, sel), non_blocking=True)
        self._wait_and_densify(h)
        hn = self._np_views[self._flip]                   # numpy views of the landing zone, made once
        dones, obs = hn["done"], dict(hn["obs"])
        terminal = None
        if self._h_term is not None and hn["term"]["_idx"][0] >= 0:      # the device gathered the finished envs' indices
            # level4: the sphere survives the reset untouched (fused_lidar.py:160-166), so obs["lidar"][i] IS the terminal
            # one.  level5: the ring is wiped by the reset and the terminal stack is not kept (terminated is never a
            # time-limit truncation here, so SB3 does not bootstrap from it): the reset stack stands in, and the dict says so.
            extra = {"stacked_spheres_is_reset_stack": True} if self.cfg.family == "level5" else {}
            tn = hn["term"]
            n_done = int(np.count_nonzero(tn["_idx"] >= 0))
            if n_done < self._term_cap:                   # ascending env order, like np.nonzero(dones)
                idx = tn["_idx"][:n_done]
                rows = {k: v[:n_done] for k, v in tn.items() if k != "_idx"}
            else:                                         # maybe more envs finished than the gather holds: fetch them all
                idx = np.nonzero(dones)[0]
                if len(idx) <= self._term_cap:
                    rows = {k: v[:len(idx)] for k, v in tn.items() if k != "_idx"}
                else:
                    sel = torch.from_numpy(idx).to(s.device)
                    rows = {k: v.index_select(0, sel).cpu().numpy() for k, v in s.terminal_obs.items()}
            terminal = (idx, rows, obs, extra)
        return obs, hn["reward"], dones, InfoList(hn["info"], terminal)

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def close(self) -> None:
        if getattr(self, "mapped", False):
            torch.cuda.synchronize(self.sim.device)
            self._unregister()
        self.sim.close()

    def seed(self, seed: Optional[int] = None):
        return [None] * self.num_envs

    def get_attr(self, attr_name: str, indices=None):
        n = self.num_envs if indices is None else len(self._indices(indices))
        return [getattr(self, attr_name, getattr(self.cfg, attr_name, None))] * n

    def set_attr(self, attr_name: str, value, indices=None) -> None:
        setattr(self, attr_name, value)

    def env_method(self, method_name: str, *args, indices=None, **kwargs):
        n = self.num_envs if indices is None else len(self._indices(indices))
        if method_name == "get_keymap":
            from .gym_env import default_keymap
            return [default_keymap()] * n
        raise AttributeError(f"env_method {method_name!r} is not available on the batched simulator")

    def env_is_wrapped(self, wrapper_class, indices=None):
        n = self.num_envs if indices is None else len(self._indices(indices))
        return [False] * n

    def _indices(self, indices) -> Sequence[int]:
        if indices is None:
            return range(self.num_envs)
        if isinstance(indices, int):
            return [indices]
        return list(indices)

    def get_images(self):
        return [None] * self.num_envs

    def render(self, mode: Optional[str] = None):
        return None
