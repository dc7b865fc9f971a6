"""Host-side mirror of the reference's environment interface (environment/boat_env.py).

``BatchedBoatEnv``  N independent env instances advanced per kernel launch; tensors stay
                    on the GPU (torch is used for device memory and streams only).
``BoatEnv``         the reference's single-env object, drop-in for main.py / Recorder /
                    BaseAgent: ``BoatEnv(config, experiment)``, ``reset()``,
                    ``step(action) -> (state, reward, done, info)``, ``return_all_data()``,
                    ``action_space``, ``observation_space``, ``info``, ``boat``, ``action``.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib
from .config import load_config, params_from_config

TERM_NAMES = ("", "reached_goal", "out_of_bounds", "out_of_fuel", "timeout", "rudder_broken")
AUTO_RESET = 1
STATE_FORMAT = 2   # layout of the opaque state blob: 2 = fp32 mode carries rudder / s_x / s_y in fixed point (common.cuh)
FIELDS = {"v_x": 0, "v_y": 1, "v_r": 2, "rudder_angle": 3, "s_x": 4, "s_y": 5, "s_r": 6,
          "episode_reward": 7, "index": 8, "episode": 9}
COUNTER_NAMES = ("reached_goal", "out_of_bounds", "out_of_fuel", "timeout", "rudder_broken",
                 "episodes", "return_sum", "return_sumsq")

class _FallbackBox:
    """Minimal stand-in for gym.spaces.Box with the attributes BaseAgent reads (base_agent.py:7-19)."""

    def __init__(self, low, high, shape=None, dtype=np.float32):
        low = np.asarray(low, dtype=dtype)
        high = np.asarray(high, dtype=dtype)
        if low.ndim == 0:  # scalar bounds and no shape: gym 0.26 infers (1,)
            low, high = low.reshape(1), high.reshape(1)
        self.low, self.high, self.shape, self.dtype = low, high, low.shape, np.dtype(dtype)

    def sample(self):
        return np.random.uniform(self.low, self.high).astype(self.dtype)


def _box_class():
    """The reference's spaces come from gym 0.26 (boat_env.py:2) and BaseAgent tests ``isinstance(action_space,
    gym.spaces.Box)`` (base_agent.py:9): whenever a ``gym`` is importable when an env is built, its Box is used, so
    that check holds for the drop-in; gym itself is not a dependency of this package."""
    try:
        from gym.spaces import Box as GymBox  # type: ignore
        return GymBox
    except Exception:
        return _FallbackBox


Box = _box_class()


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("sac_agent_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch


class BatchedBoatEnv:
    """N envs, one CUDA thread each.  Observations/rewards/dones are torch CUDA tensors.

    Episode randomness comes from Philox keyed by (seed, env_id_offset + i, episode), so
    a shard of a larger population reproduces exactly the same envs.
    """

    def __init__(self, config=None, n_envs=1, seed=0, precision="fp32", device=None,
                 env_id_offset=0, auto_reset=True):
        torch = _torch()
        self.config = config if config is not None else load_config()
        self.params = params_from_config(self.config)
        self.n_envs = int(n_envs)
        self.precision = {"fp32": 32, "fp64": 64, 32: 32, 64: 64}[precision]
        self.dtype = torch.float32 if self.precision == 32 else torch.float64
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
        self.seed, self.env_id_offset = int(seed), int(env_id_offset)
        self.auto_reset = bool(auto_reset)
        self._L = _lib.lib()
        h = C.c_void_p()
        _lib.check(self._L.boatenv_create(C.byref(self.params), self.n_envs, self.seed, self.env_id_offset,
                                          self.precision, self.device.index, C.byref(h)), "boatenv_create")
        self._h = h
        n = self.n_envs
        self.obs = torch.empty((n, 11), dtype=self.dtype, device=self.device)
        self.reward = torch.empty(n, dtype=self.dtype, device=self.device)
        self.done = torch.empty(n, dtype=torch.uint8, device=self.device)
        self.term = torch.empty(n, dtype=torch.uint8, device=self.device)
        self.final_obs = torch.zeros((n, 11), dtype=self.dtype, device=self.device)
        box = _box_class()   # resolved now, not at import time: a gym imported in between is honoured
        self.observation_space = box(low=np.array([0] * 10 + [1], dtype=np.float32),
                                     high=np.array([1] * 10 + [0], dtype=np.float32), dtype=np.float32)
        self.action_space = box(low=-1, high=1, dtype=np.float32)  # boat_env.py:37-41

    # -- life cycle ---------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._L.boatenv_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    def _actions(self, actions):
        torch = _torch()
        a = torch.as_tensor(actions, device=self.device)
        if a.dtype != self.dtype:
            a = a.to(self.dtype)
        a = a.reshape(-1, self.n_envs) if a.numel() != self.n_envs else a.reshape(self.n_envs)
        return a.contiguous()

    # -- gym API --------------------------------------------------------------------
    def reset(self, mask=None):
        """BoatEnv.reset (boat_env.py:120-126) for all (or the masked) envs."""
        torch = _torch()
        m = None
        if mask is not None:  # masked: only those envs (and their rows of self.obs) are rewritten
            m = torch.as_tensor(mask, device=self.device).to(torch.uint8).contiguous()
            if m.numel() != self.n_envs:
                raise ValueError("mask must have one entry per env")
        _lib.check(self._L.boatenv_reset(self._h, None if m is None else m.data_ptr(), self.obs.data_ptr(),
                                         self._stream()), "boatenv_reset")
        return self.obs

    def step(self, actions, done_from_term=False):
        """BoatEnv.step (boat_env.py:67-115) for every env.  Returns (obs, reward, done, info);
        info holds the per-env termination codes and, under auto-reset, the terminal
        observations of the envs that finished.  The returned tensors are the env's own output
        buffers (no allocation per step): the next step overwrites them, clone what must survive.
        ``done_from_term``: the kernel writes only the termination codes and ``done`` is returned as None
        (done == (info["term"] != 0)): one byte per env-step of HBM writes less."""
        a = self._actions(actions)
        flags = AUTO_RESET if self.auto_reset else 0
        _lib.check(self._L.boatenv_step(self._h, a.data_ptr(), self.obs.data_ptr(), self.reward.data_ptr(),
                                        None if done_from_term else self.done.data_ptr(), self.term.data_ptr(),
                                        self.final_obs.data_ptr(), flags, self._stream()), "boatenv_step")
        return (self.obs, self.reward, None if done_from_term else self.done,
                {"term": self.term, "final_obs": self.final_obs})

    def step_k(self, actions, k, steps_out=None):
        """k fused sub-steps; ``actions`` is [k, N] or [N] (repeated)."""
        torch = _torch()
        a = self._actions(actions)
        stride = self.n_envs if a.dim() == 2 else 0
        if a.dim() == 2 and a.shape[0] != k:
            raise ValueError("actions must be [k, n_envs] or [n_envs]")
        if steps_out is None:
            steps_out = torch.empty(self.n_envs, dtype=torch.int32, device=self.device)
        flags = AUTO_RESET if self.auto_reset else 0
        _lib.check(self._L.boatenv_step_k(self._h, a.data_ptr(), stride, int(k), self.obs.data_ptr(),
                                          self.reward.data_ptr(), self.done.data_ptr(), self.term.data_ptr(),
                                          steps_out.data_ptr(), flags, self._stream()), "boatenv_step_k")
        return self.obs, self.reward, self.done, {"term": self.term, "steps": steps_out}

    def step_host(self, actions_host, obs_host, reward_host, done_host, term_host=None):
        """End-to-end step through HOST (ideally pinned) buffers; blocks until the results
        are in host memory.  Ordered after the work queued on torch's current stream (an event wait,
        no device-wide synchronise)."""
        flags = AUTO_RESET if self.auto_reset else 0
        _lib.check(self._L.boatenv_step_host_stream(self._h, actions_host.data_ptr(), obs_host.data_ptr(),
                                                    reward_host.data_ptr(), done_host.data_ptr(),
                                                    None if term_host is None else term_host.data_ptr(), flags,
                                                    self._stream()), "boatenv_step_host_stream")
        return obs_host, reward_host, done_host

    def step_k_host(self, actions_host, k, obs_host, reward_host, done_host, term_host=None, steps_host=None):
        """K fused sub-steps through HOST buffers: ``actions_host`` [k, n_envs] in, one observation / summed
        reward / done (/ termination code / executed sub-steps) per env out."""
        flags = AUTO_RESET if self.auto_reset else 0
        if tuple(actions_host.shape) != (int(k), self.n_envs):
            raise ValueError("actions_host must be [k, n_envs]")
        _lib.check(self._L.boatenv_step_k_host(self._h, actions_host.data_ptr(), int(k), obs_host.data_ptr(),
                                               reward_host.data_ptr(), done_host.data_ptr(),
                                               None if term_host is None else term_host.data_ptr(),
                                               None if steps_host is None else steps_host.data_ptr(), flags,
                                               self._stream()), "boatenv_step_k_host")
        return obs_host, reward_host, done_host

    # -- state access ------------------------------------------------------------------
    def get_field(self, name):
        torch = _torch()
        f = FIELDS[name]
        dt = self.dtype if f < 8 else torch.int32
        out = torch.empty(self.n_envs, dtype=dt, device=self.device)
        _lib.check(self._L.boatenv_get_field(self._h, f, out.data_ptr(), self._stream()), "boatenv_get_field")
        return out

    def set_field(self, name, values):
        torch = _torch()
        f = FIELDS[name]
        dt = self.dtype if f < 8 else torch.int32
        v = torch.as_tensor(values, device=self.device).to(dt).contiguous()
        assert v.numel() == self.n_envs
        _lib.check(self._L.boatenv_set_field(self._h, f, v.data_ptr(), self._stream()), "boatenv_set_field")

    def record_rows(self, ids, ring, row, actions=None, reward=None, term=None):
        """One recorder row (boatenv_record_rows): state, action, reward and termination code of the LOCAL env ids
        ``ids`` (int64 device tensor) into row ``row % ring.capacity`` of ``ring`` (a ``_lib.RecordRing``).
        ``actions`` / ``reward`` / ``term`` are the step's [n_envs] device tensors, or None for zeros.  One launch on
        the current stream, no synchronisation."""
        ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        _lib.check(self._L.boatenv_record_rows(self._h, ids.data_ptr(), ids.numel(), ptr(actions), ptr(reward),
                                               ptr(term), C.byref(ring), int(row), self._stream()),
                   "boatenv_record_rows")

    @property
    def wind_length(self):
        return int(self._L.boatenv_wind_length(self._h))

    def wind_table(self, env_index=0):
        """(wind_velocity, wind_angle) of env's current episode as float64 numpy arrays."""
        torch = _torch()
        L = self.wind_length
        wv = torch.empty(L, dtype=torch.float64, device=self.device)
        wa = torch.empty(L, dtype=torch.float64, device=self.device)
        _lib.check(self._L.boatenv_wind_table(self._h, int(env_index), wv.data_ptr(), wa.data_ptr(),
                                              self._stream()), "boatenv_wind_table")
        return wv.cpu().numpy(), wa.cpu().numpy()

    def set_episode_draws(self, s_y_start=None, knots=None):
        """Validation hook: prescribe the np.random draws of every later episode."""
        torch = _torch()
        s = k = None
        if s_y_start is not None:
            s = torch.as_tensor(np.asarray(s_y_start, dtype=np.int32), device=self.device).contiguous()
            assert s.numel() == self.n_envs
        if knots is not None:
            fp = int(self.params.fixed_points)
            k = torch.as_tensor(np.ascontiguousarray(knots, dtype=np.float64), device=self.device).contiguous()
            assert k.numel() == self.n_envs * 2 * fp
        _lib.check(self._L.boatenv_set_episode_draws(self._h, None if s is None else s.data_ptr(),
                                                     None if k is None else k.data_ptr(), self._stream()),
                   "boatenv_set_episode_draws")
        torch.cuda.current_stream(self.device).synchronize()

    def episode_draws(self, env_index, episode):
        """The Philox draws of (global env, episode): (s_y_start, knots[2, fixed_points])."""
        fp = int(self.params.fixed_points)
        s = C.c_int32()
        k = (C.c_double * (2 * fp))()
        _lib.check(self._L.boatenv_episode_draws_host(C.byref(self.params), self.seed,
                                                      self.env_id_offset + int(env_index), int(episode),
                                                      C.byref(s), k), "boatenv_episode_draws_host")
        return int(s.value), np.array(k[:], dtype=np.float64).reshape(2, fp)

    def episode_draws_batch(self, env_indices, episodes, episode_begin=0):
        """The Philox draws of many (env, episode) pairs in one host call:
        (s_y_start int32[episodes, M], knots float64[episodes, M, 2, fixed_points])."""
        fp = int(self.params.fixed_points)
        ids = np.ascontiguousarray(np.asarray(env_indices, dtype=np.int64) + self.env_id_offset)
        s_y = np.empty((int(episodes), len(ids)), dtype=np.int32)
        knots = np.empty((int(episodes), len(ids), 2, fp), dtype=np.float64)
        _lib.check(self._L.boatenv_episode_draws_batch_host(C.byref(self.params), self.seed, ids.ctypes.data, len(ids),
                                                            int(episode_begin), int(episodes), s_y.ctypes.data,
                                                            knots.ctypes.data), "boatenv_episode_draws_batch_host")
        return s_y, knots

    # -- checkpoint / resume -----------------------------------------------------------
    def state_dict(self):
        """Everything needed to resume this population exactly: the opaque device state blob (per-env
        scalars, step / episode indices, wind coefficients, cumulative statistics) plus the host-side
        identity of the handle.  The Philox streams are counter-based, so nothing else is stateful."""
        torch = _torch()
        blob = torch.empty(int(self._L.boatenv_state_bytes(self._h)), dtype=torch.uint8, device=self.device)
        _lib.check(self._L.boatenv_export_state(self._h, blob.data_ptr(), self._stream()), "boatenv_export_state")
        return {"format": STATE_FORMAT, "blob": blob, "obs": self.obs.clone(), "n_envs": self.n_envs, "precision": self.precision,
                "seed": self.seed, "env_id_offset": self.env_id_offset,
                "params": bytes(memoryview(self.params).cast("B"))}

    def load_state_dict(self, sd):
        torch = _torch()
        if sd.get("format", 1) != STATE_FORMAT:
            raise ValueError(f"checkpoint state layout {sd.get('format', 1)} != {STATE_FORMAT} (the fp32 mode's rudder / position "
                             "slots changed encoding in format 2)")
        for k in ("n_envs", "precision", "seed", "env_id_offset"):
            if sd[k] != getattr(self, k):
                raise ValueError(f"checkpoint {k}={sd[k]!r} does not match this env ({getattr(self, k)!r})")
        if sd["params"] != bytes(memoryview(self.params).cast("B")):
            raise ValueError("checkpoint was taken with a different config")
        blob = sd["blob"].to(self.device).contiguous()
        if blob.numel() != int(self._L.boatenv_state_bytes(self._h)):
            raise ValueError("checkpoint blob has the wrong size")
        _lib.check(self._L.boatenv_import_state(self._h, blob.data_ptr(), self._stream()), "boatenv_import_state")
        self.obs.copy_(sd["obs"])
        torch.cuda.current_stream(self.device).synchronize()

    def counters(self):
        out = (C.c_double * 8)()
        _lib.check(self._L.boatenv_get_counters(self._h, out, self._stream()), "boatenv_get_counters")
        return dict(zip(COUNTER_NAMES, [float(x) for x in out]))

    def counters_tensor(self):
        """The 8 counters as a device tensor (input of the NCCL all-reduce)."""
        torch = _torch()
        out = torch.empty(8, dtype=torch.float64, device=self.device)
        _lib.check(self._L.boatenv_reduce_counters(self._h, out.data_ptr(), self._stream()),
                   "boatenv_reduce_counters")
        return out

    def uniform_actions(self, step_counter, scale=1.0, out=None):
        torch = _torch()
        if out is None:
            out = torch.empty(self.n_envs, dtype=self.dtype, device=self.device)
        _lib.check(self._L.boatenv_fill_uniform_actions(self._h, int(step_counter), float(scale),
                                                        out.data_ptr(), self._stream()),
                   "boatenv_fill_uniform_actions")
        return out


class _WindFacade:
    """env.boat.wind (recorder.py:46-47): wind_velocity / wind_angle arrays of length L."""

    def __init__(self, benv):
        self._b = benv

    @property
    def wind_velocity(self):
        return self._b.wind_table(0)[0]

    @property
    def wind_angle(self):
        return self._b.wind_table(0)[1]


class _BoatFacade:
    """env.boat attributes read by main.py:94 and return_all_data (boat_env.py:128-140)."""

    def __init__(self, benv, cfg):
        self._b = benv
        self.n = 20
        self.dt = cfg.base_settings.dt if hasattr(cfg, "base_settings") else cfg["base_settings"]["dt"]
        self.wind = _WindFacade(benv)

        self._state = (C.c_double * 10)()
        self._fresh = False   # BoatEnv.step / reset invalidate; the first attribute read refetches all ten

    def invalidate(self):
        self._fresh = False

    def _f(self, name):
        if not self._fresh:  # one launch for all fields (boatenv_env_state_host)
            _lib.check(self._b._L.boatenv_env_state_host(self._b._h, 0, self._state), "boatenv_env_state_host")
            self._fresh = True
        return self._state[FIELDS[name]]

    s_x = property(lambda self: self._f("s_x"))
    s_y = property(lambda self: self._f("s_y"))
    s_r = property(lambda self: self._f("s_r"))
    v_x = property(lambda self: self._f("v_x"))
    v_y = property(lambda self: self._f("v_y"))
    v_r = property(lambda self: self._f("v_r"))
    rudder_angle = property(lambda self: self._f("rudder_angle"))
    index = property(lambda self: int(self._f("index")))

    @property
    def t(self):
        return self.index * self.dt

    @property
    def fuel(self):
        return self._b.params.fuel - self.index


class BoatEnv:
    """Single-env drop-in for the reference's ``BoatEnv`` (boat_env.py:9-140), running on
    the same CUDA kernels with n_envs = 1.  Returns numpy float64 observations, Python
    floats and the reference's cumulative ``info`` dict (sticky 'termination' included)."""

    def __init__(self, config=None, experiment=None, seed=0, precision="fp64", device=None):
        self.config = config if config is not None else load_config()
        self.experiment_dir = getattr(experiment, "experiment_dir", None)
        self._b = BatchedBoatEnv(self.config, 1, seed=seed, precision=precision, device=device,
                                 auto_reset=False)
        self.action = [0]
        self.reward = 0
        self.boat = _BoatFacade(self._b, self.config)
        self.info = {"termination": "", "reached_goal": 0, "out_of_bounds": 0, "out_of_fuel": 0,
                     "rudder_broken": 0, "timeout": 0, "episode_reward": 0}
        self.action_space = self._b.action_space
        self.observation_space = self._b.observation_space
        self.low_state, self.high_state = self.observation_space.low, self.observation_space.high
        # host buffers of the one-call-per-step host path (boatenv_step_host_term; zero-copy for one env)
        ft = np.float32 if self._b.precision == 32 else np.float64
        self._h_act, self._h_obs, self._h_rew = np.zeros(1, ft), np.zeros((1, 11), ft), np.zeros(1, ft)
        self._h_done, self._h_term = np.zeros(1, np.uint8), np.zeros(1, np.uint8)
        self._ptrs = tuple(x.ctypes.data for x in (self._h_act, self._h_obs, self._h_rew, self._h_done, self._h_term))
        self._b.reset()  # BoatEnv.__init__ builds a Boat (boat_env.py:15)

    def reset(self):
        obs = self._b.reset()
        self.boat.invalidate()
        self.info["episode_reward"] = 0  # boat_env.py:122 (the other keys persist)
        self.state = obs[0].double().cpu().numpy()
        return self.state

    def step(self, action):
        self.action = action
        self._h_act[0] = np.asarray(action).reshape(-1)[0]
        b = self._b
        _lib.check(b._L.boatenv_step_host_term(b._h, *self._ptrs, 0), "boatenv_step_host_term")
        self.boat.invalidate()
        code = int(self._h_term[0])
        self.reward = float(self._h_rew[0])
        if code:
            self.info["termination"] = TERM_NAMES[code]
            self.info[TERM_NAMES[code]] += 1
        self.info["episode_reward"] += self.reward
        self.state = self._h_obs[0].astype(np.float64)  # a fresh array every call, like boat_env.py:309
        return self.state, self.reward, bool(self._h_done[0]), self.info

    def render(self):
        pass

    def return_all_data(self):
        b = self.boat
        return {"boat_position_x": b.s_x, "boat_position_y": b.s_y, "boat_velocity_x": b.v_x,
                "boat_velocity_y": b.v_y, "boat_angle": b.s_r, "action_rudder": self.action[0],
                "reward": self.reward, "rudder_angle": b.rudder_angle, "n": b.n}

    def close(self):
        self._b.close()
