"""Host-side mirror of the reference's ``ReplayBuffer`` (agent/buffer.py:3-35) on the
device-resident ring of libboatenv.so.

Drop-in for ``ContinuousAgent`` (continuous_agent.py:15-17,64,97-101):
``ReplayBuffer(max_size, input_shape, n_actions)``, ``store_transition(s, a, r, s_, done)``,
``sample_buffer(batch) -> (states, actions, rewards, states_, dones)``, ``mem_cntr``,
``mem_size``.  Additions for the batched path: ``store_batch`` (N rows per call),
``sample_buffer(..., as_torch=True)`` (results stay on the GPU) and
``BatchedBoatEnv``-fused ``step_store``.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib


def _torch():
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("sac_agent_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch


class ReplayBuffer:
    def __init__(self, max_size, input_shape, n_actions, precision="fp64", device=None, seed=0,
                 as_torch=False):
        torch = _torch()
        self.mem_size = int(max_size)
        self.obs_dim = int(np.prod(input_shape))
        self.input_shape = tuple(input_shape)
        self.n_actions = int(n_actions)
        self.precision = {"fp32": 32, "fp64": 64, 32: 32, 64: 64}[precision]
        self.dtype = torch.float32 if self.precision == 32 else torch.float64
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
        self.seed = int(seed)
        self.as_torch = bool(as_torch)
        self._samples = 0  # Philox counter: one per sample_buffer call
        self._L = _lib.lib()
        h = C.c_void_p()
        _lib.check(self._L.boatreplay_create(self.mem_size, self.obs_dim, self.n_actions, self.precision,
                                             self.device.index, C.byref(h)), "boatreplay_create")
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._L.boatreplay_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(_torch().cuda.current_stream(self.device).cuda_stream)

    @property
    def mem_cntr(self):
        return int(self._L.boatreplay_mem_cntr(self._h))

    # -- store -------------------------------------------------------------------------
    def _dev(self, x, shape):
        torch = _torch()
        if not isinstance(x, torch.Tensor):
            x = torch.as_tensor(np.asarray(x, dtype=np.float64))
        return x.to(device=self.device, dtype=self.dtype).reshape(shape).contiguous()

    def store_batch(self, states, actions, rewards, states_, dones):
        """n transitions, row i going to slot (mem_cntr + i) % mem_size."""
        torch = _torch()
        n = int(np.prod(rewards.shape)) if hasattr(rewards, "shape") else 1
        s = self._dev(states, (n, self.obs_dim))
        s2 = self._dev(states_, (n, self.obs_dim))
        a = self._dev(actions, (n, self.n_actions))
        r = self._dev(rewards, (n,))
        if not isinstance(dones, torch.Tensor):
            dones = torch.as_tensor(np.asarray(dones).astype(np.uint8))
        d = dones.to(device=self.device).to(torch.uint8).reshape(n).contiguous()
        _lib.check(self._L.boatreplay_store(self._h, n, s.data_ptr(), a.data_ptr(), r.data_ptr(), s2.data_ptr(),
                                            d.data_ptr(), self._stream()), "boatreplay_store")

    def store_transition(self, state, action, reward, state_, done):
        """buffer.py:13-22 -- one transition (numpy / python scalars, like the reference)."""
        self.store_batch(np.asarray(state, dtype=np.float64).reshape(1, -1),
                         np.asarray(action, dtype=np.float64).reshape(1, -1),
                         np.asarray([reward], dtype=np.float64), np.asarray(state_, dtype=np.float64).reshape(1, -1),
                         np.asarray([bool(done)]))

    # -- sample --------------------------------------------------------------------------
    def _outputs(self, batch):
        torch = _torch()
        kw = dict(dtype=self.dtype, device=self.device)
        return (torch.empty((batch, self.obs_dim), **kw), torch.empty((batch, self.n_actions), **kw),
                torch.empty(batch, **kw), torch.empty((batch, self.obs_dim), **kw),
                torch.empty(batch, dtype=torch.uint8, device=self.device))

    def _finish(self, s, a, r, s2, d, as_torch):
        if as_torch:
            return s.reshape(-1, *self.input_shape), a, r, s2.reshape(-1, *self.input_shape), d.bool()
        return (s.double().cpu().numpy().reshape(-1, *self.input_shape), a.double().cpu().numpy(),
                r.double().cpu().numpy(), s2.double().cpu().numpy().reshape(-1, *self.input_shape),
                d.cpu().numpy().astype(bool))

    def sample_buffer(self, batch_size, as_torch=None, return_indices=False, out=None):
        """buffer.py:24-35: uniform with replacement over [0, min(mem_cntr, mem_size)).
        ``out`` = (states, actions, rewards, states_, dones-as-uint8) device tensors to fill in place
        (a learner's static batch: no allocation, nothing but the gather kernel is launched); they
        are returned as they are."""
        torch = _torch()
        batch = int(batch_size)
        if self.mem_cntr == 0:
            raise ValueError("a must be non-empty")  # np.random.choice(0, n)
        if out is not None:
            s, a, r, s2, d = out
            if (s.shape[0] != batch or s.dtype != self.dtype or d.dtype != torch.uint8
                    or not all(t.is_contiguous() and t.device == self.device for t in out)):
                raise ValueError("out: five contiguous tensors on the buffer's device, dtype of the buffer / uint8")
            _lib.check(self._L.boatreplay_sample(self._h, batch, self.seed, self._samples, s.data_ptr(), a.data_ptr(),
                                                 r.data_ptr(), s2.data_ptr(), d.data_ptr(), None, self._stream()),
                       "boatreplay_sample")
            self._samples += 1
            return out
        s, a, r, s2, d = self._outputs(batch)
        idx = torch.empty(batch, dtype=torch.int64, device=self.device) if return_indices else None
        _lib.check(self._L.boatreplay_sample(self._h, batch, self.seed, self._samples, s.data_ptr(), a.data_ptr(),
                                             r.data_ptr(), s2.data_ptr(), d.data_ptr(),
                                             None if idx is None else idx.data_ptr(), self._stream()),
                   "boatreplay_sample")
        self._samples += 1
        out = self._finish(s, a, r, s2, d, self.as_torch if as_torch is None else as_torch)
        return (*out, idx) if return_indices else out

    def gather(self, indices, as_torch=None):
        """The fancy-index gather of buffer.py:29-33 with caller-supplied indices."""
        torch = _torch()
        idx = torch.as_tensor(np.asarray(indices, dtype=np.int64) if not isinstance(indices, torch.Tensor)
                              else indices).to(device=self.device, dtype=torch.int64).contiguous()
        batch = idx.numel()
        s, a, r, s2, d = self._outputs(batch)
        _lib.check(self._L.boatreplay_gather(self._h, batch, idx.data_ptr(), s.data_ptr(), a.data_ptr(),
                                             r.data_ptr(), s2.data_ptr(), d.data_ptr(), self._stream()),
                   "boatreplay_gather")
        return self._finish(s, a, r, s2, d, self.as_torch if as_torch is None else as_torch)

    # -- checkpoint / resume (SURVEY.md 8f rank 4) -----------------------------------------
    def state_dict(self):
        """The ring's five arrays (only the rows written so far), its store counter and its Philox sample counter:
        a restored buffer stores to the same slots and draws the same batches."""
        torch = _torch()
        n = min(self.mem_cntr, self.mem_size)
        s, a, r, s2, d = self._outputs(n) if n else self._outputs(0)
        if n:
            idx = torch.arange(n, dtype=torch.int64, device=self.device)
            _lib.check(self._L.boatreplay_gather(self._h, n, idx.data_ptr(), s.data_ptr(), a.data_ptr(), r.data_ptr(),
                                                 s2.data_ptr(), d.data_ptr(), self._stream()), "boatreplay_gather")
        return {"state": s, "action": a, "reward": r, "new_state": s2, "terminal": d, "mem_cntr": self.mem_cntr,
                "mem_size": self.mem_size, "samples": self._samples, "seed": self.seed, "precision": self.precision}

    def load_state_dict(self, sd):
        torch = _torch()
        if int(sd["mem_size"]) != self.mem_size or int(sd["precision"]) != self.precision:
            raise ValueError("checkpoint was taken from a ring of another size / precision")
        n = min(int(sd["mem_cntr"]), self.mem_size)
        _lib.check(self._L.boatreplay_set_mem_cntr(self._h, 0), "boatreplay_set_mem_cntr")
        if n:   # rows 0..n-1 go back to slots 0..n-1, then the counter jumps to its old value
            mv = lambda t, dt: t.to(device=self.device, dtype=dt).contiguous()  # noqa: E731
            _lib.check(self._L.boatreplay_store(self._h, n, mv(sd["state"], self.dtype).data_ptr(),
                                                mv(sd["action"], self.dtype).data_ptr(), mv(sd["reward"], self.dtype).data_ptr(),
                                                mv(sd["new_state"], self.dtype).data_ptr(),
                                                mv(sd["terminal"], torch.uint8).data_ptr(), self._stream()), "boatreplay_store")
            torch.cuda.current_stream(self.device).synchronize()   # the staging tensors above die here
        _lib.check(self._L.boatreplay_set_mem_cntr(self._h, int(sd["mem_cntr"])), "boatreplay_set_mem_cntr")
        self._samples, self.seed = int(sd["samples"]), int(sd["seed"])

    # -- fused env.step + agent.remember (main.py:81-88) ---------------------------------
    def step_store(self, env, actions, done_flag_mode=1):
        """Steps every env of ``env`` (a BatchedBoatEnv) and writes the transitions
        (env.obs as s, action, reward, new obs as s', done flag) into the ring in the same
        kernel.  done_flag_mode 1 stores ``termination == 'reached_goal'`` like
        main.py:83-88, 0 stores ``done``."""
        a = env._actions(actions)
        flags = 1 if env.auto_reset else 0
        _lib.check(self._L.boatenv_step_store(env._h, self._h, a.data_ptr(), env.obs.data_ptr(),
                                              env.reward.data_ptr(), env.done.data_ptr(), env.term.data_ptr(),
                                              int(done_flag_mode), flags, self._stream()), "boatenv_step_store")
        return env.obs, env.reward, env.done, {"term": env.term}


class PrioritizedReplayBuffer(ReplayBuffer):
    """Prioritized experience replay (Schaul et al. 2016, proportional variant) over the device ring: a sum tree of
    the slots' priorities (libboatenv's boatper_*), stratified draws with importance weights, and priorities set from
    the learner's TD errors.  A new row gets the largest priority given so far; ``update_priorities`` sets a drawn
    row's priority to (|TD| + eps)^alpha.  The ring's store paths (store_batch, step_store, collect) are unchanged:
    the rows stored since the last draw get their priority at the next ``sample_buffer``."""

    def __init__(self, max_size, input_shape, n_actions, precision="fp64", device=None, seed=0, as_torch=False,
                 alpha=0.6, eps=1e-6):
        if not float(alpha) >= 0.0 or not float(eps) > 0.0:
            raise ValueError(f"PrioritizedReplayBuffer: alpha >= 0 and eps > 0 (got alpha {alpha}, eps {eps})")
        super().__init__(max_size, input_shape, n_actions, precision=precision, device=device, seed=seed,
                         as_torch=as_torch)
        self.alpha, self.eps = float(alpha), float(eps)
        self._per_samples = 0   # Philox counter of the stratified draws: one per sample_buffer call
        self._filled = 0        # mem_cntr at the last fill: rows from here on have no priority yet
        p = C.c_void_p()
        _lib.check(self._L.boatper_create(self.mem_size, self.device.index, C.byref(p)), "boatper_create")
        self._p = p

    def close(self):
        if getattr(self, "_p", None):
            self._L.boatper_destroy(self._p)
            self._p = None
        super().close()

    def _fill_new(self):
        n = self.mem_cntr - self._filled
        if n:
            _lib.check(self._L.boatper_fill_new(self._p, self._filled, n, self._stream()), "boatper_fill_new")
            self._filled += n

    def sample_buffer(self, batch_size, beta=0.4, as_torch=None, out=None, idx_out=None, weight_out=None):
        """``batch_size`` stratified draws: row j from the j-th of equal slices of the priority mass.  Returns the five
        batch arrays, then the drawn slots (int64) and the importance weights (n P(j))^-beta normalised by their batch
        maximum (float32), both device tensors.  ``out`` as in ReplayBuffer.sample_buffer; ``idx_out`` / ``weight_out``
        are filled in place when given.  Nothing waits for the device."""
        torch = _torch()
        batch = int(batch_size)
        if self.mem_cntr == 0:
            raise ValueError("a must be non-empty")
        self._fill_new()
        if idx_out is None:
            idx_out = torch.empty(batch, dtype=torch.int64, device=self.device)
        if weight_out is None:
            weight_out = torch.empty(batch, dtype=torch.float32, device=self.device)
        if (idx_out.shape != (batch,) or idx_out.dtype != torch.int64 or weight_out.shape != (batch,)
                or weight_out.dtype != torch.float32 or not idx_out.is_contiguous() or not weight_out.is_contiguous()
                or idx_out.device != self.device or weight_out.device != self.device):
            raise ValueError("idx_out / weight_out: contiguous int64 / float32 [batch] tensors on the buffer's device")
        if out is not None:
            s, a, r, s2, d = out
            if (s.shape[0] != batch or s.dtype != self.dtype or d.dtype != torch.uint8
                    or not all(t.is_contiguous() and t.device == self.device for t in out)):
                raise ValueError("out: five contiguous tensors on the buffer's device, dtype of the buffer / uint8")
        else:
            s, a, r, s2, d = self._outputs(batch)
        _lib.check(self._L.boatper_sample(self._p, batch, self.seed, self._per_samples, float(beta), idx_out.data_ptr(),
                                          weight_out.data_ptr(), self._stream()), "boatper_sample")
        self._per_samples += 1
        _lib.check(self._L.boatreplay_gather(self._h, batch, idx_out.data_ptr(), s.data_ptr(), a.data_ptr(),
                                             r.data_ptr(), s2.data_ptr(), d.data_ptr(), self._stream()),
                   "boatreplay_gather")
        rows = out if out is not None else self._finish(s, a, r, s2, d, self.as_torch if as_torch is None else as_torch)
        return (*rows, idx_out, weight_out)

    def find(self, targets):
        """The slots whose priority prefix ranges hold `targets` (inverse CDF over the sum tree, the descent of
        sample_buffer): an int64 device tensor.  Targets lie in [0, total), total the one entry of the last tree level;
        a target that rounding puts on or past an edge takes the last slot of non-zero priority before it."""
        torch = _torch()
        self._fill_new()
        t = torch.as_tensor(targets).to(device=self.device, dtype=torch.float64).reshape(-1).contiguous()
        out = torch.empty(t.numel(), dtype=torch.int64, device=self.device)
        _lib.check(self._L.boatper_find(self._p, t.numel(), t.data_ptr(), out.data_ptr(), self._stream()),
                   "boatper_find")
        return out

    def update_priorities(self, idx, td):
        """Slot idx[j] gets priority (td[j] + eps)^alpha (a slot drawn twice: the larger); td holds absolute TD errors.
        Device tensors of one length, int64 and float32.  Rows with an index outside the ring, a negative or NaN
        td, or a priority that is not finite are skipped and reported by ``check()``."""
        torch = _torch()
        idx = idx.to(device=self.device, dtype=torch.int64).contiguous()
        td = td.to(device=self.device, dtype=torch.float32).contiguous()
        if idx.numel() != td.numel():
            raise ValueError("update_priorities: idx and td must have the same length")
        _lib.check(self._L.boatper_update(self._p, idx.numel(), idx.data_ptr(), td.data_ptr(), self.alpha, self.eps,
                                          self._stream()), "boatper_update")

    def check(self):
        """Waits for the device; raises if an update since the last check skipped a row."""
        _lib.check(self._L.boatper_check(self._p, self._stream()),
                   "boatper_update: an index outside the ring or a priority that is not finite")

    def tree_level(self, level):
        """A copy of sum-tree level `level`: 0 the fp32 leaf priorities [mem_size], 1.. the fp64 block sums up to the
        one-entry total, -1 max_priority [1]."""
        torch = _torch()
        n = 1 if level < 0 else int(self._L.boatper_level_size(self._p, int(level)))
        if n < 0:
            raise ValueError(f"tree_level: no level {level}")
        t = torch.empty(n, dtype=torch.float64 if level > 0 else torch.float32, device=self.device)
        _lib.check(self._L.boatper_read(self._p, int(level), t.data_ptr(), self._stream()), "boatper_read")
        return t

    def tree_levels(self):
        n = 0
        while self._L.boatper_level_size(self._p, n) > 0:
            n += 1
        return n

    def state_dict(self):
        """ReplayBuffer.state_dict plus the priorities of the filled slots, max_priority, the fill point and the
        stratified-draw counter: a restored buffer draws the same batches."""
        self._fill_new()
        sd = super().state_dict()
        n = min(self._filled, self.mem_size)
        sd.update({"priorities": self.tree_level(0)[:n].clone(), "max_priority": self.tree_level(-1),
                   "priority_filled": self._filled, "priority_samples": self._per_samples,
                   "priority_alpha": self.alpha, "priority_eps": self.eps})
        return sd

    def load_state_dict(self, sd):
        torch = _torch()
        super().load_state_dict(sd)
        if "priorities" not in sd:
            raise ValueError("PrioritizedReplayBuffer.load_state_dict: the checkpoint holds no priorities")
        pr = sd["priorities"].to(device=self.device, dtype=torch.float32).contiguous()
        mp = sd["max_priority"].to(device=self.device, dtype=torch.float32).contiguous()
        self._filled = int(sd["priority_filled"])
        _lib.check(self._L.boatper_load(self._p, pr.data_ptr(), pr.numel(), mp.data_ptr(),
                                        min(self._filled, self.mem_size), self._stream()), "boatper_load")
        torch.cuda.current_stream(self.device).synchronize()   # the staging tensors above die here
        self._per_samples = int(sd["priority_samples"])
        self.alpha, self.eps = float(sd["priority_alpha"]), float(sd["priority_eps"])

