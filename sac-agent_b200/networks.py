"""The three SAC-v1 networks of the reference (networks/networks.py:14-133), device-resident and
batched over envs.  Layer names, shapes and the order they are created in are the reference's
(`fc1, fc2, mean, std` / `fc1, fc2, q` / `fc1, fc2, v`, all 256 wide), so a `state_dict` saved by the
reference's `BaseNetwork.save_checkpoint` (networks/base_network.py:13-17) loads here unchanged and
vice versa.  The dense layers are cuBLAS; the element-wise tail of the policy (tanh-squashed Gaussian
draw and its log-probability: ~60 tiny launches forward + backward in PyTorch) is one libboatenv kernel
each way on the GPU (csrc/agent_ops.cu).  How the learner is driven is in continuous_agent.py (one CUDA
graph per update, batch gathered on the device by libboatenv's replay kernels).
"""
from __future__ import annotations

import ctypes as C
import math
import os

import torch
import torch.nn as nn
import torch.nn.functional as F

LOG_STD_MAX, LOG_STD_MIN = 2.0, -5.0   # networks.py:48-49
REPARAM_NOISE = 1e-6                   # networks.py:22
_HALF_LOG_2PI = 0.5 * math.log(2.0 * math.pi)


class _FusedGaussianHead(torch.autograd.Function):
    """sample_normal after the linear heads as one libboatenv kernel forward and one backward
    (csrc/agent_ops.cu).  Backward is that of the reparameterised draw."""

    @staticmethod
    def forward(ctx, mean, raw_std, eps, max_action):
        from . import _lib
        L = _lib.lib()
        mean, raw_std, eps = mean.contiguous(), raw_std.contiguous(), eps.contiguous()
        rows, n_actions = mean.shape
        action = torch.empty_like(mean)
        log_prob = torch.empty((rows, 1), dtype=mean.dtype, device=mean.device)
        with torch.cuda.device(mean.device):  # the ABI launches on the current device
            stream = torch.cuda.current_stream().cuda_stream
            _lib.check(L.boatagent_gaussian_head_forward(mean.data_ptr(), raw_std.data_ptr(), eps.data_ptr(),
                                                         max_action.data_ptr(), rows, n_actions, action.data_ptr(),
                                                         log_prob.data_ptr(), stream), "boatagent_gaussian_head_forward")
        ctx.save_for_backward(mean, raw_std, eps, max_action)
        ctx.set_materialize_grads(False)
        return action, log_prob

    @staticmethod
    def backward(ctx, grad_action, grad_log_prob):
        from . import _lib
        L = _lib.lib()
        mean, raw_std, eps, max_action = ctx.saved_tensors
        rows, n_actions = mean.shape
        ga = None if grad_action is None else grad_action.contiguous()
        gl = None if grad_log_prob is None else grad_log_prob.contiguous()
        grad_mean, grad_raw = torch.empty_like(mean), torch.empty_like(mean)
        with torch.cuda.device(mean.device):
            stream = torch.cuda.current_stream().cuda_stream
            _lib.check(L.boatagent_gaussian_head_backward(mean.data_ptr(), raw_std.data_ptr(), eps.data_ptr(),
                                                          max_action.data_ptr(), None if ga is None else ga.data_ptr(),
                                                          None if gl is None else gl.data_ptr(), rows, n_actions,
                                                          grad_mean.data_ptr(), grad_raw.data_ptr(), stream),
                       "boatagent_gaussian_head_backward")
        return grad_mean, grad_raw, None, None


class BaseNetwork(nn.Module):
    """networks/base_network.py:5-17 -- checkpoint path = <experiment_dir>/checkpoints/<name>."""

    def __init__(self, name, experiment_dir):
        super().__init__()
        self.name = name
        self.experiment_dir = experiment_dir
        self.checkpoints_dir = os.path.join(experiment_dir, "checkpoints") if experiment_dir is not None else None
        self.checkpoint_file = os.path.join(self.checkpoints_dir, name) if experiment_dir is not None else None

    def save_checkpoint(self):
        os.makedirs(self.checkpoints_dir, exist_ok=True)
        torch.save(self.state_dict(), self.checkpoint_file)

    def load_checkpoint(self):
        dev = next(self.parameters()).device
        self.load_state_dict(torch.load(self.checkpoint_file, map_location=dev))


class ActorNetwork(BaseNetwork):
    """networks.py:14-70: tanh-squashed Gaussian policy; the std head goes through tanh into
    log_std in [-5, 2]."""

    def __init__(self, experiment_dir, input_dims, max_action, fc1_dims=256, fc2_dims=256, n_actions=1,
                 name="actor_network"):
        super().__init__(name, experiment_dir)
        self.fc1 = nn.Linear(*input_dims, fc1_dims)
        self.fc2 = nn.Linear(fc1_dims, fc2_dims)
        self.mean = nn.Linear(fc2_dims, n_actions)
        self.std = nn.Linear(fc2_dims, n_actions)
        self.register_buffer("max_action", torch.as_tensor(max_action, dtype=torch.float32).reshape(-1), persistent=False)

    def forward(self, state):
        prob = F.relu(self.fc1(state))
        prob = F.relu(self.fc2(prob))
        return self.mean(prob), self.std(prob)

    def act(self, state, precision="fp32"):
        """A non-reparameterised action for every row of `state` without gradients (what choose_action
        needs).  precision "tf32" / "bf16" runs the three dense layers on the tensor cores through cuBLAS
        (acting over ~1e6 envs is GEMM bound in fp32); the head stays fp32.  The learner never uses this."""
        with torch.no_grad():
            if precision == "fp32":
                return self.sample_normal(state, reparameterize=False)[0]
            if precision == "bf16":
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    mean, std = self.forward(state)
            elif precision == "tf32":
                prev = torch.backends.cuda.matmul.allow_tf32
                torch.backends.cuda.matmul.allow_tf32 = True
                try:
                    mean, std = self.forward(state)
                finally:
                    torch.backends.cuda.matmul.allow_tf32 = prev
            else:
                raise ValueError("precision: fp32, tf32 or bf16")
            return self.sample_normal(state, reparameterize=False, heads=(mean.float(), std.float()))[0]

    def sample_normal(self, state, reparameterize=True, eps=None, heads=None):
        """networks.py:47-70.  `eps` (standard-normal, shape [B, n_actions]) replaces the draw -- the
        parity tests inject the reference's noise through it.  `heads` = (mean, std) already computed."""
        mean, std = self.forward(state) if heads is None else heads
        if eps is None:
            eps = torch.randn_like(mean)
        if mean.is_cuda and mean.dtype == torch.float32 and (reparameterize or not torch.is_grad_enabled()):
            # on the GPU the whole head is one kernel (and one for its backward); a non-reparameterised
            # draw is only fused where no gradient is wanted, which is how the update and acting use it
            if not reparameterize:
                mean, std = mean.detach(), std.detach()
            return _FusedGaussianHead.apply(mean, std, eps.to(mean.dtype), self.max_action)
        log_std = LOG_STD_MIN + 0.5 * (LOG_STD_MAX - LOG_STD_MIN) * (torch.tanh(std) + 1.0)
        std = log_std.exp()
        if reparameterize:
            u = mean + eps * std              # Normal.rsample
        else:
            with torch.no_grad():             # Normal.sample: the draw carries no gradient
                u = mean + eps * std
        action = torch.tanh(u) * self.max_action
        # Normal.log_prob(u) - log(1 - action^2 + 1e-6), summed over the action dimensions
        log_probs = -((u - mean) ** 2) / (2.0 * std * std) - log_std - _HALF_LOG_2PI
        log_probs = log_probs - torch.log(1.0 - action.pow(2) + REPARAM_NOISE)
        return action, log_probs.sum(1, keepdim=True)


class CriticNetwork(BaseNetwork):
    """networks.py:73-104: Q(s, a) on cat([state, action])."""

    def __init__(self, experiment_dir, input_dims, n_actions, fc1_dims=256, fc2_dims=256, name="critic_network"):
        super().__init__(name, experiment_dir)
        self.fc1 = nn.Linear(input_dims[0] + n_actions, fc1_dims)
        self.fc2 = nn.Linear(fc1_dims, fc2_dims)
        self.q = nn.Linear(fc2_dims, 1)

    def forward(self, state, action):
        x = F.relu(self.fc1(torch.cat([state, action], dim=1)))
        x = F.relu(self.fc2(x))
        return self.q(x)


class ValueNetwork(BaseNetwork):
    """networks.py:107-133: V(s)."""

    def __init__(self, experiment_dir, input_dims, fc1_dims=256, fc2_dims=256, name="value_network"):
        super().__init__(name, experiment_dir)
        self.fc1 = nn.Linear(*input_dims, fc1_dims)
        self.fc2 = nn.Linear(fc1_dims, fc2_dims)
        self.v = nn.Linear(fc2_dims, 1)

    def forward(self, state):
        x = F.relu(self.fc1(state))
        x = F.relu(self.fc2(x))
        return self.v(x)


class TensorCorePolicy:
    """choose_action over N envs as ONE tcgen05 kernel (csrc/policy_mlp.cu): the actor's three dense layers
    with bf16 inputs / fp32 accumulation and the tanh-squashed draw, a 128-env tile staying on chip from
    the observations to the actions.  Holds the packed bf16 copy of the actor's weights; call `refresh()`
    after the learner changed them.  Acting only -- the learner never uses it."""

    BLOB_BYTES = 256 * 16 * 2 + 256 * 256 * 2 + 16 * 256 * 4 + 256 * 4 + 256 * 4 + 16 * 4

    def __init__(self, actor: ActorNetwork, seed=0):
        from . import _lib
        self._lib, self._L = _lib, _lib.lib()
        self.actor, self.seed = actor, int(seed)
        w1 = actor.fc1.weight
        self.obs_dim, self.n_actions = w1.shape[1], actor.mean.weight.shape[0]
        if (w1.shape[0] != 256 or actor.fc2.weight.shape != (256, 256) or self.obs_dim > 16
                or self.n_actions not in (1, 2, 4, 8)):
            raise ValueError("TensorCorePolicy: 256-wide layers, obs_dim <= 16, n_actions 1, 2, 4 or 8")
        if not w1.is_cuda:
            raise RuntimeError("TensorCorePolicy needs the actor on a CUDA device")
        self.blob = torch.empty(self.BLOB_BYTES, dtype=torch.uint8, device=w1.device)
        self.steps = 0
        self.refresh()

    @staticmethod
    def _cores(w, rows, cols):
        """[r, k] fp32 -> zero-padded [rows, cols] bf16 in 8x8 core-matrix order [cols / 8][rows][8], as bytes."""
        p = torch.zeros((rows, cols), dtype=torch.bfloat16, device=w.device)
        p[: w.shape[0], : w.shape[1]] = w.to(torch.bfloat16)
        return p.view(rows, cols // 8, 8).permute(1, 0, 2).contiguous().view(torch.uint8).reshape(-1)

    @torch.no_grad()
    def refresh(self):
        a = self.actor
        heads_w = torch.zeros((16, 256), dtype=torch.float32, device=self.blob.device)   # fp32, row-major
        heads_w[: 2 * self.n_actions] = torch.cat([a.mean.weight, a.std.weight], 0)
        b3 = torch.zeros(16, dtype=torch.float32, device=self.blob.device)
        b3[: 2 * self.n_actions] = torch.cat([a.mean.bias, a.std.bias], 0)
        parts = [self._cores(a.fc1.weight, 256, 16), self._cores(a.fc2.weight, 256, 256), heads_w.view(torch.uint8).reshape(-1),
                 a.fc1.bias.float().contiguous().view(torch.uint8), a.fc2.bias.float().contiguous().view(torch.uint8),
                 b3.view(torch.uint8)]
        self.blob.copy_(torch.cat(parts))

    @torch.no_grad()
    def act(self, obs, eps=None, out=None):
        """obs float32 [N, obs_dim] (contiguous, on the actor's device) -> actions float32 [N, n_actions].
        eps: optional standard-normal draws [N, n_actions]; otherwise Philox(seed; env, call number)."""
        n = obs.shape[0]
        if obs.dtype != torch.float32 or not obs.is_contiguous() or obs.shape[1] != self.obs_dim:
            raise ValueError("obs: contiguous float32 [N, obs_dim]")
        if out is None:
            out = torch.empty((n, self.n_actions), dtype=torch.float32, device=obs.device)
        if eps is not None:
            eps = eps.to(torch.float32).contiguous()
        with torch.cuda.device(obs.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._lib.check(self._L.boatagent_policy_act(self.blob.data_ptr(), obs.data_ptr(),
                                                         None if eps is None else eps.data_ptr(),
                                                         self.actor.max_action.data_ptr(), self.seed, self.steps, n,
                                                         self.obs_dim, self.n_actions, out.data_ptr(), stream),
                            "boatagent_policy_act")
        self.steps += 1
        return out

    @torch.no_grad()
    def rollout(self, env, max_steps, deterministic=False):
        """Runs every env of the fp32 BatchedBoatEnv `env` under this policy for up to `max_steps` steps in ONE
        kernel (boatagent_rollout, csrc/rollout.cu): each step is the action `act` would draw for that env's row at
        that call, then one env step without auto-reset.  An env whose episode ends is frozen in its terminal state
        (reset() starts the next round).  `deterministic`: action = tanh(mean) * max_action.  Reads and updates
        `env.obs` (the last, or terminal, observation of every env) and advances `steps` by `max_steps`, so later
        `act` calls draw fresh noise.  Returns device tensors (returns float32: the episode_reward slot, steps int32:
        steps taken in this call, term uint8: the termination code, 0 = still running); launches on the current
        stream and does not synchronise."""
        if self.n_actions != 1 or self.obs_dim != 11:
            raise ValueError("rollout: the BoatEnv actor (11 observations, one action)")
        if env.device != self.blob.device:
            raise ValueError("rollout: the env and the policy must be on the same device")
        n = env.n_envs
        returns = torch.empty(n, dtype=torch.float32, device=env.device)
        steps = torch.empty(n, dtype=torch.int32, device=env.device)
        term = torch.empty(n, dtype=torch.uint8, device=env.device)
        flags = 1 if deterministic else 0   # BOATAGENT_ROLLOUT_DETERMINISTIC
        with torch.cuda.device(env.device):
            stream = torch.cuda.current_stream().cuda_stream
            self._lib.check(self._L.boatagent_rollout(env._h, self.blob.data_ptr(), self.actor.max_action.data_ptr(),
                                                      self.seed, self.steps, int(max_steps), flags, env.obs.data_ptr(),
                                                      env.obs.data_ptr(), returns.data_ptr(), steps.data_ptr(),
                                                      term.data_ptr(), stream), "boatagent_rollout")
        self.steps += int(max_steps)
        return returns, steps, term

    @torch.no_grad()
    def collect(self, env, memory, steps, done_flag_mode=1, recorder=None):
        """`steps` rounds of the training loop body -- `act(env.obs)`, then `memory.step_store(env, actions,
        done_flag_mode)` -- over every env of the fp32 auto-resetting BatchedBoatEnv `env`, in ONE kernel
        (boatagent_collect, csrc/rollout.cu): the same actions, env steps, resets and ring rows (fp32 ReplayBuffer
        `memory`) as that loop.  Advances `steps` by `steps`.  Returns (env.obs, env.reward, env.done, {"term":
        env.term}) of the last step, as ReplayBuffer.step_store does; launches on the current stream and does not
        synchronise.
        `recorder`: a DeviceRecorder of `env`; the same kernel (boatagent_collect_record) then writes the `steps`
        rows that a `recorder.capture(actions)` after each round would, flushing the recorder first if they do not
        fit beside its pending rows.  `steps` may not exceed its capacity."""
        steps = int(steps)
        if self.n_actions != 1 or self.obs_dim != 11:
            raise ValueError("collect: the BoatEnv actor (11 observations, one action)")
        if not env.auto_reset:
            raise ValueError("collect: the env must auto-reset (created with auto_reset=True)")
        if env.precision != 32 or memory.precision != 32:
            raise ValueError("collect: fp32 env and replay buffer only")
        if env.device != self.blob.device or memory.device != self.blob.device:
            raise ValueError("collect: the env, the replay buffer and the policy must be on the same device")
        if steps * env.n_envs > memory.mem_size:
            raise ValueError(f"collect: {steps} steps x {env.n_envs} envs exceed the ring's {memory.mem_size} slots "
                             "(rows of one call may not share a slot)")
        if recorder is not None:
            if recorder.env is not env:
                raise ValueError("collect: the recorder records another env")
            if steps > recorder.capacity:
                raise ValueError(f"collect: {steps} steps exceed the recorder's {recorder.capacity} rows "
                                 "(one call would overwrite its own rows)")
        args = (env._h, memory._h, self.blob.data_ptr(), self.actor.max_action.data_ptr(), self.seed, self.steps, steps,
                int(done_flag_mode), env.obs.data_ptr(), env.reward.data_ptr(), env.done.data_ptr(),
                env.term.data_ptr())
        with torch.cuda.device(env.device):
            stream = torch.cuda.current_stream().cuda_stream
            if recorder is None:
                self._lib.check(self._L.boatagent_collect(*args, stream), "boatagent_collect")
            else:
                recorder._record(steps, True, lambda row: self._lib.check(
                    self._L.boatagent_collect_record(*args, recorder._local.data_ptr(), recorder._local.numel(),
                                                     C.byref(recorder._ring), int(row), stream),
                    "boatagent_collect_record"))
        self.steps += steps
        return env.obs, env.reward, env.done, {"term": env.term}
