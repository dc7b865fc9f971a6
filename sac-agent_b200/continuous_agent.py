"""Device-resident mirror of the reference's SAC-v1 agent (agent/continuous_agent.py:9-154,
agent/base_agent.py:3-19) -- SURVEY.md 8(f) rank 1, BASELINE.json configs[4].

Same constructor, attributes and methods as the reference (`choose_action`, `remember`, `learn`,
`update_network_parameters`, `save_models`, `load_models`, `memory`, `actor`, `critic_1`,
`critic_2`, `value`, `target_value`), same update rule and hyper-parameters.  What changes is where
the data lives and how the update is driven:

* the replay memory is libboatenv's device ring (buffer.py); `learn()` gathers its batch with the
  sample kernel straight into the learner's static input tensors -- no host round trip, no H2D
  copies (the reference does five per update, continuous_agent.py:103-107);
* the update of one `learn()` is ONE CUDA-graph launch: the three forward/backward passes and one
  fused Adam + Polyak kernel for all networks (`DeviceAdam`) are captured once and replayed (about a
  hundred small kernels whose launch latency otherwise dominates a 1024 x 256 update); batch and
  Gaussian draws are static inputs of the graph;
* with `data_parallel`, the ranks of a process group train ONE agent: each samples its own ring and computes the
  gradients of its own batch, one all-reduce averages them, and every rank applies the same Adam step;
* `choose_action` takes the [N, 11] observation tensor of a BatchedBoatEnv and returns [N, 1]
  actions without leaving the GPU (the reference syncs one action per env step through
  `.cpu().numpy()`, continuous_agent.py:61); a numpy observation of one env still works and
  returns a numpy action like the reference.

`SACLearner` is the update rule on plain tensors (any torch device): the parity tests drive it with
the batch, initial weights and Gaussian draws of a recorded run of the reference's own `learn()`.
"""
from __future__ import annotations

import copy
import ctypes as C
import math

import numpy as np
import torch
import torch.nn.functional as F

from .buffer import ReplayBuffer
from .networks import ActorNetwork, CriticNetwork, ValueNetwork


class _AdamSlot(C.Structure):
    """Mirror of `boatagent_adam_slot` (include/boatenv.h)."""
    _fields_ = [("param", C.c_void_p), ("grad", C.c_void_p), ("exp_avg", C.c_void_p), ("exp_avg_sq", C.c_void_p),
                ("target", C.c_void_p), ("numel", C.c_int64), ("lr", C.c_float), ("_pad", C.c_int32)]


class DeviceAdam:
    """torch.optim.Adam (default betas / eps, as networks.py:31,88,121 constructs it) for a list of
    (parameters, learning rate) groups, fused with the Polyak average of the target network, as ONE
    libboatenv launch per step (`boatagent_adam_polyak_step`, csrc/agent_ops.cu).  The moment tensors
    and the step counter are ordinary torch tensors (`state_dict()` for checkpoints)."""

    def __init__(self, groups, polyak=None, tau=0.0, betas=(0.9, 0.999), eps=1e-8):
        from . import _lib
        self._lib, self._L = _lib, _lib.lib()
        self.params, lrs = [], []
        for ps, lr in groups:
            for p in ps:
                if not (p.is_cuda and p.dtype == torch.float32 and p.is_contiguous()):
                    raise ValueError("DeviceAdam: contiguous float32 CUDA parameters only")
                self.params.append(p)
                lrs.append(float(lr))
        if len(self.params) > 64:
            raise ValueError("DeviceAdam: at most 64 tensors (BOATAGENT_ADAM_MAX_SLOTS)")
        self.exp_avg = [torch.zeros_like(p) for p in self.params]
        self.exp_avg_sq = [torch.zeros_like(p) for p in self.params]
        self.state = torch.zeros(2, dtype=torch.int64, device=self.params[0].device)  # [steps taken, ticket]
        self.betas, self.eps, self.tau = betas, float(eps), float(tau)
        targets = {id(p): t for p, t in (polyak or [])}
        self._slots = (_AdamSlot * len(self.params))()
        for k, p in enumerate(self.params):
            t = targets.get(id(p))
            self._slots[k] = _AdamSlot(p.data_ptr(), 0, self.exp_avg[k].data_ptr(), self.exp_avg_sq[k].data_ptr(),
                                       None if t is None else t.data_ptr(), p.numel(), lrs[k], 0)

    def step(self, grads):
        """grads: one contiguous float32 tensor per parameter, in construction order."""
        for k, g in enumerate(grads):
            if g.dtype != torch.float32 or not g.is_contiguous() or g.shape != self.params[k].shape:
                raise ValueError(f"DeviceAdam.step: gradient {k} must be a contiguous float32 tensor of the parameter's shape")
            self._slots[k].grad = g.data_ptr()
        with torch.cuda.device(self.params[0].device):  # the ABI launches on the current device
            stream = torch.cuda.current_stream().cuda_stream
            self._lib.check(self._L.boatagent_adam_polyak_step(self._slots, len(self.params), self.betas[0],
                                                               self.betas[1], self.eps, self.tau,
                                                               self.state.data_ptr(), stream),
                            "boatagent_adam_polyak_step")

    def state_tensors(self):
        return [self.state] + self.exp_avg + self.exp_avg_sq

    def state_dict(self):
        return {"state": self.state, "exp_avg": self.exp_avg, "exp_avg_sq": self.exp_avg_sq}


class SACLearner:
    """The five networks, their Adam optimisers and one SAC-v1 update (continuous_agent.py:96-154)."""

    def __init__(self, input_dims, n_actions, max_action, alpha, beta, gamma, tau, reward_scale, experiment_dir=None,
                 device="cuda", torch_reference_math=False):
        self.device = torch.device(device)
        if self.device.type != "cuda" and not torch_reference_math:
            # no silent CPU fallback: off the GPU the head and the optimiser are plain PyTorch (the restatement
            # the parity tests compare the reference's learn() with), and that has to be asked for
            raise RuntimeError("SACLearner needs a CUDA device; pass torch_reference_math=True for the PyTorch "
                               "restatement of the update (parity tests only)")
        self.gamma, self.tau, self.scale = float(gamma), float(tau), float(reward_scale)
        d = tuple(input_dims)
        # creation order = the reference's (continuous_agent.py:19-52): identical torch seeds give identical weights
        self.actor = ActorNetwork(experiment_dir, d, max_action, n_actions=n_actions, name="actor_network")
        self.critic_1 = CriticNetwork(experiment_dir, d, n_actions, name="critic_network_1")
        self.critic_2 = CriticNetwork(experiment_dir, d, n_actions, name="critic_network_2")
        self.value = ValueNetwork(experiment_dir, d, name="value_network")
        self.target_value = ValueNetwork(experiment_dir, d, name="target_value_network")
        for net in self.networks():
            net.to(self.device)
        # The reference keeps one Adam per network (networks.py:31,88,121) and steps them at three points of
        # learn().  Nothing computed after a step reads the stepped weights (the critics are stepped last, the
        # value net is only read again by the Polyak update), so ONE optimiser step over two learning rates
        # after the three backward passes is the same arithmetic.  On the GPU that step and the Polyak
        # average are one libboatenv launch (DeviceAdam); on the CPU (parity tests) it is torch.optim.Adam.
        self._actor_params = list(self.actor.parameters())
        self._critic_params = list(self.critic_1.parameters()) + list(self.critic_2.parameters())
        self._value_params = list(self.value.parameters())
        if self.device.type == "cuda":
            self.optimizer = DeviceAdam([(self._actor_params, alpha), (self._critic_params + self._value_params, beta)],
                                        polyak=list(zip(self._value_params, self.target_value.parameters())), tau=self.tau)
        else:
            self.optimizer = torch.optim.Adam([{"params": self._actor_params, "lr": alpha},
                                               {"params": self._critic_params + self._value_params, "lr": beta}])
        for p in self.target_value.parameters():
            p.requires_grad_(False)
        self.update_network_parameters(tau=1.0)  # continuous_agent.py:55

    def networks(self):
        return (self.actor, self.critic_1, self.critic_2, self.value, self.target_value)

    @torch.no_grad()
    def update_network_parameters(self, tau=None):
        """target = tau * value + (1 - tau) * target (continuous_agent.py:66-80)."""
        tau = self.tau if tau is None else float(tau)
        tgt, src = list(self.target_value.parameters()), list(self.value.parameters())
        if tau == 1.0:
            torch._foreach_copy_(tgt, src)
            return
        torch._foreach_mul_(tgt, 1.0 - tau)
        torch._foreach_add_(tgt, src, alpha=tau)

    def update(self, state, action, reward, new_state, done, eps_sample=None, eps_rsample=None):
        """One update on a batch (state [B, obs], action [B, n_actions], reward [B], new_state [B, obs],
        done [B] bool).  eps_*: optional standard-normal draws for the two `sample_normal` calls.
        Returns (value_loss, actor_loss, critic_loss) as 0-d tensors."""
        losses, grads_v, grads_a, grads_c = self._losses_and_grads(state, action, reward, new_state, done, eps_sample,
                                                                   eps_rsample)
        for p, g in zip(self._value_params + self._actor_params + self._critic_params, grads_v + grads_a + grads_c):
            p.grad = g
        if isinstance(self.optimizer, DeviceAdam):   # Adam for all four networks + update_network_parameters (:154)
            self.optimizer.step(grads_a + grads_c + grads_v)
        else:
            self.optimizer.step()
            self.update_network_parameters()                                    # :154
        return losses

    def gradients(self, state, action, reward, new_state, done, eps_sample, eps_rsample, out, scale=1.0):
        """`update` without the optimiser step: writes `scale` times the batch gradients into `out[:-3]` (one tensor
        per parameter in DeviceAdam's order: actor, critic 1, critic 2, value) and `scale` times the three losses
        into `out[-3:]` (0-d tensors).  Leaves weights, optimiser state and `.grad` bindings alone."""
        losses, grads_v, grads_a, grads_c = self._losses_and_grads(state, action, reward, new_state, done, eps_sample,
                                                                   eps_rsample)
        torch._foreach_copy_(out, list(grads_a + grads_c + grads_v) + list(losses))
        if scale != 1.0:
            torch._foreach_mul_(out, scale)

    def _losses_and_grads(self, state, action, reward, new_state, done, eps_sample, eps_rsample):
        """The three losses (detached) and the gradients of the value, actor and critic parameters."""
        with torch.no_grad():
            value_ = self.target_value(new_state).view(-1)
            value_ = torch.where(done, torch.zeros_like(value_), value_)        # value_[done] = 0.0   (:111)
            q_hat = self.scale * reward + self.gamma * value_                     # :141
            # value target: a fresh non-reparameterised action under the current critics (:113-124).  The
            # reference leaves this target attached to the graph, but every gradient it sends to the
            # actor and the critics is zeroed before their own backward passes (:134, :138-139)
            actions, log_probs = self.actor.sample_normal(state, reparameterize=False, eps=eps_sample)
            critic_value = torch.min(self.critic_1(state, actions), self.critic_2(state, actions)).view(-1)
            value_target = critic_value - log_probs.view(-1)
        value = self.value(state).view(-1)
        value_loss = 0.5 * F.mse_loss(value, value_target)
        grads_v = torch.autograd.grad(value_loss, self._value_params)

        actions, log_probs = self.actor.sample_normal(state, reparameterize=True, eps=eps_rsample)  # :127-136
        critic_value = torch.min(self.critic_1(state, actions), self.critic_2(state, actions)).view(-1)
        actor_loss = torch.mean(log_probs.view(-1) - critic_value)
        # only the actor's gradients: what this loss sends into the critics is discarded by the reference too (:138-139)
        grads_a = torch.autograd.grad(actor_loss, self._actor_params)

        q1_old = self.critic_1(state, action).view(-1)                          # :138-152
        q2_old = self.critic_2(state, action).view(-1)
        critic_loss = 0.5 * F.mse_loss(q1_old, q_hat) + 0.5 * F.mse_loss(q2_old, q_hat)
        grads_c = torch.autograd.grad(critic_loss, self._critic_params)
        return (value_loss.detach(), actor_loss.detach(), critic_loss.detach()), grads_v, grads_a, grads_c


class DataParallelState(list):
    """`training_tensors()` of a data-parallel agent: ONE agent's state, held equal by every rank of its group, so
    population rounds (population.exploit_explore) must not hand it between ranks."""


class ContinuousAgent:
    """agent/continuous_agent.py:9-154 on the GPU-resident env and replay ring.

    data_parallel: a torch.distributed process group (True: the default group) whose ranks train this one agent.  Each
    rank keeps its own env shard, ring, sampler seed and Gaussian draws; every update averages the ranks' gradients and
    losses with one all-reduce and applies the same Adam step everywhere, so the weights stay bit-identical without
    being re-broadcast.  Rank 0's weights and optimiser state are broadcast at construction.  Every rank must hold the
    same number of envs (`learn()` updates on all ranks or on none without a vote)."""

    def __init__(self, config, experiment_dir, input_dims, env, device=None, seed=0, use_cuda_graph=True,
                 memory=None, policy_precision="fp32", learner_precision="fp32", data_parallel=None):
        if not torch.cuda.is_available():
            raise RuntimeError("sac_agent_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.env = env
        self.config = config
        a = config.agent
        self.gamma, self.tau, self.scale = a.gamma, a.tvn_parameter_modulation_tau, a.reward_scale
        self.batch_size = int(a.batch_size)
        self.input_dims = tuple(input_dims)
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
        self.memory = memory if memory is not None else ReplayBuffer(
            a.max_size, self.input_dims, self.get_n_actions(), precision="fp32", device=self.device.index, seed=seed,
            as_torch=True)
        self.learner = SACLearner(self.input_dims, self.get_n_actions(), self.get_max_actions(), a.learning_rate_alpha,
                                  a.learning_rate_beta, a.gamma, a.tvn_parameter_modulation_tau, a.reward_scale,
                                  experiment_dir=experiment_dir, device=self.device)
        L = self.learner
        self.actor, self.critic_1, self.critic_2 = L.actor, L.critic_1, L.critic_2
        self.value, self.target_value = L.value, L.target_value
        self.use_cuda_graph = bool(use_cuda_graph)
        if policy_precision not in ("fp32", "tf32", "bf16", "tcgen05"):
            raise ValueError("policy_precision: fp32, tf32, bf16 or tcgen05")
        # acting only: "tf32" / "bf16" run the policy's dense layers through cuBLAS on tensor-core inputs;
        # "tcgen05" is libboatenv's fused kernel (csrc/policy_mlp.cu: bf16 inputs, fp32 accumulation, the
        # whole forward pass and the draw in one launch, weights re-packed after every update)
        self.policy_precision = policy_precision
        if learner_precision not in ("fp32", "tcgen05"):
            raise ValueError("learner_precision: fp32 or tcgen05")
        # "tcgen05": one update is libboatenv's two fused kernels (csrc/learner.cu: bf16 operands for the 256-wide
        # products, fp32 accumulation, everything else fp32) instead of the captured fp32 graph; same tensors, state
        # and checkpoints
        self.learner_precision = learner_precision
        self._tc_policy = None
        self._weight_listeners = []   # callables run after load_models / load_state_dict (acting copies republish)
        B, O, A = self.batch_size, int(np.prod(self.input_dims)), self.get_n_actions()
        kw = dict(dtype=torch.float32, device=self.device)
        # static inputs of the captured update: sample_buffer writes them in place
        self._batch = (torch.zeros((B, O), **kw), torch.zeros((B, A), **kw), torch.zeros(B, **kw),
                       torch.zeros((B, O), **kw), torch.zeros(B, dtype=torch.uint8, device=self.device))
        self._eps = torch.zeros((2, B, A), **kw)  # the Gaussian draws of the two sample_normal calls of one update
        self._graph = None
        self.capture_stream = None   # stream the update graph is captured on (None: torch's own capture stream)
        self._losses = None
        self._act_graphs = {}
        self.updates = 0
        if learner_precision == "tcgen05":
            self._init_fused_learner()
        self._dp = None   # (group, flat gradient + loss buffer, its gradient views, grad_scale) in data-parallel mode
        if data_parallel is not None and data_parallel is not False:
            self._init_data_parallel(None if data_parallel is True else data_parallel)

    # -- base_agent.py:7-19 -------------------------------------------------------------
    def get_n_actions(self):
        space = self.env.action_space
        return space.shape[0] if hasattr(space, "shape") and hasattr(space, "high") else space.n

    def get_max_actions(self):
        space = self.env.action_space
        if hasattr(space, "high"):
            return space.high
        raise NotImplementedError

    # -- acting ---------------------------------------------------------------------------
    @torch.no_grad()
    def choose_action(self, observation):
        """continuous_agent.py:57-61.  A torch tensor [N, obs] (a BatchedBoatEnv's `obs`) gives a device
        tensor [N, n_actions]; a numpy observation of ONE env gives a numpy action like the reference."""
        if isinstance(observation, torch.Tensor):
            obs = observation.to(device=self.device, dtype=torch.float32)
            if self.policy_precision == "tcgen05":
                return self.tensor_core_policy().act(obs.reshape(-1, *self.input_dims).contiguous())
            return self.actor.act(obs.reshape(-1, *self.input_dims), self.policy_precision)
        state = torch.as_tensor(np.array([observation]), dtype=torch.float32, device=self.device)
        actions, _ = self.actor.sample_normal(state, reparameterize=False)
        return actions.cpu().numpy()[0]

    def tensor_core_policy(self):
        """The fused tcgen05 policy of this agent's actor (created on first use; `learn()` keeps its packed
        weights current)."""
        if self._tc_policy is None:
            from .networks import TensorCorePolicy
            self._tc_policy = TensorCorePolicy(self.actor, seed=0x5ac)
        return self._tc_policy

    @torch.no_grad()
    def evaluate(self, env, max_steps=None, deterministic=True):
        """render_model (main.py:137-172) over every env of the fp32 BatchedBoatEnv `env`: one episode per env
        under the current actor, run from the env's current state (call ``env.reset()`` first for fresh episodes)
        in one fused kernel (TensorCorePolicy.rollout).  Always acts through the tcgen05 copy of the actor, whatever
        `policy_precision` is, so evaluation acts with bf16 inputs (fp32 accumulation).  `max_steps` defaults to
        enough steps for every episode to end, at the latest by timeout (t_max / dt).  `deterministic`: the mean
        action tanh(mean) * max_action, else a draw as in training.  After ``OverlappedActorLearner`` use, call its
        ``sync()`` first.  Returns (returns, steps, term, summary): the per-env device tensors of the rollout and a
        host dict -- envs, episodes ended, still running, counts per termination kind, goal fraction (of all envs),
        mean / std / min / max return and mean length of the ended episodes."""
        from .boat_env import TERM_NAMES
        if max_steps is None:
            max_steps = int(math.ceil(env.params.t_max / env.params.dt)) + 1
        pol = self.tensor_core_policy()
        pol.refresh()
        returns, steps, term = pol.rollout(env, max_steps, deterministic=deterministic)
        t, r, s = term.cpu().numpy(), returns.double().cpu().numpy(), steps.cpu().numpy()
        ended = t != 0
        rr = r[ended]
        summary = {"envs": int(t.size), "episodes": int(ended.sum()), "running": int((~ended).sum()),
                   "terminations": {TERM_NAMES[k]: int((t == k).sum()) for k in range(1, len(TERM_NAMES))},
                   "goal_fraction": float((t == 1).mean()) if t.size else float("nan"),
                   "return_mean": float(rr.mean()) if rr.size else float("nan"),
                   "return_std": float(rr.std()) if rr.size else float("nan"),
                   "return_min": float(rr.min()) if rr.size else float("nan"),
                   "return_max": float(rr.max()) if rr.size else float("nan"),
                   "length_mean": float(s[ended].mean()) if rr.size else float("nan")}
        return returns, steps, term, summary

    def choose_action_graphed(self, observation):
        """`choose_action` for a PERSISTENT observation tensor (BatchedBoatEnv.obs): the policy's forward
        pass is captured once per tensor and replayed; the result lives in a static output tensor."""
        if self.policy_precision == "tcgen05":   # already one launch (and its Philox counter is a launch argument)
            return self.choose_action(observation)
        key = (observation.data_ptr(), tuple(observation.shape))
        entry = self._act_graphs.get(key)
        if entry is None:
            side = torch.cuda.Stream(self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(side):
                for _ in range(2):
                    self.choose_action(observation)
            torch.cuda.current_stream(self.device).wait_stream(side)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                out = self.choose_action(observation)
            entry = self._act_graphs[key] = (g, out)
        entry[0].replay()
        return entry[1]

    def remember(self, state, action, reward, new_state, done):
        """continuous_agent.py:63-64: one transition, or N of them (leading batch dimension)."""
        if np.ndim(reward) == 0:
            self.memory.store_transition(state, action, reward, new_state, done)
        else:
            self.memory.store_batch(state, action, reward, new_state, done)

    def step_and_remember(self, env, actions, done_flag_mode=1):
        """main.py:81-88 for every env in one kernel: env.step + remember (ReplayBuffer.step_store)."""
        return self.memory.step_store(env, actions, done_flag_mode=done_flag_mode)

    def collect(self, env, steps, done_flag_mode=1, recorder=None):
        """`steps` rounds of choose_action + step_and_remember over every env in ONE kernel
        (TensorCorePolicy.collect): the same actions, steps, resets and ring rows as that loop with
        policy_precision "tcgen05", the only precision it serves.  `recorder`: a DeviceRecorder of `env`, which
        gets the rows a capture() after every round would give, written by the same kernel."""
        if self.policy_precision != "tcgen05":
            raise ValueError(f"collect acts through the tcgen05 policy; this agent acts in {self.policy_precision!r} "
                             "(create it with policy_precision='tcgen05')")
        return self.tensor_core_policy().collect(env, self.memory, steps, done_flag_mode=done_flag_mode,
                                                 recorder=recorder)

    # -- learning -------------------------------------------------------------------------
    def _update_static(self):
        s, a, r, s2, d = self._batch
        return self.learner.update(s, a, r, s2, d.bool(), eps_sample=self._eps[0], eps_rsample=self._eps[1])

    def _init_fused_learner(self):
        B, L = self.batch_size, self.learner
        if self.input_dims != (11,) or self.get_n_actions() != 1 or B <= 0 or B % 128:
            raise ValueError("learner_precision='tcgen05': the BoatEnv agent (11 observations, one action) and a "
                             f"batch size that is a positive multiple of 128 (got {self.input_dims}, "
                             f"{self.get_n_actions()} actions, batch {B})")
        if any(tuple(p.shape) != (256, 256) for p in (L.actor.fc2.weight, L.critic_1.fc2.weight,
                                                      L.critic_2.fc2.weight, L.value.fc2.weight)):
            raise ValueError("learner_precision='tcgen05': 256-wide hidden layers only")
        nbytes = int(L.optimizer._L.boatagent_sac_update_workspace_bytes(B))
        self._ws = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        self._loss_buf = torch.zeros(3, dtype=torch.float32, device=self.device)
        self._losses = tuple(self._loss_buf[k] for k in range(3))

    def _fused_update(self):
        """One update in the two kernels of boatagent_sac_update on the current stream (no sync)."""
        L, o = self.learner, self.learner.optimizer
        for k, p in enumerate(o.params):   # the kernels write the batch gradient where the fp32 learner leaves it
            if p.grad is None:
                p.grad = torch.zeros_like(p)
            o._slots[k].grad = p.grad.data_ptr()
        s, a, r, s2, d = self._batch
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            o._lib.check(o._L.boatagent_sac_update(
                s.data_ptr(), a.data_ptr(), r.data_ptr(), s2.data_ptr(), d.data_ptr(), self._eps.data_ptr(),
                L.actor.max_action.data_ptr(), self.batch_size, float(L.gamma), float(L.scale), o._slots, len(o.params),
                o.betas[0], o.betas[1], o.eps, o.tau, o.state.data_ptr(), self._loss_buf.data_ptr(),
                self._ws.data_ptr(), self._ws.numel(), stream), "boatagent_sac_update")
        return self._losses

    def _init_data_parallel(self, group):
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()):
            raise ValueError("data_parallel needs an initialised torch.distributed process group")
        world = dist.get_world_size(group)
        n = torch.tensor([getattr(self.env, "n_envs", 1)] * 2, dtype=torch.int64, device=self.device)
        n[1].neg_()
        dist.all_reduce(n, op=dist.ReduceOp.MAX, group=group)
        if int(n[0]) != -int(n[1]):
            raise ValueError(f"data_parallel: every rank needs the same number of envs (they hold {-int(n[1])} to "
                             f"{int(n[0])}); make the total divisible by the world size {world}")
        o = self.learner.optimizer
        # every trained parameter's .grad is a view into one flat buffer, followed by the three losses: ONE all-reduce
        flat = torch.zeros(sum(p.numel() for p in o.params) + 3, dtype=torch.float32, device=self.device)
        grads, off = [], 0
        for p in o.params:
            p.grad = flat[off:off + p.numel()].view_as(p)
            grads.append(p.grad)
            off += p.numel()
        self._losses = tuple(flat[off + k] for k in range(3))
        # grad_scale 1 / world: the SUM all-reduce is the mean (exact for power-of-two world sizes)
        self._dp = (group, flat, grads, 1.0 / world)
        src = 0 if group is None else dist.get_global_rank(group, 0)
        for t in self.training_tensors():   # the ranks start from rank 0's agent
            dist.broadcast(t, src=src, group=group)
        self._weights_changed()

    @property
    def data_parallel(self):
        """True when this agent is trained by a process group (constructor argument `data_parallel`)."""
        return self._dp is not None

    def _dp_gradients_static(self):
        s, a, r, s2, d = self._batch
        _, flat, grads, scale = self._dp
        self.learner.gradients(s, a, r, s2, d.bool(), self._eps[0], self._eps[1], grads + list(self._losses), scale)

    def _dp_update(self):
        """gradients (scaled by 1 / world) -> all-reduce of gradients and losses -> Adam + Polyak on every rank."""
        import torch.distributed as dist
        group, flat, grads, scale = self._dp
        L, o = self.learner, self.learner.optimizer
        if self.learner_precision == "tcgen05":
            for k, g in enumerate(grads):
                o._slots[k].grad = g.data_ptr()
            s, a, r, s2, d = self._batch
            stream = torch.cuda.current_stream(self.device).cuda_stream
            with torch.cuda.device(self.device):
                o._lib.check(o._L.boatagent_sac_gradients(
                    s.data_ptr(), a.data_ptr(), r.data_ptr(), s2.data_ptr(), d.data_ptr(), self._eps.data_ptr(),
                    L.actor.max_action.data_ptr(), self.batch_size, float(L.gamma), float(L.scale), o._slots,
                    len(o.params), scale, self._losses[0].data_ptr(), self._ws.data_ptr(), self._ws.numel(), stream),
                    "boatagent_sac_gradients")
        elif not self.use_cuda_graph:
            self._dp_gradients_static()
        else:
            if self._graph is None:
                self._capture_dp()
            self._graph[0].replay()
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)   # eager, between the graphs (NCCL and gloo)
        if self.learner_precision == "fp32" and self.use_cuda_graph:
            self._graph[1].replay()
        else:
            o.step(grads)

    def _capture_dp(self):
        """Capture the data-parallel update as two graphs around the all-reduce: A = forward and backward passes into
        the flat buffer, B = DeviceAdam's step.  A writes nothing but the buffer, so its warm-up runs need no undo."""
        cur = torch.cuda.current_stream(self.device)
        side = torch.cuda.Stream(self.device)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(3):
                self._dp_gradients_static()
        cur.wait_stream(side)
        ga, gb = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
        with torch.cuda.graph(ga, stream=self.capture_stream):
            self._dp_gradients_static()
        with torch.cuda.graph(gb, stream=self.capture_stream):
            self.learner.optimizer.step(self._dp[2])
        self._graph = (ga, gb)

    def _run_update(self):
        if self._dp is not None:
            self._dp_update()
        elif self.learner_precision == "tcgen05":
            self._fused_update()
        elif not self.use_cuda_graph:
            self._losses = self._update_static()
        else:
            if self._graph is None:
                self._capture()
            self._graph.replay()
        self.updates += 1
        if self._tc_policy is not None:
            self._tc_policy.refresh()   # the packed bf16 copy follows the actor
        return self._losses

    def learn(self):
        """continuous_agent.py:96-154.  Returns None before the memory holds one batch (like the
        reference); afterwards the three losses (value, actor, critic) as device tensors (no sync).
        Three launches: the sample-gather kernel, the Gaussian draws, the captured update (learner_precision
        "tcgen05": the two kernels of the fused update)."""
        if self.memory.mem_cntr < self.batch_size:
            return None
        self.memory.sample_buffer(self.batch_size, as_torch=True, out=self._batch)
        self._eps.normal_()
        return self._run_update()

    def learn_from(self, state, action, reward, new_state, done, eps=None):
        """One update on a caller-supplied batch (device or host arrays of the batch size); `eps`
        [2, B, n_actions] prescribes the Gaussian draws (parity tests), else they are drawn here."""
        for dst, src in zip(self._batch, (state, action, reward, new_state, done)):
            dst.copy_(torch.as_tensor(src).reshape(dst.shape))
        if eps is None:
            self._eps.normal_()
        else:
            self._eps.copy_(torch.as_tensor(eps).reshape(self._eps.shape))
        return self._run_update()

    def _capture(self):
        """Capture one update into a CUDA graph.  Gradients and Adam's state must exist (as the tensors the
        graph will keep using) before capture, so three throw-away eager updates run first on a side
        stream; weights and optimiser state are then put back, i.e. every `learn()` -- the first one
        included -- is exactly one update."""
        L = self.learner
        params = [p for net in L.networks() for p in net.parameters()]
        opt_state = L.optimizer.state_tensors()   # Adam moments + step counter (fresh or carried over from eager updates)
        saved_params = [p.detach().clone() for p in params]
        saved_state = [t.clone() for t in opt_state]
        cur = torch.cuda.current_stream(self.device)
        side = torch.cuda.Stream(self.device)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(3):
                self._update_static()
            with torch.no_grad():
                torch._foreach_copy_(params, saved_params)
                torch._foreach_copy_(opt_state, saved_state)
        cur.wait_stream(side)
        self._graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph, stream=self.capture_stream):  # kernel nodes keep the capture stream's priority
            self._losses = self._update_static()

    def update_network_parameters(self, tau=None):
        self.learner.update_network_parameters(tau)

    def save_models(self):
        """base_network.py:13-14 for the five networks (weights only, the reference's checkpoint format)."""
        for net in self.learner.networks():
            net.save_checkpoint()

    def load_models(self):
        """base_network.py:16-17; the derived acting copies (the packed bf16 blob of the tcgen05 policy) follow."""
        for net in self.learner.networks():
            net.load_checkpoint()
        self._weights_changed()

    # -- population-based training hooks (population.py) -------------------------------------------------------
    def hyperparameters(self):
        """The four keys the reference's tuner draws (utils/hyperparameter_tuner.py:9-52)."""
        o = self.learner.optimizer
        n_actor = len(self.learner._actor_params)
        return {"alpha": float(o._slots[0].lr), "beta": float(o._slots[n_actor].lr), "gamma": float(self.learner.gamma),
                "tau": float(self.learner.tau)}

    def set_hyperparameters(self, alpha=None, beta=None, gamma=None, tau=None):
        """New learning rates / discount / target smoothing for the following updates.  The captured update graph
        holds the old values as kernel arguments, so it is dropped and re-captured by the next learn()."""
        L, o = self.learner, self.learner.optimizer
        n_actor = len(L._actor_params)
        for k in range(len(o.params)):
            if k < n_actor and alpha is not None:
                o._slots[k].lr = float(alpha)
            if k >= n_actor and beta is not None:
                o._slots[k].lr = float(beta)
        if gamma is not None:
            L.gamma = self.gamma = float(gamma)
        if tau is not None:
            L.tau = o.tau = self.tau = float(tau)
        self._graph = None

    def training_tensors(self):
        """Weights of the five networks + Adam moments and step counter: what a population member hands over."""
        L = self.learner
        tensors = [p.data for net in L.networks() for p in net.parameters()] + L.optimizer.state_tensors()
        return DataParallelState(tensors) if self._dp is not None else tensors

    def _weights_changed(self):
        if self._tc_policy is not None:
            self._tc_policy.refresh()
        for hook in self._weight_listeners:
            hook()

    # -- full training-state checkpoint (SURVEY.md 8f rank 4) -------------------------------------------------------
    def state_dict(self):
        """Everything `learn()` depends on beyond the env: the five networks, the Adam moments and step counter
        (`DeviceAdam`), the replay ring with its store counter and its Philox sample counter, the update count.
        The reference saves weights only (base_network.py:13-17) and loses the rest on restart."""
        L = self.learner
        return {"networks": {net.name: net.state_dict() for net in L.networks()},
                "optimizer": {k: ([t.clone() for t in v] if isinstance(v, list) else v.clone())
                              for k, v in L.optimizer.state_dict().items()},
                "memory": self.memory.state_dict(), "updates": self.updates,
                "rng": torch.cuda.get_rng_state(self.device)}

    def load_state_dict(self, sd):
        L = self.learner
        for net in L.networks():
            net.load_state_dict(sd["networks"][net.name])
        cur = L.optimizer.state_dict()
        with torch.no_grad():
            for k, v in sd["optimizer"].items():
                if isinstance(v, list):
                    torch._foreach_copy_(cur[k], [t.to(self.device) for t in v])
                else:
                    cur[k].copy_(v.to(self.device))
        self.memory.load_state_dict(sd["memory"])
        self.updates = int(sd["updates"])
        torch.cuda.set_rng_state(sd["rng"].cpu(), self.device)
        self._weights_changed()

    def save_training_state(self, path=None):
        """torch.save of `state_dict()` next to the reference-format checkpoints (<experiment_dir>/checkpoints/
        training_state.pt)."""
        import os
        path = path or os.path.join(self.actor.checkpoints_dir, "training_state.pt")
        torch.save(self.state_dict(), path)
        return path

    def load_training_state(self, path=None):
        import os
        path = path or os.path.join(self.actor.checkpoints_dir, "training_state.pt")
        self.load_state_dict(torch.load(path, map_location=self.device, weights_only=False))


class OverlappedActorLearner:
    """The loop of main.py:72-90 with acting and learning on two CUDA streams.

    Sequentially, one iteration is policy (0.44 ms for 65536 envs) -> fused step + remember -> sample ->
    update (0.84 ms), and the many small kernels of the update leave most of the GPU idle.  Here the env
    stream runs policy(t + 1) and step(t + 1) while the learner stream runs update(t):

        env stream     | policy(t)  step+store(t) | policy(t+1)  step+store(t+1) | ...
        learner stream |            ............. | sample(t)  update(t)  publish | sample(t+1) ...

    The policy reads one of two ACTING copies of the actor; update(t) publishes its weights into the copy
    that policy(t + 2) reads, so acting lags the learner by one update (the reference's strictly
    sequential loop is `ContinuousAgent.learn()` after every step; this class is the throughput mode).
    Events order everything that shares memory: the ring rows of step t are complete before sample(t);
    sample(t) has read the ring before step(t + 1) may overwrite its oldest rows; a copy is published
    only after the policy launch that read it has finished, and read only after it was published.

    The two streams are NON-BLOCKING: nothing the caller does on its own (default) stream is ordered against them.
    Call ``sync()`` before saving checkpoints, reading ``env.counters()`` or the losses, or loading weights; the
    next ``step()`` then waits for the caller's stream in turn.  ``finish()`` is ``sync()`` at the end of a run.
    """

    def __init__(self, agent: ContinuousAgent, env, done_flag_mode=1, recorder=None):
        if agent.data_parallel:
            raise ValueError("OverlappedActorLearner: a data-parallel agent is not supported")
        self.agent, self.env, self.done_flag_mode = agent, env, int(done_flag_mode)
        self.recorder = recorder   # a DeviceRecorder: captures every step on the env stream
        dev = agent.device
        # the learner's small kernels go first whenever an SM frees up: without a priority they queue behind
        # the thousand CTAs of each policy GEMM and the two streams do not overlap at all
        self.s_env, self.s_learn = torch.cuda.Stream(dev), torch.cuda.Stream(dev, priority=-1)
        if agent._graph is None:
            agent.capture_stream = torch.cuda.Stream(dev, priority=-1)
        self.acting = [copy.deepcopy(agent.actor).requires_grad_(False) for _ in range(2)]
        ev = lambda: torch.cuda.Event()  # noqa: E731
        self.ev_published, self.ev_policy = [ev(), ev()], [ev(), ev()]
        self.ev_store, self.ev_sample = ev(), ev()
        self._policy = [None, None]   # (graph, static action tensor) per acting copy
        self.t = 0
        self.losses = None
        self._rejoin = False
        agent._weight_listeners.append(self._republish)
        cur = torch.cuda.current_stream(dev)
        self.s_env.wait_stream(cur)
        self.s_learn.wait_stream(cur)

    @torch.no_grad()
    def _act(self, k):
        obs = self.env.obs
        prec = self.agent.policy_precision
        if prec == "tcgen05":
            if self._policy[k] is None:
                from .networks import TensorCorePolicy
                self._policy[k] = TensorCorePolicy(self.acting[k], seed=0x5ac + k)
                self._policy[k].steps = k   # the two copies draw from interleaved Philox counters
            pol = self._policy[k]
            pol.refresh()                   # acting[k] was just published into (stream-ordered after the copy)
            out = pol.act(obs)
            pol.steps += 1                  # act() advanced by one: keep the copies interleaved
            return out
        if not self.agent.use_cuda_graph:
            return self.acting[k].act(obs, prec)
        if self._policy[k] is None:
            for _ in range(2):
                self.acting[k].act(obs, prec)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                out = self.acting[k].act(obs, prec)
            self._policy[k] = (g, out)
        self._policy[k][0].replay()
        return self._policy[k][1]

    def step(self):
        """One env step over all envs and (once the memory holds a batch) one update."""
        a, k = self.agent, self.t & 1
        if self._rejoin:   # after sync(): whatever the caller did on its stream (checkpoint, counters) comes first
            cur = torch.cuda.current_stream(a.device)
            self.s_env.wait_stream(cur)
            self.s_learn.wait_stream(cur)
            self._rejoin = False
        with torch.cuda.stream(self.s_env):
            self.s_env.wait_event(self.ev_published[k])     # update(t - 2) has been written into acting[k]
            actions = self._act(k)
            self.ev_policy[k].record(self.s_env)
            self.s_env.wait_event(self.ev_sample)           # sample(t - 1) is done with the ring
            a.step_and_remember(self.env, actions.squeeze(-1), done_flag_mode=self.done_flag_mode)
            self.ev_store.record(self.s_env)
            if self.recorder is not None:
                self.recorder.capture(actions.squeeze(-1))
        with torch.cuda.stream(self.s_learn):
            self.s_learn.wait_event(self.ev_store)          # the rows of step t are complete
            if a.memory.mem_cntr >= a.batch_size:
                a.memory.sample_buffer(a.batch_size, as_torch=True, out=a._batch)
                self.ev_sample.record(self.s_learn)
                a._eps.normal_()
                self.losses = a._run_update()
                self.s_learn.wait_event(self.ev_policy[k])  # policy(t) has finished reading acting[k]
                with torch.no_grad():
                    torch._foreach_copy_(list(self.acting[k].parameters()), list(a.actor.parameters()))
                self.ev_published[k].record(self.s_learn)
        self.t += 1
        return self.losses

    def finish(self):
        """Joins both streams into the caller's stream."""
        self.sync()

    def sync(self):
        """Makes the caller's current stream wait for both pipeline streams, and the pipeline's next step wait for
        the caller's stream.  REQUIRED before anything outside the pipeline touches what it owns -- agent.save_models()
        / save_training_state(), env.counters(), reading the losses, agent.load_models(): the two streams are
        non-blocking, the default stream is not ordered against them (torch.save would otherwise copy weights while
        the fused Adam + Polyak kernel rewrites them)."""
        cur = torch.cuda.current_stream(self.agent.device)
        cur.wait_stream(self.s_env)
        cur.wait_stream(self.s_learn)
        self._rejoin = True

    def _republish(self):
        """The actor was replaced from outside (load_models): both acting copies follow."""
        with torch.no_grad():
            for c in self.acting:
                torch._foreach_copy_(list(c.parameters()), list(self.agent.actor.parameters()))
        for p in self._policy:
            if p is not None and hasattr(p, "refresh"):
                p.refresh()
