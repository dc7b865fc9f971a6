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
`SAC2Learner` (`ContinuousAgent(algorithm="sac2")`) is SAC with twin target critics and a learned entropy temperature
instead of the reference's value networks.
"""
from __future__ import annotations

import copy
import ctypes as C
import math

import numpy as np
import torch
import torch.nn.functional as F

from .buffer import PrioritizedReplayBuffer, ReplayBuffer
from .networks import ActorNetwork, CriticNetwork, TemperatureNetwork, ValueNetwork


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


class FusedLearner:
    """The fused tcgen05 update (csrc/learner.cu) of 1 to 16 `ContinuousAgent`s with learner_precision "tcgen05", one
    batch size and one device: each agent's batch (`_batch`, `_eps`), networks, `DeviceAdam` and hyper-parameters, one
    member of every launch.  A launch writes each agent's batch gradients into its parameters' `.grad` tensors and its
    three losses into its `_loss_buf`, on the current stream (no sync):

      update()          one SAC update of every agent (boatagent_sac_update_members, two launches);
      gradients(scale)  scale times the gradients and losses only (boatagent_sac_gradients_members, two launches),
                        for an all-reduce before
      adam()            Adam + Polyak of every agent from its `.grad` tensors (boatagent_adam_polyak_members, one
                        launch).

    Agents of algorithm "sac2" (all or none) run boatagent_sac2_update_members (three launches) and have no split
    launches.  A prioritized agent (one member only) runs boatagent_sac[2]_update_prioritized_members: its `_weights`
    scale the critic loss rows and its `_td` receives the rows' TD errors.
    The learning rates are read from the agents' DeviceAdam slots and gamma, reward scale and tau from their learners at
    every launch, so `ContinuousAgent.set_hyperparameters` reaches the next one.  The other pointers (batch, draws,
    `.grad` tensors, losses) are taken at the first launch and must stay the same tensors after it."""

    @staticmethod
    def check(agent):
        """The agent the kernels are written for: 11 observations, one action, 256-wide hidden layers and a batch size
        that is a positive multiple of 128."""
        B, L = agent.batch_size, agent.learner
        if agent.input_dims != (11,) or agent.get_n_actions() != 1 or B <= 0 or B % 128:
            raise ValueError("learner_precision='tcgen05': the BoatEnv agent (11 observations, one action) and a "
                             f"batch size that is a positive multiple of 128 (got {agent.input_dims}, "
                             f"{agent.get_n_actions()} actions, batch {B})")
        if any(tuple(net.fc2.weight.shape) != (256, 256) for net in L.networks() if hasattr(net, "fc2")):
            raise ValueError("learner_precision='tcgen05': 256-wide hidden layers only")

    def __init__(self, agents):
        self.agents = list(agents)
        a0 = self.agents[0]
        if not 1 <= len(self.agents) <= 16 or any(a.batch_size != a0.batch_size or a.device != a0.device or
                                                  a.algorithm != a0.algorithm for a in self.agents):
            raise ValueError("FusedLearner: 1 to 16 agents (BOATAGENT_SAC_MAX_MEMBERS) of one batch size, device and "
                             "algorithm")
        for a in self.agents:
            self.check(a)
        o0 = a0.learner.optimizer
        self._lib, self._L, self.device, self.batch_size = o0._lib, o0._L, a0.device, a0.batch_size
        self.v2 = a0.algorithm == "sac2"   # boatagent_sac2_update_members (the update only)
        self.per = a0.prioritized          # boatagent_sac[2]_update_prioritized_members (the update only)
        if any(a.prioritized for a in self.agents) and len(self.agents) > 1:
            raise ValueError("FusedLearner: a prioritized agent is updated on its own, not as a population member")
        ws_bytes = (self._L.boatagent_sac2_update_workspace_bytes if self.v2 else
                    self._L.boatagent_sac_update_workspace_bytes)(self.batch_size)
        self.ws = torch.empty(len(self.agents) * int(ws_bytes), dtype=torch.uint8, device=self.device)
        self._table = None

    def _launch(self, name, *args):
        if self._table is None:   # on the first launch: like the fp32 learner, no .grad before the first update
            entry = {(False, False): self._lib.SacMember, (True, False): self._lib.Sac2Member,
                     (False, True): self._lib.SacPrioritizedMember, (True, True): self._lib.Sac2PrioritizedMember}
            self._table = (entry[self.v2, self.per] * len(self.agents))()
            for m, a in enumerate(self.agents):
                o = a.learner.optimizer
                for k, p in enumerate(o.params):   # the batch gradient goes where the fp32 learner leaves it
                    if p.grad is None:
                        p.grad = torch.zeros_like(p)
                    o._slots[k].grad = p.grad.data_ptr()
                s, act, r, s2, d = a._batch
                e = self._lib.SacMember(
                    s.data_ptr(), act.data_ptr(), r.data_ptr(), s2.data_ptr(), d.data_ptr(), a._eps.data_ptr(),
                    a.learner.actor.max_action.data_ptr(), C.cast(o._slots, C.c_void_p), len(o.params), 0.0, 0.0, 0.0,
                    o.state.data_ptr(), a._loss_buf.data_ptr())
                e = self._lib.Sac2Member(e, 0.0) if self.v2 else e
                if self.per:
                    e = (self._lib.Sac2PrioritizedMember if self.v2 else self._lib.SacPrioritizedMember)(
                        e, a._weights.data_ptr(), a._td.data_ptr())
                self._table[m] = e
        for e, a in zip(self._table, self.agents):
            L = a.learner
            e2 = e.base if self.per else e   # the (v1 or v2) member entry
            b = e2.base if self.v2 else e2
            b.gamma, b.reward_scale, b.tau = float(L.gamma), float(L.scale), float(L.optimizer.tau)
            if self.v2:
                e2.target_entropy = float(L.target_entropy)
        with torch.cuda.device(self.device):   # the ABI launches on the current device
            stream = torch.cuda.current_stream().cuda_stream
            self._lib.check(getattr(self._L, name)(self._table, len(self.agents), *args, stream), name)

    def update(self):
        o = self.agents[0].learner.optimizer
        name = "boatagent_sac2_update" if self.v2 else "boatagent_sac_update"
        self._launch(name + ("_prioritized_members" if self.per else "_members"), self.batch_size,
                     o.betas[0], o.betas[1], o.eps, self.ws.data_ptr(), self.ws.numel())

    def gradients(self, scale):
        self._split_v1_only()
        self._launch("boatagent_sac_gradients_members", self.batch_size, scale, self.ws.data_ptr(), self.ws.numel())

    def adam(self):
        self._split_v1_only()
        o = self.agents[0].learner.optimizer
        self._launch("boatagent_adam_polyak_members", o.betas[0], o.betas[1], o.eps)

    def _split_v1_only(self):
        if self.v2 or self.per:
            raise ValueError("FusedLearner: the split gradients / Adam launches (data-parallel training) are for "
                             "SAC-v1 with uniform replay")


def point_grads_into(agent, row):
    """Makes the agent's `.grad` tensors (DeviceAdam's order) and its three losses (`_loss_buf`, `_losses`) views of
    `row`, a contiguous float32 tensor of n_params + 3 elements, so that one all-reduce of `row` averages them all."""
    off = 0
    for p in agent.learner.optimizer.params:
        p.grad = row[off:off + p.numel()].view_as(p)
        off += p.numel()
    agent._loss_buf = row[off:off + 3]
    agent._losses = tuple(agent._loss_buf[k] for k in range(3))


def _critic_loss(q1, q2, target, weights, td_out):
    """0.5 mse(q1, target) + 0.5 mse(q2, target); with importance weights (prioritized replay) the means are weighted,
    0.5 mean(w (q1 - target)^2) + 0.5 mean(w (q2 - target)^2), which equals the unweighted loss and its gradients bit
    for bit when every weight is 1 and the batch size is a power of two.  td_out receives the rows' TD errors."""
    if td_out is not None:
        with torch.no_grad():
            td_out.copy_(0.5 * ((q1 - target).abs() + (q2 - target).abs()))
    if weights is None:
        return 0.5 * F.mse_loss(q1, target) + 0.5 * F.mse_loss(q2, target)
    return 0.5 * torch.mean(weights * (q1 - target) ** 2) + 0.5 * torch.mean(weights * (q2 - target) ** 2)


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

    def update(self, state, action, reward, new_state, done, eps_sample=None, eps_rsample=None, weights=None,
               td_out=None):
        """One update on a batch (state [B, obs], action [B, n_actions], reward [B], new_state [B, obs],
        done [B] bool).  eps_*: optional standard-normal draws for the two `sample_normal` calls.
        weights [B] (prioritized replay): importance weights of the critic loss rows; td_out [B] receives the rows' TD
        errors 0.5 (|Q1 - q_hat| + |Q2 - q_hat|).
        Returns (value_loss, actor_loss, critic_loss) as 0-d tensors."""
        losses, grads_v, grads_a, grads_c = self._losses_and_grads(state, action, reward, new_state, done, eps_sample,
                                                                   eps_rsample, weights, td_out)
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

    def _losses_and_grads(self, state, action, reward, new_state, done, eps_sample, eps_rsample, weights=None,
                          td_out=None):
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
        critic_loss = _critic_loss(q1_old, q2_old, q_hat, weights, td_out)
        grads_c = torch.autograd.grad(critic_loss, self._critic_params)
        return (value_loss.detach(), actor_loss.detach(), critic_loss.detach()), grads_v, grads_a, grads_c


class SAC2Learner:
    """SAC with automatic entropy tuning (Haarnoja et al. 2018, "Soft Actor-Critic Algorithms and Applications"): the
    actor, two critics with Polyak target critics, no value network, and a temperature alpha = exp(log_alpha) learned
    towards `target_entropy` (default -n_actions).  Same interface as SACLearner; losses are (temperature, actor,
    critic).

    Every loss of one update reads the weights and alpha as they were before it; ONE Adam step over three learning rates
    (actor: alpha, critics: beta, log_alpha: temperature_lr, default beta) and the Polyak average of both target critics
    follow, as SACLearner argues for v1."""

    def __init__(self, input_dims, n_actions, max_action, alpha, beta, gamma, tau, reward_scale, experiment_dir=None,
                 device="cuda", torch_reference_math=False, target_entropy=None, init_temperature=1.0,
                 temperature_lr=None):
        self.device = torch.device(device)
        if self.device.type != "cuda" and not torch_reference_math:
            raise RuntimeError("SAC2Learner needs a CUDA device; pass torch_reference_math=True for the PyTorch "
                               "restatement of the update (parity tests only)")
        self.gamma, self.tau, self.scale = float(gamma), float(tau), float(reward_scale)
        self.target_entropy = float(-n_actions if target_entropy is None else target_entropy)
        temperature_lr = beta if temperature_lr is None else temperature_lr
        d = tuple(input_dims)
        # a fixed creation order: identical torch seeds give identical weights
        self.actor = ActorNetwork(experiment_dir, d, max_action, n_actions=n_actions, name="actor_network")
        self.critic_1 = CriticNetwork(experiment_dir, d, n_actions, name="critic_network_1")
        self.critic_2 = CriticNetwork(experiment_dir, d, n_actions, name="critic_network_2")
        self.target_critic_1 = CriticNetwork(experiment_dir, d, n_actions, name="target_critic_network_1")
        self.target_critic_2 = CriticNetwork(experiment_dir, d, n_actions, name="target_critic_network_2")
        self.temperature = TemperatureNetwork(experiment_dir, init_temperature)
        for net in self.networks():
            net.to(self.device)
        self._actor_params = list(self.actor.parameters())
        self._critic_params = list(self.critic_1.parameters()) + list(self.critic_2.parameters())
        self._temperature_params = [self.temperature.log_alpha]
        self._target_params = list(self.target_critic_1.parameters()) + list(self.target_critic_2.parameters())
        groups = [(self._actor_params, alpha), (self._critic_params, beta), (self._temperature_params, temperature_lr)]
        if self.device.type == "cuda":
            self.optimizer = DeviceAdam(groups, polyak=list(zip(self._critic_params, self._target_params)), tau=self.tau)
        else:
            self.optimizer = torch.optim.Adam([{"params": ps, "lr": lr} for ps, lr in groups])
        for p in self._target_params:
            p.requires_grad_(False)
        self.update_network_parameters(tau=1.0)

    def networks(self):
        return (self.actor, self.critic_1, self.critic_2, self.target_critic_1, self.target_critic_2, self.temperature)

    def alpha(self):
        """alpha = exp(log_alpha), a detached [1] tensor."""
        return self.temperature.log_alpha.detach().exp()

    @torch.no_grad()
    def update_network_parameters(self, tau=None):
        """target_critic_k = tau * critic_k + (1 - tau) * target_critic_k."""
        tau = self.tau if tau is None else float(tau)
        tgt, src = self._target_params, self._critic_params
        if tau == 1.0:
            torch._foreach_copy_(tgt, src)
            return
        torch._foreach_mul_(tgt, 1.0 - tau)
        torch._foreach_add_(tgt, src, alpha=tau)

    def update(self, state, action, reward, new_state, done, eps_sample=None, eps_rsample=None, weights=None,
               td_out=None):
        """One update on a batch (shapes as SACLearner.update; eps_sample draws a' on new_state, eps_rsample the
        reparameterised action on state; weights and td_out as SACLearner.update, with y in place of q_hat).
        Returns (temperature_loss, actor_loss, critic_loss) as 0-d tensors."""
        losses, grads = self._losses_and_grads(state, action, reward, new_state, done, eps_sample, eps_rsample,
                                               weights, td_out)
        for p, g in zip(self.optimizer_params(), grads):
            p.grad = g
        if isinstance(self.optimizer, DeviceAdam):   # Adam for the three groups + both Polyak averages, one launch
            self.optimizer.step(grads)
        else:
            self.optimizer.step()
            self.update_network_parameters()
        return losses

    def optimizer_params(self):
        """The trained tensors in DeviceAdam's order: actor 8, critic 1 6, critic 2 6, log_alpha 1."""
        return self._actor_params + self._critic_params + self._temperature_params

    def gradients(self, state, action, reward, new_state, done, eps_sample, eps_rsample, out, scale=1.0):
        """`update` without the optimiser step, as SACLearner.gradients (out: the 21 gradients, then the 3 losses)."""
        losses, grads = self._losses_and_grads(state, action, reward, new_state, done, eps_sample, eps_rsample)
        torch._foreach_copy_(out, list(grads) + list(losses))
        if scale != 1.0:
            torch._foreach_mul_(out, scale)

    def _losses_and_grads(self, state, action, reward, new_state, done, eps_sample, eps_rsample, weights=None,
                          td_out=None):
        """The three losses (detached) and the gradients of the trained tensors in DeviceAdam's order."""
        alpha = self.alpha()
        with torch.no_grad():
            a_next, lp_next = self.actor.sample_normal(new_state, reparameterize=False, eps=eps_sample)
            q_next = torch.min(self.target_critic_1(new_state, a_next), self.target_critic_2(new_state, a_next)).view(-1)
            v_next = q_next - alpha * lp_next.view(-1)
            y = self.scale * reward + self.gamma * torch.where(done, torch.zeros_like(v_next), v_next)

        actions, log_probs = self.actor.sample_normal(state, reparameterize=True, eps=eps_rsample)
        critic_value = torch.min(self.critic_1(state, actions), self.critic_2(state, actions)).view(-1)
        actor_loss = torch.mean(alpha * log_probs.view(-1) - critic_value)
        # only the actor's gradients: what this loss sends into the critics is discarded, as in v1
        grads_a = torch.autograd.grad(actor_loss, self._actor_params)

        entropy_gap = torch.mean(log_probs.detach().view(-1) + self.target_entropy)
        temperature_loss = -(self.temperature.log_alpha * entropy_gap).sum()
        grads_t = torch.autograd.grad(temperature_loss, self._temperature_params)

        q1 = self.critic_1(state, action).view(-1)
        q2 = self.critic_2(state, action).view(-1)
        critic_loss = _critic_loss(q1, q2, y, weights, td_out)
        grads_c = torch.autograd.grad(critic_loss, self._critic_params)
        losses = (temperature_loss.detach(), actor_loss.detach(), critic_loss.detach())
        return losses, tuple(grads_a) + tuple(grads_c) + tuple(grads_t)


class DataParallelState(list):
    """`training_tensors()` of a data-parallel agent: ONE agent's state, held equal by every rank of its group, so
    population rounds (population.exploit_explore) must not hand it between ranks."""


class ContinuousAgent:
    """agent/continuous_agent.py:9-154 on the GPU-resident env and replay ring.

    data_parallel: a torch.distributed process group (True: the default group) whose ranks train this one agent.  Each
    rank keeps its own env shard, ring, sampler seed and Gaussian draws; every update averages the ranks' gradients and
    losses with one all-reduce and applies the same Adam step everywhere, so the weights stay bit-identical without
    being re-broadcast.  Rank 0's weights and optimiser state are broadcast at construction.  Every rank must hold the
    same number of envs (`learn()` updates on all ranks or on none without a vote).

    prioritized: prioritized experience replay (Schaul et al. 2016).  The memory is a PrioritizedReplayBuffer (created
    here with priority_alpha and priority_eps unless one is passed in, whose own alpha and eps then apply); `learn()`
    draws its batch by priority, weights the critic loss rows by their importance weights and sets the drawn rows'
    priorities from their TD errors.  The weights' exponent beta rises linearly from priority_beta to 1 over
    priority_beta_updates updates (0: it stays priority_beta).  Works with both algorithms and both learner
    precisions; not with data_parallel, as an AgentPopulation member or under OverlappedActorLearner."""

    def __init__(self, config, experiment_dir, input_dims, env, device=None, seed=0, use_cuda_graph=True,
                 memory=None, policy_precision="fp32", learner_precision="fp32", data_parallel=None, algorithm="sac1",
                 target_entropy=None, init_temperature=1.0, temperature_lr=None, prioritized=False,
                 priority_alpha=0.6, priority_beta=0.4, priority_beta_updates=0, priority_eps=1e-6):
        if algorithm not in ("sac1", "sac2"):
            raise ValueError(f"algorithm: sac1 or sac2, got {algorithm!r}")
        if algorithm == "sac1" and (target_entropy is not None or init_temperature != 1.0 or temperature_lr is not None):
            raise ValueError("target_entropy, init_temperature and temperature_lr belong to algorithm='sac2'")
        if algorithm == "sac2" and data_parallel is not None and data_parallel is not False:
            raise ValueError("algorithm='sac2' does not train data-parallel")
        self.prioritized = bool(prioritized)
        if not self.prioritized:
            if (priority_alpha, priority_beta, priority_beta_updates, priority_eps) != (0.6, 0.4, 0, 1e-6):
                raise ValueError("priority_alpha, priority_beta, priority_beta_updates and priority_eps belong to "
                                 "prioritized=True")
            if isinstance(memory, PrioritizedReplayBuffer):
                raise ValueError("a PrioritizedReplayBuffer memory needs prioritized=True")
        else:
            if data_parallel is not None and data_parallel is not False:
                raise ValueError("prioritized=True does not train data-parallel")
            if not (priority_alpha >= 0 and priority_eps > 0 and 0 <= priority_beta <= 1 and priority_beta_updates >= 0):
                raise ValueError("prioritized: priority_alpha >= 0, 0 <= priority_beta <= 1, priority_beta_updates >= 0 "
                                 f"and priority_eps > 0 (got {priority_alpha}, {priority_beta}, {priority_beta_updates}, "
                                 f"{priority_eps})")
            if memory is not None and not isinstance(memory, PrioritizedReplayBuffer):
                raise ValueError("prioritized=True needs a PrioritizedReplayBuffer memory (or none: it is created)")
        self._beta = (float(priority_beta), int(priority_beta_updates))
        if not torch.cuda.is_available():
            raise RuntimeError("sac_agent_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.env = env
        self.config = config
        a = config.agent
        self.gamma, self.tau, self.scale = a.gamma, a.tvn_parameter_modulation_tau, a.reward_scale
        self.batch_size = int(a.batch_size)
        self.input_dims = tuple(input_dims)
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else int(device))
        if memory is not None:
            self.memory = memory
        elif self.prioritized:
            self.memory = PrioritizedReplayBuffer(a.max_size, self.input_dims, self.get_n_actions(), precision="fp32",
                                                  device=self.device.index, seed=seed, as_torch=True,
                                                  alpha=priority_alpha, eps=priority_eps)
        else:
            self.memory = ReplayBuffer(a.max_size, self.input_dims, self.get_n_actions(), precision="fp32",
                                       device=self.device.index, seed=seed, as_torch=True)
        # algorithm "sac2": SAC2Learner (twin target critics, learned temperature) instead of the reference's SAC-v1
        self.algorithm = algorithm
        learner_args = (self.input_dims, self.get_n_actions(), self.get_max_actions(), a.learning_rate_alpha,
                        a.learning_rate_beta, a.gamma, a.tvn_parameter_modulation_tau, a.reward_scale)
        if algorithm == "sac2":
            self.learner = SAC2Learner(*learner_args, experiment_dir=experiment_dir, device=self.device,
                                       target_entropy=target_entropy, init_temperature=init_temperature,
                                       temperature_lr=temperature_lr)
        else:
            self.learner = SACLearner(*learner_args, experiment_dir=experiment_dir, device=self.device)
        L = self.learner
        self.actor, self.critic_1, self.critic_2 = L.actor, L.critic_1, L.critic_2
        if algorithm == "sac2":
            self.target_critic_1, self.target_critic_2 = L.target_critic_1, L.target_critic_2
        else:
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
        if self.prioritized:   # the drawn slots, their importance weights and the TD errors of one update
            self._idx = torch.zeros(B, dtype=torch.int64, device=self.device)
            self._weights = torch.ones(B, **kw)
            self._td = torch.zeros(B, **kw)
        self._graph = None
        self.capture_stream = None   # stream the update graph is captured on (None: torch's own capture stream)
        self._losses = None
        self._act_graphs = {}
        self.updates = 0
        self._fused = None   # this agent's one-member FusedLearner, created by its first update
        if learner_precision == "tcgen05":
            FusedLearner.check(self)
            self._loss_buf = torch.zeros(3, **kw)
            self._losses = tuple(self._loss_buf[k] for k in range(3))
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
        per = dict(weights=self._weights, td_out=self._td) if self.prioritized else {}
        return self.learner.update(s, a, r, s2, d.bool(), eps_sample=self._eps[0], eps_rsample=self._eps[1], **per)

    def _fused_learner(self):
        """This agent's one-member FusedLearner.  Created on first use, so that the members of an AgentPopulation,
        which the population's own FusedLearner updates, hold no workspace of their own."""
        if self._fused is None:
            self._fused = FusedLearner([self])
        return self._fused

    @property
    def _ws(self):
        """The workspace of this agent's one-member FusedLearner (boatagent_sac_update_workspace_bytes(batch) bytes)."""
        return self._fused_learner().ws

    def _fused_update(self):
        """One update in the two fused learner kernels on the current stream (no sync)."""
        self._fused_learner().update()
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
        flat = torch.zeros(sum(p.numel() for p in o.params) + 3, dtype=torch.float32, device=self.device)
        point_grads_into(self, flat)
        # grad_scale 1 / world: the SUM all-reduce is the mean (exact for power-of-two world sizes)
        self._dp = (group, flat, [p.grad for p in o.params], 1.0 / world)
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
        if self.learner_precision == "tcgen05":
            self._fused_learner().gradients(scale)
        elif not self.use_cuda_graph:
            self._dp_gradients_static()
        else:
            if self._graph is None:
                self._capture_dp()
            self._graph[0].replay()
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)   # eager, between the graphs (NCCL and gloo)
        if self.learner_precision == "tcgen05":
            self._fused.adam()
        elif self.use_cuda_graph:
            self._graph[1].replay()
        else:
            self.learner.optimizer.step(grads)

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
        if self.prioritized:   # draw by priority, update with the importance weights, re-prioritise from the TD errors
            self.memory.sample_buffer(self.batch_size, self.priority_beta(), out=self._batch, idx_out=self._idx,
                                      weight_out=self._weights)
            self._eps.normal_()
            losses = self._run_update()
            self.memory.update_priorities(self._idx, self._td)
            return losses
        self.memory.sample_buffer(self.batch_size, as_torch=True, out=self._batch)
        self._eps.normal_()
        return self._run_update()

    def priority_beta(self):
        """prioritized: the importance-weight exponent of the next learn(), priority_beta rising linearly to 1 over
        priority_beta_updates updates."""
        b0, n = self._beta
        return b0 if n <= 0 else b0 + (1.0 - b0) * min(1.0, self.updates / n)

    def learn_from(self, state, action, reward, new_state, done, eps=None):
        """One update on a caller-supplied batch (device or host arrays of the batch size); `eps`
        [2, B, n_actions] prescribes the Gaussian draws (parity tests), else they are drawn here."""
        for dst, src in zip(self._batch, (state, action, reward, new_state, done)):
            dst.copy_(torch.as_tensor(src).reshape(dst.shape))
        if eps is None:
            self._eps.normal_()
        else:
            self._eps.copy_(torch.as_tensor(eps).reshape(self._eps.shape))
        if self.prioritized:   # a caller's batch carries no priorities: unit weights, no re-prioritisation
            self._weights.fill_(1.0)
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

    def temperature(self):
        """algorithm "sac2": the entropy temperature alpha = exp(log_alpha) as a 0-d device tensor (no sync)."""
        if self.algorithm != "sac2":
            raise ValueError("temperature(): SAC-v1 has no learned temperature (algorithm='sac2' has)")
        return self.learner.alpha()[0]

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
        holds the old values as kernel arguments, so it is dropped and re-captured by the next learn().  beta is the
        critics' (and v1's value network's) learning rate; SAC-v2's temperature keeps its own."""
        L, o = self.learner, self.learner.optimizer
        n_actor = len(L._actor_params)
        n_beta = len(o.params) - n_actor - len(getattr(L, "_temperature_params", ()))
        for k in range(len(o.params)):
            if k < n_actor and alpha is not None:
                o._slots[k].lr = float(alpha)
            if n_actor <= k < n_actor + n_beta and beta is not None:
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
        if agent.prioritized:
            raise ValueError("OverlappedActorLearner: a prioritized agent is not supported")
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
