"""SAC-GRU on the marllb_b200 policy kernels -- API mirror of simulation-mode/problem-04-sac-gru/src.

  PolicyNetwork   networks.py:19-155    GRU -> fc1(ReLU) -> mean / log_std, tanh-Gaussian sample
  QNetwork        networks.py:158-245   GRU over [state, action] -> fc1 -> fc2 -> fc3
  ReplayBuffer    replay_buffer.py:13-102
  SAC_GRU_Agent   sac_agent.py:19-318   select_action / update_parameters / save / load

Reference behaviours kept on purpose (SURVEY App. C #5, #6): the stored *policy* hidden state is
reused as the critics' hidden state and for next_states; the tanh correction is
log(action_scale*(1-y^2)+1e-6).  Gaussian noise comes from torch's generator unless `eps` is
passed (parity tests pass the reference's draws).
"""
from __future__ import annotations

import contextlib
import random
from collections import deque
from pathlib import Path

import numpy as np
import torch

from . import ops
from .nn import Adam, FlatBucket, GRUCellSeq, Params, linear_backward, wgrad_on
from .qmix import _device


def _init_like_reference(gru, linears):
    for name, p in gru.named_parameters():                     # networks.py:69-80
        if 'weight' in name:
            torch.nn.init.orthogonal_(p)
        else:
            torch.nn.init.constant_(p, 0.0)
    for fc in linears:
        torch.nn.init.xavier_uniform_(fc.weight)
        torch.nn.init.constant_(fc.bias, 0.0)


class PolicyNetwork:
    """networks.py:19-155."""

    def __init__(self, state_dim, action_dim, hidden_dim=256, gru_dim=128, action_scale=1.0, action_bias=0.0,
                 log_std_min=-20, log_std_max=2, device=None):
        self.state_dim, self.action_dim, self.hidden_dim, self.gru_dim = state_dim, action_dim, hidden_dim, gru_dim
        self.action_scale, self.action_bias = float(action_scale), float(action_bias)
        self.log_std_min, self.log_std_max = float(log_std_min), float(log_std_max)
        self.device = _device(device)
        gru = torch.nn.GRU(state_dim, gru_dim, batch_first=True)
        fc1 = torch.nn.Linear(gru_dim, hidden_dim)
        fc_mean = torch.nn.Linear(hidden_dim, action_dim)
        fc_logstd = torch.nn.Linear(hidden_dim, action_dim)
        _init_like_reference(gru, [fc1, fc_mean, fc_logstd])
        self.P = Params(self.device)
        for name, p in gru.named_parameters():
            self.P.add("gru." + name, p)
        for n, fc in (("fc1", fc1), ("fc_mean", fc_mean), ("fc_logstd", fc_logstd)):
            self.P.add(n + ".weight", fc.weight)
            self.P.add(n + ".bias", fc.bias)
        self.gru = GRUCellSeq(self.P)

    def _heads(self, state, hidden, save):
        P = self.P.p
        x = state.to(self.device, torch.float32).reshape(-1, self.state_dim).contiguous()
        h0 = hidden.to(self.device, torch.float32).reshape(-1, self.gru_dim).contiguous()
        hs, tape = self.gru.forward_seq(x.unsqueeze(0), h0)
        h1 = hs[0]
        a1 = ops.linear(h1, P["fc1.weight"], P["fc1.bias"], ops.ACT_RELU)
        mean = ops.linear(a1, P["fc_mean.weight"], P["fc_mean.bias"])
        lsr = ops.linear(a1, P["fc_logstd.weight"], P["fc_logstd.bias"])
        if save:
            self._tape = (tape, h1, a1, mean, lsr)
        return mean, lsr, h1

    def forward(self, state, hidden):
        """-> (mean, log_std clamped to [log_std_min, log_std_max], hidden_new [1,B,gru]); networks.py:82-110."""
        mean, lsr, h1 = self._heads(state, hidden, save=False)
        return mean, lsr.clamp(self.log_std_min, self.log_std_max), h1.unsqueeze(0)

    def sample(self, state, hidden, eps=None, save=False):
        """networks.py:112-147 -> (action, log_prob [B,1], mean_action, hidden_new)."""
        mean, lsr, h1 = self._heads(state, hidden, save)
        if eps is None:
            eps = torch.randn(mean.shape, device=self.device, dtype=torch.float32)
        eps = eps.to(self.device, torch.float32).contiguous()
        action, logp, mean_action = ops.tanh_gaussian_forward(mean, lsr, eps, self.log_std_min, self.log_std_max,
                                                              self.action_scale, self.action_bias)
        if save:
            self._eps = eps
        return action, logp, mean_action, h1.unsqueeze(0)

    def backward(self, d_action, d_logp):
        """Gradients of a scalar loss w.r.t. the sampled action [B,A] and log_prob [B,1]."""
        tape, h1, a1, mean, lsr = self._tape
        d_mean, d_lsr = ops.tanh_gaussian_backward(mean, lsr, self._eps, d_action, d_logp, self.log_std_min,
                                                   self.log_std_max, self.action_scale)
        da1 = linear_backward(self.P, "fc_mean.weight", "fc_mean.bias", a1, d_mean)
        ops.axpby(1.0, linear_backward(self.P, "fc_logstd.weight", "fc_logstd.bias", a1, d_lsr), 1.0, da1)
        dh1 = linear_backward(self.P, "fc1.weight", "fc1.bias", h1, ops.relu_backward(a1, da1))
        self.gru.backward_seq(dh1.unsqueeze(0).contiguous(), tape)
        self._tape = None

    def init_hidden(self, batch_size=1):
        return torch.zeros(1, batch_size, self.gru_dim, device=self.device)

    def to(self, device):
        return self

    def state_dict(self):
        return self.P.state_dict()

    def load_state_dict(self, sd):
        self.P.load_state_dict(sd)

    def parameters(self):
        return self.P.tensors()


class QNetwork:
    """networks.py:158-245."""

    def __init__(self, state_dim, action_dim, hidden_dim=256, gru_dim=128, device=None):
        self.state_dim, self.action_dim, self.hidden_dim, self.gru_dim = state_dim, action_dim, hidden_dim, gru_dim
        self.device = _device(device)
        gru = torch.nn.GRU(state_dim + action_dim, gru_dim, batch_first=True)
        fc1 = torch.nn.Linear(gru_dim, hidden_dim)
        fc2 = torch.nn.Linear(hidden_dim, hidden_dim)
        fc3 = torch.nn.Linear(hidden_dim, 1)
        _init_like_reference(gru, [fc1, fc2, fc3])
        self.P = Params(self.device)
        for name, p in gru.named_parameters():
            self.P.add("gru." + name, p)
        for n, fc in (("fc1", fc1), ("fc2", fc2), ("fc3", fc3)):
            self.P.add(n + ".weight", fc.weight)
            self.P.add(n + ".bias", fc.bias)
        self.gru = GRUCellSeq(self.P)

    def forward(self, state, action, hidden, save=False):
        """-> (q [B,1], hidden_new [1,B,gru]); networks.py:209-237."""
        P = self.P.p
        s = state.to(self.device, torch.float32).reshape(-1, self.state_dim)
        a = action.to(self.device, torch.float32).reshape(-1, self.action_dim)
        sa = torch.cat([s, a], dim=1).contiguous()
        h0 = hidden.to(self.device, torch.float32).reshape(-1, self.gru_dim).contiguous()
        hs, tape = self.gru.forward_seq(sa.unsqueeze(0), h0)
        h1 = hs[0]
        a1 = ops.linear(h1, P["fc1.weight"], P["fc1.bias"], ops.ACT_RELU)
        a2 = ops.linear(a1, P["fc2.weight"], P["fc2.bias"], ops.ACT_RELU)
        q = ops.linear(a2, P["fc3.weight"], P["fc3.bias"])
        if save:
            self._tape = (tape, h1, a1, a2)
        return q, h1.unsqueeze(0)

    __call__ = forward

    def backward(self, dq, need_daction=False):
        tape, h1, a1, a2 = self._tape
        dq = dq.reshape(-1, 1).contiguous()
        da2 = ops.relu_backward(a2, linear_backward(self.P, "fc3.weight", "fc3.bias", a2, dq))
        da1 = ops.relu_backward(a1, linear_backward(self.P, "fc2.weight", "fc2.bias", a1, da2))
        dh1 = linear_backward(self.P, "fc1.weight", "fc1.bias", h1, da1)
        dxs, _ = self.gru.backward_seq(dh1.unsqueeze(0).contiguous(), tape, need_dx=need_daction)
        self._tape = None
        return dxs[0][:, self.state_dim:].contiguous() if need_daction else None

    def init_hidden(self, batch_size=1):
        return torch.zeros(1, batch_size, self.gru_dim, device=self.device)

    def to(self, device):
        return self

    def state_dict(self):
        return self.P.state_dict()

    def load_state_dict(self, sd):
        self.P.load_state_dict(sd)

    def parameters(self):
        return self.P.tensors()


def soft_update(source, target, tau):
    """networks.py:248-260: target = tau*source + (1-tau)*target.  One launch when both parameter sets live in flat
    buffers of the same layout (the agent's networks do), else one per tensor."""
    fs, ft = getattr(source.P, "_flat_p", None), getattr(target.P, "_flat_p", None)
    if fs is not None and ft is not None and fs.numel() == ft.numel():
        ops.axpby(tau, fs, 1.0 - tau, ft)
        return
    for ps, pt in zip(source.P.tensors(), target.P.tensors()):
        ops.axpby(tau, ps, 1.0 - tau, pt)


def hard_update(source, target):
    target.load_state_dict(source.state_dict())


class ReplayBuffer:
    """replay_buffer.py:13-102 (host-side storage, same sampling call on Python's `random`)."""

    def __init__(self, capacity=1_000_000, seed=None):
        self.capacity = capacity
        self.buffer = deque(maxlen=capacity)
        if seed is not None:
            random.seed(seed)
            np.random.seed(seed)

    def push(self, state, action, reward, next_state, done, hidden=None):
        conv = lambda x: x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else x
        self.buffer.append((conv(state), conv(action), reward, conv(next_state), done,
                            conv(hidden) if hidden is not None else None))

    def sample(self, batch_size, device='cpu'):
        batch = random.sample(self.buffer, batch_size)                                # replay_buffer.py:70
        states, actions, rewards, next_states, dones, hiddens = zip(*batch)
        f = lambda x: torch.as_tensor(np.array(x), dtype=torch.float32).to(device)
        out = [f(states), f(actions), f(rewards).unsqueeze(1), f(next_states), f(dones).unsqueeze(1)]
        if hiddens[0] is not None:
            h = np.array(hiddens)
            if h.ndim == 4:
                h = np.expand_dims(h.squeeze(axis=2).squeeze(axis=1), axis=0)
            elif h.ndim == 2:
                h = np.expand_dims(h, axis=0)
            out.append(torch.as_tensor(h, dtype=torch.float32).to(device))
        else:
            out.append(None)
        return tuple(out)

    def __len__(self):
        return len(self.buffer)

    def is_ready(self, batch_size):
        return len(self.buffer) >= batch_size


class PrioritizedReplayBuffer:
    """replay_buffer.py:105-221: proportional prioritised replay (host-side storage, the reference's own numpy
    sampling call, so the same numpy seed draws the same indices)."""

    def __init__(self, capacity=1_000_000, alpha=0.6, beta=0.4, beta_increment=0.001, epsilon=1e-6, seed=None):
        self.capacity, self.alpha, self.beta = capacity, alpha, beta
        self.beta_increment, self.epsilon = beta_increment, epsilon
        self.buffer = []
        self.priorities = np.zeros(capacity, dtype=np.float32)
        self.position = 0
        self.size = 0
        if seed is not None:
            random.seed(seed)
            np.random.seed(seed)

    def push(self, state, action, reward, next_state, done, hidden=None):
        conv = lambda x: x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else x
        max_priority = self.priorities[:self.size].max() if self.size > 0 else 1.0    # :158
        item = (conv(state), conv(action), reward, conv(next_state), done, conv(hidden) if hidden is not None else None)
        if len(self.buffer) < self.capacity:
            self.buffer.append(item)
        else:
            self.buffer[self.position] = item
        self.priorities[self.position] = max_priority
        self.position = (self.position + 1) % self.capacity
        self.size = min(self.size + 1, self.capacity)

    def sample(self, batch_size, device='cpu'):
        """-> (states, actions, rewards, next_states, dones, hiddens, weights, indices)        :170-208"""
        priorities = self.priorities[:self.size]
        probabilities = priorities ** self.alpha
        probabilities /= probabilities.sum()
        indices = np.random.choice(self.size, batch_size, p=probabilities)
        weights = (self.size * probabilities[indices]) ** (-self.beta)
        weights /= weights.max()
        self.beta = min(1.0, self.beta + self.beta_increment)
        states, actions, rewards, next_states, dones, hiddens = zip(*[self.buffer[i] for i in indices])
        f = lambda x: torch.as_tensor(np.array(x), dtype=torch.float32).to(device)
        hid = f(hiddens) if hiddens[0] is not None else None
        return (f(states), f(actions), f(rewards).unsqueeze(1), f(next_states), f(dones).unsqueeze(1), hid,
                f(weights).unsqueeze(1), indices)

    def update_priorities(self, indices, priorities):
        for idx, priority in zip(indices, priorities):
            self.priorities[idx] = priority + self.epsilon

    def __len__(self):
        return self.size

    def is_ready(self, batch_size):
        return self.size >= batch_size


class SAC_GRU_Agent:
    """sac_agent.py:19-318."""

    def __init__(self, state_dim, action_dim, hidden_dim=256, gru_dim=128, lr_policy=3e-4, lr_q=3e-4,
                 lr_alpha=3e-4, gamma=0.99, tau=0.005, alpha=0.2, auto_entropy_tuning=True, target_entropy=None,
                 buffer_size=1_000_000, batch_size=256, device=None):
        self.state_dim, self.action_dim = state_dim, action_dim
        self.gamma, self.tau, self.batch_size = gamma, tau, batch_size
        self.auto_entropy_tuning = auto_entropy_tuning
        self.device = _device(device)
        self.policy = PolicyNetwork(state_dim, action_dim, hidden_dim, gru_dim, device=self.device)
        self.q1 = QNetwork(state_dim, action_dim, hidden_dim, gru_dim, self.device)
        self.q2 = QNetwork(state_dim, action_dim, hidden_dim, gru_dim, self.device)
        self.q1_target = QNetwork(state_dim, action_dim, hidden_dim, gru_dim, self.device)
        self.q2_target = QNetwork(state_dim, action_dim, hidden_dim, gru_dim, self.device)
        hard_update(self.q1, self.q1_target)
        hard_update(self.q2, self.q2_target)
        self._target_buckets = [FlatBucket([self.q1_target.P]), FlatBucket([self.q2_target.P])]   # flat: one-launch soft update
        # four optimisers like the reference (sac_agent.py:93-106), each over one flat bucket that is
        # all-reduced once per step in the reference's step order (SURVEY 8e)
        self.policy_optimizer = Adam(FlatBucket([self.policy.P]), lr_policy)
        self.q1_optimizer = Adam(FlatBucket([self.q1.P]), lr_q)
        self.q2_optimizer = Adam(FlatBucket([self.q2.P]), lr_q)
        if auto_entropy_tuning:
            self.target_entropy = -action_dim if target_entropy is None else target_entropy   # sac_agent.py:99-102
            self.log_alpha = torch.zeros(1, dtype=torch.float32, device=self.device)
            self._log_alpha_grad = torch.zeros_like(self.log_alpha)
            self.alpha = ops.exp_scalar(self.log_alpha)
            ab = FlatBucket([], extra=[(self.log_alpha, self._log_alpha_grad)])
            self.log_alpha, self._log_alpha_grad = ab.params[0], ab.grads[0]
            self.alpha_optimizer = Adam(ab, lr_alpha)
        else:
            self.alpha = torch.tensor([alpha], dtype=torch.float32, device=self.device)
            self.target_entropy = None
        self.replay_buffer = ReplayBuffer(capacity=buffer_size)
        self._twin = None
        self.total_steps = 0
        self.training_stats = {'q1_loss': [], 'q2_loss': [], 'policy_loss': [], 'alpha_loss': [], 'alpha': []}

    def _twin_stream(self):
        return self._aux_stream(0)

    def _aux_stream(self, k):
        """Side streams of update_parameters: 0 = Q2's passes, 1 / 2 = parameter gradients of the pass on the caller's
        stream / on stream 0, 3 = the actor's forward for the new actions."""
        if self._twin is None:
            self._twin = [torch.cuda.Stream(device=self.device) for _ in range(4)]
        return self._twin[k]

    def select_action(self, state, hidden, evaluate=False, eps=None):
        """sac_agent.py:124-149 -> (action numpy [action_dim], hidden_new [1,1,gru])."""
        if isinstance(state, np.ndarray):
            state = torch.as_tensor(state, dtype=torch.float32).unsqueeze(0)
        if hidden is None:
            hidden = self.policy.init_hidden(1)
        action, _, mean_action, hidden_new = self.policy.sample(state, hidden, eps=eps)
        out = mean_action if evaluate else action
        return out.cpu().numpy()[0], hidden_new

    def select_action_batch(self, states, hiddens=None, evaluate=False, eps=None):
        """Batched rollout form: states [E, state_dim] CUDA -> (actions [E, action_dim], hiddens [1,E,gru])."""
        if hiddens is None:
            hiddens = self.policy.init_hidden(states.shape[0])
        action, _, mean_action, hidden_new = self.policy.sample(states, hiddens, eps=eps)
        return (mean_action if evaluate else action), hidden_new

    def update_parameters(self, updates=1, batch=None, eps_next=None, eps_new=None, sync_stats=True):
        """sac_agent.py:151-255.  `batch`, `eps_next`, `eps_new` may be supplied for parity tests.
        sync_stats=False keeps the losses on the device (no host synchronisation: the whole update can
        then be captured in a CUDA graph) and returns them as 0-d tensors."""
        if batch is None and not self.replay_buffer.is_ready(self.batch_size):
            return None
        losses = {'q1': 0, 'q2': 0, 'policy': 0, 'alpha': 0}
        for _ in range(updates):
            b = batch if batch is not None else self.replay_buffer.sample(self.batch_size, self.device)
            states, actions, rewards, next_states, dones, hiddens = [None if x is None else x.to(self.device) for x in b]
            B = states.shape[0]
            if hiddens is None:
                policy_hidden = self.policy.init_hidden(B)
                q_hidden = self.q1.init_hidden(B)
            else:
                policy_hidden = q_hidden = hiddens                                    # sac_agent.py:171-172
            # The twin critics are independent until their outputs meet (min(Q1', Q2') in the target, min(Q1, Q2) in the
            # actor loss): every Q2 pass is issued on a second stream (`fork` .. `join`), concurrently with the Q1 pass
            # on the caller's stream.  At batch 256 each network is a dependent chain of small kernels that leave most
            # of the 148 SMs idle, so the two chains overlap almost entirely; inside a CUDA graph they become parallel
            # branches.  Arithmetic and step order are unchanged (sac_agent.py:201-231: Q1 step, Q2 step, actor, alpha).
            # Only while the update is being captured: launched eagerly it is bound by Python launch overhead, and the
            # stream switches would only add to it.
            cur = torch.cuda.current_stream(self.device)
            twin = self._twin_stream() if torch.cuda.is_current_stream_capturing() else None

            def fork():
                if twin is not None:
                    twin.wait_stream(cur)

            def join():
                if twin is not None:
                    cur.wait_stream(twin)

            branch = (lambda: ops.side_branch(twin)) if twin is not None else contextlib.nullcontext
            wg1 = (lambda: wgrad_on(self._aux_stream(1), 2)) if twin is not None else contextlib.nullcontext
            wg2 = (lambda: wgrad_on(self._aux_stream(2), 3)) if twin is not None else contextlib.nullcontext
            # ---- critic targets (no gradient), :175-190
            next_actions, next_logp, _, _ = self.policy.sample(next_states, policy_hidden, eps=eps_next)
            # the actor's forward for the new actions (:211) depends on nothing the critic steps change: it runs on its
            # own stream from here (same draw order: next-state noise first) and is joined before the actor's critic passes
            pol = self._aux_stream(3) if twin is not None else None
            if pol is not None:
                pol.wait_stream(cur)
                with ops.side_branch(pol, 4):
                    new_actions, logp, _, _ = self.policy.sample(states, policy_hidden, eps=eps_new, save=True)
            fork()
            with branch():
                q2n, _ = self.q2_target.forward(next_states, next_actions, q_hidden)
            q1n, _ = self.q1_target.forward(next_states, next_actions, q_hidden)
            join()
            y = ops.sac_q_target(rewards.reshape(-1).contiguous(), dones.reshape(-1).contiguous(),
                                 q1n.reshape(-1), q2n.reshape(-1), next_logp.reshape(-1), self.alpha, self.gamma)
            # ---- critics, :193-207.  Under data parallelism each bucket's all-reduce starts on the communication stream
            # as soon as its backward pass is done and the optimiser step that consumes it is issued as late as the data
            # dependencies allow, so the collective overlaps the next network's forward / backward.
            fork()
            with branch():
                q_cur2, _ = self.q2.forward(states, actions, q_hidden, save=True)
                loss2, dq = ops.mse_loss(q_cur2.reshape(-1), y)
                self.q2.P.zero_grad()
                with wg2():
                    self.q2.backward(dq)
                self.q2_optimizer.reduce_async()
            q_cur1, _ = self.q1.forward(states, actions, q_hidden, save=True)
            loss1, dq = ops.mse_loss(q_cur1.reshape(-1), y)
            self.q1.P.zero_grad()
            with wg1():
                self.q1.backward(dq)
            self.q1_optimizer.reduce_async()
            join()
            q_losses = [loss1, loss2]
            self.q1_optimizer.step()
            # ---- actor, :210-220
            if pol is None:
                new_actions, logp, _, _ = self.policy.sample(states, policy_hidden, eps=eps_new, save=True)   # overlaps Q2's all-reduce
            else:
                cur.wait_stream(pol)
            self.q2_optimizer.step()
            fork()
            with branch():
                q2_new, _ = self.q2.forward(states, new_actions, q_hidden, save=True)
            q1_new, _ = self.q1.forward(states, new_actions, q_hidden, save=True)
            join()
            p_loss, d_logp, dq1, dq2 = ops.sac_policy_loss(logp.reshape(-1), q1_new.reshape(-1), q2_new.reshape(-1), self.alpha)
            fork()
            with branch():
                with wg2():
                    d_action2 = self.q2.backward(dq2, need_daction=True)
            with wg1():
                d_action = self.q1.backward(dq1, need_daction=True)
            join()
            ops.axpby(1.0, d_action2, 1.0, d_action)
            self.policy.P.zero_grad()
            with wg1():
                self.policy.backward(d_action, d_logp)
            self.policy_optimizer.reduce_async()
            # ---- temperature, :223-231 (its 4-byte gradient rides along; both overlap the soft updates below)
            a_loss = None
            if self.auto_entropy_tuning:
                a_loss, d_la = ops.sac_alpha_loss(logp.reshape(-1), self.log_alpha, float(self.target_entropy))
                self._log_alpha_grad.copy_(d_la)
                self.alpha_optimizer.reduce_async()
            # ---- targets, :234-235
            soft_update(self.q1, self.q1_target, self.tau)
            soft_update(self.q2, self.q2_target, self.tau)
            self.policy_optimizer.step()
            if self.auto_entropy_tuning:
                self.alpha_optimizer.step()
                # in place: a CUDA graph that holds this update reads alpha from the same address on every replay
                ops.exp_scalar(self.log_alpha, out=self.alpha)
            conv = (lambda t: float(t.item())) if sync_stats else (lambda t: t.reshape(()).detach())
            losses['q1'] = losses['q1'] + conv(q_losses[0])
            losses['q2'] = losses['q2'] + conv(q_losses[1])
            losses['policy'] = losses['policy'] + conv(p_loss)
            if a_loss is not None:
                losses['alpha'] = losses['alpha'] + conv(a_loss)
            self.total_steps += 1
            if twin is None:
                ops.reserve_workspace_slots(5)      # a later capture of this update finds its side streams' split-K workspaces
        for k in losses:
            losses[k] = losses[k] / updates
        if not sync_stats:
            return losses
        self.training_stats['q1_loss'].append(losses['q1'])
        self.training_stats['q2_loss'].append(losses['q2'])
        self.training_stats['policy_loss'].append(losses['policy'])
        self.training_stats['alpha_loss'].append(losses['alpha'])
        self.training_stats['alpha'].append(float(self.alpha.item()))
        return losses

    def save(self, filepath):
        """sac_agent.py:257-287 (same checkpoint keys)."""
        filepath = Path(filepath)
        filepath.parent.mkdir(parents=True, exist_ok=True)
        ck = {'policy_state_dict': self.policy.state_dict(), 'q1_state_dict': self.q1.state_dict(),
              'q2_state_dict': self.q2.state_dict(), 'q1_target_state_dict': self.q1_target.state_dict(),
              'q2_target_state_dict': self.q2_target.state_dict(),
              'policy_optimizer_state_dict': self.policy_optimizer.state_dict(),
              'q1_optimizer_state_dict': self.q1_optimizer.state_dict(),
              'q2_optimizer_state_dict': self.q2_optimizer.state_dict(), 'total_steps': self.total_steps,
              'config': {'state_dim': self.state_dim, 'action_dim': self.action_dim, 'gamma': self.gamma,
                         'tau': self.tau, 'auto_entropy_tuning': self.auto_entropy_tuning,
                         'target_entropy': self.target_entropy}}
        if self.auto_entropy_tuning:
            ck['log_alpha'] = self.log_alpha
            ck['alpha_optimizer_state_dict'] = self.alpha_optimizer.state_dict()
        torch.save(ck, filepath)
        print(f"Agent saved to {filepath}")

    def load(self, filepath):
        ck = torch.load(filepath, map_location=self.device)
        self.policy.load_state_dict(ck['policy_state_dict'])
        self.q1.load_state_dict(ck['q1_state_dict'])
        self.q2.load_state_dict(ck['q2_state_dict'])
        self.q1_target.load_state_dict(ck['q1_target_state_dict'])
        self.q2_target.load_state_dict(ck['q2_target_state_dict'])
        for name, opt in (('policy_optimizer_state_dict', self.policy_optimizer),
                          ('q1_optimizer_state_dict', self.q1_optimizer), ('q2_optimizer_state_dict', self.q2_optimizer)):
            if isinstance(ck.get(name), dict):
                opt.load_state_dict(ck[name])                     # torch.optim.Adam layout (sac_agent.py:300-302)
            else:
                import warnings
                warnings.warn(f"SAC checkpoint holds no {name}: Adam restarts from zero moments")
        if self.auto_entropy_tuning and 'log_alpha' in ck:
            self.log_alpha.copy_(ck['log_alpha'].detach().to(self.device))
            ops.exp_scalar(self.log_alpha, out=self.alpha)
            if isinstance(ck.get('alpha_optimizer_state_dict'), dict):
                self.alpha_optimizer.load_state_dict(ck['alpha_optimizer_state_dict'])
        self.total_steps = ck['total_steps']
        print(f"Agent loaded from {filepath}")

    def get_stats(self):
        return {'total_updates': self.total_steps, 'alpha': float(self.alpha.item()), 'training_stats': self.training_stats}
