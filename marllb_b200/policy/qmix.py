"""QMIX on the marllb_b200 policy kernels -- API mirror of simulation-mode/problem-05-qmix/src.

  AgentQNetwork      agent_network.py:13-95     GRU(obs->gru) -> fc1 -> fc2 -> fc3, ReLU between
  QMixingNetwork     mixing_network.py:15-117   hypernetworks, |.|, ELU mixing
  VDNMixingNetwork   mixing_network.py:154-184  sum
  EpisodeBuffer      episode_buffer.py:11-178   host-side episode store (unchanged semantics)
  QMIXAgent          qmix_agent.py:19-347       select_actions / store_episode / update / save / load

`strict_reference=True` (default) reproduces the reference's update bit-for-bit in structure,
including its gather quirk (SURVEY App. C #1): the per-agent Q tensors are concatenated on the
action axis and gathered with indices < action_dim, so every "chosen Q" comes from agent 0's
block.  `strict_reference=False` gathers each agent's own Q.
"""
from __future__ import annotations

import contextlib
import random
from collections import deque
from pathlib import Path

import numpy as np
import torch

from . import ops
from .nn import Adam, FlatBucket, GRUCellSeq, Params, linear_backward


def _device(device):
    if not torch.cuda.is_available():
        raise RuntimeError("marllb_b200 needs a CUDA device (there is no CPU fallback)")
    if device is None or str(device) == "cuda":
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device(device)


class AgentQNetwork:
    """agent_network.py:13-95."""

    def __init__(self, obs_dim, action_dim, hidden_dim=128, gru_dim=64, device=None):
        self.obs_dim, self.action_dim, self.hidden_dim, self.gru_dim = obs_dim, action_dim, hidden_dim, gru_dim
        self.device = _device(device)
        # same construction + init order as the reference (agent_network.py:41-61)
        gru = torch.nn.GRU(obs_dim, gru_dim, batch_first=True)
        fc1 = torch.nn.Linear(gru_dim, hidden_dim)
        fc2 = torch.nn.Linear(hidden_dim, hidden_dim)
        fc3 = torch.nn.Linear(hidden_dim, action_dim)
        for name, p in gru.named_parameters():
            (torch.nn.init.orthogonal_ if 'weight' in name else lambda t: torch.nn.init.constant_(t, 0.0))(p)
        for fc in (fc1, fc2, fc3):
            torch.nn.init.xavier_uniform_(fc.weight)
            torch.nn.init.constant_(fc.bias, 0.0)
        self.P = Params(self.device)
        for name, p in gru.named_parameters():
            self.P.add("gru." + name, p)
        for n, fc in (("fc1", fc1), ("fc2", fc2), ("fc3", fc3)):
            self.P.add(n + ".weight", fc.weight)
            self.P.add(n + ".bias", fc.bias)
        self.gru = GRUCellSeq(self.P)

    # -- reference API
    def forward(self, obs, hidden):
        """obs [B, obs_dim], hidden [1, B, gru] -> (q [B, action_dim], hidden_new [1, B, gru])."""
        P = self.P.p
        obs = obs.to(self.device, torch.float32)
        if not (obs.dim() == 2 and obs.shape[0] >= ops.TC_MIN_M and obs.stride(1) == 1):
            obs = obs.contiguous()      # large strided batches (one agent's rows of [E, A, obs]) go to TMA as they are
        h = hidden.to(self.device, torch.float32).reshape(-1, self.gru_dim).contiguous()
        h_new = self.gru.step(obs, h)
        x = ops.linear(h_new, P["fc1.weight"], P["fc1.bias"], ops.ACT_RELU)
        x = ops.linear(x, P["fc2.weight"], P["fc2.bias"], ops.ACT_RELU)
        q = ops.linear(x, P["fc3.weight"], P["fc3.bias"])
        return q, h_new.unsqueeze(0)

    __call__ = forward

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

    # -- training path: whole sequences, time-major
    def forward_seq(self, obs_tb, save=True):
        """obs_tb [T, B, obs_dim] -> q [T, B, action_dim] (zero initial hidden, qmix_agent.py:219)."""
        P = self.P.p
        T, B, _ = obs_tb.shape
        h0 = torch.zeros((B, self.gru_dim), dtype=torch.float32, device=self.device)
        hs, tape = self.gru.forward_seq(obs_tb, h0)
        hs2 = hs.reshape(T * B, self.gru_dim)
        a1 = ops.linear(hs2, P["fc1.weight"], P["fc1.bias"], ops.ACT_RELU)
        a2 = ops.linear(a1, P["fc2.weight"], P["fc2.bias"], ops.ACT_RELU)
        q = ops.linear(a2, P["fc3.weight"], P["fc3.bias"])
        self._tape = (tape, hs2, a1, a2) if save else None
        return q.reshape(T, B, self.action_dim)

    def backward_seq(self, dq_tb):
        tape, hs2, a1, a2 = self._tape
        T, B, K = dq_tb.shape
        dq = dq_tb.reshape(T * B, K).contiguous()
        da2 = ops.relu_backward(a2, linear_backward(self.P, "fc3.weight", "fc3.bias", a2, dq))
        da1 = ops.relu_backward(a1, linear_backward(self.P, "fc2.weight", "fc2.bias", a1, da2))
        dhs = linear_backward(self.P, "fc1.weight", "fc1.bias", hs2, da1)
        self.gru.backward_seq(dhs.reshape(T, B, self.gru_dim), tape)
        self._tape = None


class QMixingNetwork:
    """mixing_network.py:15-117."""

    _LAYERS = ["hyper_w1.0", "hyper_w1.2", "hyper_b1.0", "hyper_w2.0", "hyper_w2.2", "hyper_b2.0", "hyper_b2.2"]

    def __init__(self, num_agents, state_dim, mixing_embed_dim=32, hypernet_embed_dim=64, device=None):
        self.num_agents, self.state_dim = num_agents, state_dim
        self.mixing_embed_dim, self.hypernet_embed_dim = mixing_embed_dim, hypernet_embed_dim
        self.device = _device(device)
        A, S, E, Hh = num_agents, state_dim, mixing_embed_dim, hypernet_embed_dim
        shapes = [(S, Hh), (Hh, A * E), (S, E), (S, Hh), (Hh, E), (S, Hh), (Hh, 1)]   # construction order :51-76
        self.P = Params(self.device)
        for name, (i, o) in zip(self._LAYERS, shapes):
            lin = torch.nn.Linear(i, o)        # default nn.Linear init, like the reference
            self.P.add(name + ".weight", lin.weight)
            self.P.add(name + ".bias", lin.bias)

    def forward(self, agent_qs, state, save=False):
        """agent_qs [M, A], state [M, S] -> q_tot [M, 1]."""
        P = self.P.p
        q = agent_qs.to(self.device, torch.float32).reshape(-1, self.num_agents).contiguous()
        s = state.to(self.device, torch.float32).contiguous()
        h1 = ops.linear(s, P["hyper_w1.0.weight"], P["hyper_w1.0.bias"], ops.ACT_RELU)
        pre1 = ops.linear(h1, P["hyper_w1.2.weight"], P["hyper_w1.2.bias"])
        w1 = ops.abs_forward(pre1)                                                     # :92
        b1 = ops.linear(s, P["hyper_b1.0.weight"], P["hyper_b1.0.bias"])
        h2 = ops.linear(s, P["hyper_w2.0.weight"], P["hyper_w2.0.bias"], ops.ACT_RELU)
        pre2 = ops.linear(h2, P["hyper_w2.2.weight"], P["hyper_w2.2.bias"])
        w2 = ops.abs_forward(pre2)                                                     # :99
        h3 = ops.linear(s, P["hyper_b2.0.weight"], P["hyper_b2.0.bias"], ops.ACT_RELU)
        b2 = ops.linear(h3, P["hyper_b2.2.weight"], P["hyper_b2.2.bias"])
        q_tot, hidden = ops.mixer_forward(q, w1, b1, w2, b2.reshape(-1), save_hidden=save)
        if save:
            self._tape = (q, s, h1, pre1, w1, h2, pre2, w2, h3, hidden)
        return q_tot.reshape(-1, 1)

    __call__ = forward

    def backward(self, dq_tot):
        """dq_tot [M] -> d agent_qs [M, A]; accumulates hypernet gradients."""
        q, s, h1, pre1, w1, h2, pre2, w2, h3, hidden = self._tape
        dq, dw1, db1, dw2, db2 = ops.mixer_backward(dq_tot.reshape(-1).contiguous(), q, w1, w2, hidden)
        P = self.P
        dpre1 = ops.abs_backward(pre1, dw1)
        dh1 = ops.relu_backward(h1, linear_backward(P, "hyper_w1.2.weight", "hyper_w1.2.bias", h1, dpre1))
        linear_backward(P, "hyper_w1.0.weight", "hyper_w1.0.bias", s, dh1, need_dx=False)
        linear_backward(P, "hyper_b1.0.weight", "hyper_b1.0.bias", s, db1, need_dx=False)
        dpre2 = ops.abs_backward(pre2, dw2)
        dh2 = ops.relu_backward(h2, linear_backward(P, "hyper_w2.2.weight", "hyper_w2.2.bias", h2, dpre2))
        linear_backward(P, "hyper_w2.0.weight", "hyper_w2.0.bias", s, dh2, need_dx=False)
        dh3 = ops.relu_backward(h3, linear_backward(P, "hyper_b2.2.weight", "hyper_b2.2.bias", h3, db2))
        linear_backward(P, "hyper_b2.0.weight", "hyper_b2.0.bias", s, dh3, need_dx=False)
        self._tape = None
        return dq

    def get_monotonicity_info(self, agent_qs, state):
        """dQ_tot/dQ_i for every agent, [M, A] (mixing_network.py:119-151): the mixer's own backward pass with
        dq_tot = 1; the hypernet gradients it would accumulate are discarded."""
        saved = [g.clone() for g in self.P.grads()]
        q_tot = self.forward(agent_qs, state, save=True)
        dq = self.backward(torch.ones(q_tot.shape[0], dtype=torch.float32, device=self.device))
        for g, s0 in zip(self.P.grads(), saved):
            g.copy_(s0)
        return dq

    def to(self, device):
        return self

    def state_dict(self):
        return self.P.state_dict()

    def load_state_dict(self, sd):
        self.P.load_state_dict(sd)

    def parameters(self):
        return self.P.tensors()


class WeightedQMixingNetwork:
    """mixing_network.py:187-246 (WQMIX): Q_tot = sum_i w_i(s) Q_i with w = softmax(MLP(s)); forward returns
    (q_tot [M, 1], weights [M, A]) like the reference."""

    def __init__(self, num_agents, state_dim, hidden_dim=64, device=None):
        self.num_agents, self.state_dim, self.hidden_dim = num_agents, state_dim, hidden_dim
        self.device = _device(device)
        if num_agents > 64:
            raise ValueError("at most 64 agents (softmax kernel row length)")
        self.P = Params(self.device)
        for name, (i, o) in (("weight_network.0", (state_dim, hidden_dim)), ("weight_network.2", (hidden_dim, num_agents))):
            lin = torch.nn.Linear(i, o)
            self.P.add(name + ".weight", lin.weight)
            self.P.add(name + ".bias", lin.bias)

    def forward(self, agent_qs, state, save=False):
        P = self.P.p
        q = agent_qs.to(self.device, torch.float32).reshape(-1, self.num_agents).contiguous()
        s = state.to(self.device, torch.float32).contiguous()
        h = ops.linear(s, P["weight_network.0.weight"], P["weight_network.0.bias"], ops.ACT_RELU)
        w = ops.softmax_forward(ops.linear(h, P["weight_network.2.weight"], P["weight_network.2.bias"]))
        q_tot = ops.weighted_sum_forward(q, w)
        if save:
            self._tape = (q, s, h, w)
        return q_tot.reshape(-1, 1), w

    __call__ = forward

    def backward(self, dq_tot):
        """dq_tot [M] -> d agent_qs [M, A]; accumulates the weight network's gradients."""
        q, s, h, w = self._tape
        dq, dw = ops.weighted_sum_backward(dq_tot.reshape(-1).contiguous(), q, w)
        dlogits = ops.softmax_backward(w, dw)
        dh = ops.relu_backward(h, linear_backward(self.P, "weight_network.2.weight", "weight_network.2.bias", h, dlogits))
        linear_backward(self.P, "weight_network.0.weight", "weight_network.0.bias", s, dh, need_dx=False)
        self._tape = None
        return dq

    def to(self, device):
        return self

    def state_dict(self):
        return self.P.state_dict()

    def load_state_dict(self, sd):
        self.P.load_state_dict(sd)

    def parameters(self):
        return self.P.tensors()


class VDNMixingNetwork:
    """mixing_network.py:154-184: Q_tot = sum_i Q_i."""

    def __init__(self, num_agents, device=None):
        self.num_agents = num_agents
        self.device = _device(device)
        self.P = Params(self.device)

    def forward(self, agent_qs, state=None, save=False):
        q = agent_qs.to(self.device, torch.float32).reshape(-1, self.num_agents).contiguous()
        ones = torch.ones((1, self.num_agents), dtype=torch.float32, device=self.device)
        return ops.linear(q, ones)                    # [M,1] = q . 1

    __call__ = forward

    def backward(self, dq_tot):
        return dq_tot.reshape(-1, 1).expand(-1, self.num_agents).contiguous()

    def to(self, device):
        return self

    def state_dict(self):
        return {}

    def load_state_dict(self, sd):
        pass

    def parameters(self):
        return []


class EpisodeBuffer:
    """episode_buffer.py:11-178 (host-side storage; same sampling calls on Python's `random`)."""

    def __init__(self, capacity=5000, num_agents=4):
        self.capacity, self.num_agents = capacity, num_agents
        self.buffer = deque(maxlen=capacity)
        self.current_episode = None

    def start_episode(self):
        self.current_episode = {'observations': [], 'actions': [], 'rewards': [], 'states': [], 'dones': [], 'hiddens': []}

    def add_transition(self, observations, actions, rewards, state, done, hiddens=None):
        if self.current_episode is None:
            self.start_episode()
        ep = self.current_episode
        ep['observations'].append(observations)
        ep['actions'].append(actions)
        ep['rewards'].append(rewards)
        ep['states'].append(state)
        ep['dones'].append(done)
        if hiddens is not None:
            ep['hiddens'].append(hiddens)

    def end_episode(self):
        if self.current_episode is not None and len(self.current_episode['observations']) > 0:
            self.buffer.append(self.current_episode)
            self.current_episode = None

    def sample_batch(self, batch_size, max_seq_len=None):
        if len(self.buffer) < batch_size:
            return None
        episodes = random.sample(self.buffer, batch_size)                           # episode_buffer.py:104
        longest = max(len(ep['observations']) for ep in episodes)
        seq_len = longest if max_seq_len is None else min(max_seq_len, longest)
        obs_dim = len(episodes[0]['observations'][0][0])
        a0 = episodes[0]['actions'][0][0]
        action_dim = len(a0) if hasattr(a0, '__len__') else 1
        state_dim = len(episodes[0]['states'][0])
        A = self.num_agents
        batch = {'observations': np.zeros((batch_size, seq_len, A, obs_dim)),
                 'actions': np.zeros((batch_size, seq_len, A, action_dim)),
                 'rewards': np.zeros((batch_size, seq_len, A)),
                 'states': np.zeros((batch_size, seq_len, state_dim)),
                 'dones': np.zeros((batch_size, seq_len)),
                 'seq_lengths': np.zeros(batch_size, dtype=np.int32)}
        for i, ep in enumerate(episodes):
            L = min(len(ep['observations']), seq_len)
            batch['seq_lengths'][i] = L
            batch['observations'][i, :L] = np.asarray(ep['observations'][:L], dtype=np.float64).reshape(L, A, obs_dim)
            batch['actions'][i, :L] = np.asarray(ep['actions'][:L], dtype=np.float64).reshape(L, A, action_dim)
            batch['rewards'][i, :L] = np.asarray(ep['rewards'][:L], dtype=np.float64).reshape(L, A)
            batch['states'][i, :L] = np.asarray(ep['states'][:L], dtype=np.float64).reshape(L, state_dim)
            batch['dones'][i, :L] = np.asarray(ep['dones'][:L], dtype=np.float64)
        return batch

    def __len__(self):
        return len(self.buffer)

    def is_ready(self, batch_size):
        return len(self.buffer) >= batch_size

    def get_stats(self):
        if len(self.buffer) == 0:
            return {}
        lengths = [len(ep['observations']) for ep in self.buffer]
        returns = [sum(sum(r) for r in ep['rewards']) for ep in self.buffer]
        return {'num_episodes': len(self.buffer), 'avg_length': np.mean(lengths), 'max_length': np.max(lengths),
                'min_length': np.min(lengths), 'avg_return': np.mean(returns), 'max_return': np.max(returns),
                'min_return': np.min(returns)}


class QMIXAgent:
    """qmix_agent.py:19-347."""

    def __init__(self, num_agents, state_dim, obs_dim, action_dim, hidden_dim=128, gru_dim=64,
                 mixing_embed_dim=32, hypernet_embed_dim=64, lr=5e-4, gamma=0.99, target_update_interval=200,
                 buffer_capacity=5000, batch_size=32, max_seq_len=50, device=None, use_vdn=False,
                 strict_reference=True):
        self.num_agents, self.state_dim, self.obs_dim, self.action_dim = num_agents, state_dim, obs_dim, action_dim
        self.gamma, self.target_update_interval = gamma, target_update_interval
        self.batch_size, self.max_seq_len = batch_size, max_seq_len
        self.strict_reference = strict_reference
        self.device = _device(device)
        mk = lambda: AgentQNetwork(obs_dim, action_dim, hidden_dim, gru_dim, self.device)
        self.agent_networks = [mk() for _ in range(num_agents)]                        # qmix_agent.py:83-86
        self.agent_networks_target = []
        for i in range(num_agents):                                                    # :89-93
            t = mk()
            t.load_state_dict(self.agent_networks[i].state_dict())
            self.agent_networks_target.append(t)
        if use_vdn:
            self.mixer, self.mixer_target = VDNMixingNetwork(num_agents, self.device), VDNMixingNetwork(num_agents, self.device)
        else:
            self.mixer = QMixingNetwork(num_agents, state_dim, mixing_embed_dim, hypernet_embed_dim, self.device)
            self.mixer_target = QMixingNetwork(num_agents, state_dim, mixing_embed_dim, hypernet_embed_dim, self.device)
            self.mixer_target.load_state_dict(self.mixer.state_dict())
        # one optimiser over all agent nets + mixer (:108-113) = one flat bucket; gradient clipping
        # (:284) uses the global norm AFTER the data-parallel all-reduce
        self._bucket = FlatBucket([net.P for net in self.agent_networks + [self.mixer]])
        self._params, self._grads = self._bucket.params, self._bucket.grads
        self.optimizer = Adam(self._bucket, lr, max_grad_norm=10.0)
        self.episode_buffer = EpisodeBuffer(capacity=buffer_capacity, num_agents=num_agents)
        self.graph_updates = False      # True: replay the device part of update() as a CUDA graph
        self._graphs = {}
        self._aux = None
        self.total_updates = 0
        self.training_stats = {'loss': [], 'q_tot': [], 'target_q_tot': []}

    # ------------------------------------------------------------------ acting
    def select_actions(self, observations, hiddens=None, evaluate=False, epsilon=0.0):
        """qmix_agent.py:126-170 for ONE env: list of A observations -> (actions, new_hiddens, q_values).
        Exploration consumes numpy's global RNG in the reference's order (rand per agent, randint only
        when exploring); the comparison itself runs in the selection kernel."""
        actions, new_hiddens, q_values = [], [], []
        for a in range(self.num_agents):
            obs = torch.as_tensor(np.asarray(observations[a], dtype=np.float32)).unsqueeze(0)
            hidden = self.agent_networks[a].init_hidden(1) if (hiddens is None or hiddens[a] is None) else hiddens[a]
            q, new_hidden = self.agent_networks[a](obs, hidden)
            u = rnd = None
            if not evaluate:
                draw = np.random.rand()
                r = np.random.randint(0, self.action_dim) if draw < epsilon else 0
                u = torch.tensor([draw], dtype=torch.float32, device=self.device)
                rnd = torch.tensor([r], dtype=torch.int32, device=self.device)
            act, qsel = ops.egreedy_select(q, epsilon, u, rnd)
            actions.append(int(act.item()))
            new_hiddens.append(new_hidden)
            q_values.append(float(qsel.item()))
        return actions, new_hiddens, q_values

    def select_actions_batch(self, observations, hiddens=None, epsilon=0.0, u=None, rnd=None):
        """Batched form for vectorised envs: observations [E, A, obs_dim] (CUDA), hiddens [A, E, gru] or None,
        u [E, A] uniforms and rnd [E, A] int32 pre-drawn (None = greedy).
        Returns (actions int32 [E, A], new hiddens [A, E, gru], q_selected [E, A])."""
        E = observations.shape[0]
        acts, hs, qs = [], [], []
        for a in range(self.num_agents):
            obs = observations[:, a]
            h = self.agent_networks[a].init_hidden(E) if hiddens is None else hiddens[a].unsqueeze(0)
            q, hn = self.agent_networks[a](obs, h)
            ua = u[:, a].contiguous() if u is not None else None
            ra = rnd[:, a].contiguous() if rnd is not None else None
            act, qsel = ops.egreedy_select(q, epsilon, ua, ra)
            acts.append(act); hs.append(hn[0]); qs.append(qsel)
        return torch.stack(acts, 1), torch.stack(hs, 0), torch.stack(qs, 1)

    def store_episode(self, episode_data):
        self.episode_buffer.start_episode()
        for t in range(len(episode_data['observations'])):
            self.episode_buffer.add_transition(observations=episode_data['observations'][t],
                                               actions=episode_data['actions'][t], rewards=episode_data['rewards'][t],
                                               state=episode_data['states'][t], done=episode_data['dones'][t])
        self.episode_buffer.end_episode()

    # ------------------------------------------------------------------ learning
    def update(self, batch=None):
        """qmix_agent.py:192-307.  `batch` may be supplied (parity tests); default samples the buffer."""
        if batch is None:
            if not self.episode_buffer.is_ready(self.batch_size):
                return None
            batch = self.episode_buffer.sample_batch(self.batch_size, self.max_seq_len)
        dev, f32 = self.device, torch.float32
        obs = torch.as_tensor(batch['observations'], dtype=f32).to(dev)               # [B,T,A,obs]
        actions = torch.as_tensor(batch['actions']).to(dev).long()                    # [B,T,A,adim]
        rewards = torch.as_tensor(batch['rewards'], dtype=f32).to(dev)                # [B,T,A]
        states = torch.as_tensor(batch['states'], dtype=f32).to(dev)                  # [B,T,S]
        dones = torch.as_tensor(batch['dones'], dtype=f32).to(dev).contiguous()       # [B,T]
        seq_len = torch.as_tensor(np.asarray(batch['seq_lengths'], dtype=np.int32)).to(dev)
        key = (tuple(obs.shape), tuple(actions.shape), tuple(states.shape))
        if self.graph_updates:
            stats = self._update_graphed(key, obs, actions, rewards, states, dones, seq_len)
        else:
            stats = self._update_device(obs, actions, rewards, states, dones, seq_len)
        return self._finish_update(stats)

    @staticmethod
    def _dp_active():
        import torch.distributed as dist
        return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1

    def _update_graphed(self, key, *inputs):
        """Replay the whole device part of update() (~900 launches at C3 sizes) as one CUDA graph; one
        graph per batch shape, static input buffers.  Under data parallelism the NCCL all-reduce of the
        gradient bucket is captured with it (every rank replays its graph once per update, in lock-step)."""
        g = self._graphs.get(key)
        if g is None:
            static = [t.clone() for t in inputs]
            side = torch.cuda.Stream(device=self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            snap = self._snapshot()
            with torch.cuda.stream(side):
                self._update_device(*static)            # warm-up (allocations, lazy inits); undone below
            torch.cuda.current_stream(self.device).wait_stream(side)
            torch.cuda.synchronize(self.device)
            self._restore(snap)
            ops.reserve_workspace_slots(4)          # split-K workspaces of the side lanes (nothing can be allocated in a capture)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = self._update_device(*static)
            self._restore(snap)                          # capture does not execute, but keep the host mirrors honest
            g = self._graphs[key] = (graph, static, out)
        graph, static, out = g
        for dst, src in zip(static, inputs):
            dst.copy_(src)
        graph.replay()
        self.optimizer.t += 1
        return out

    def _snapshot(self):
        o = self.optimizer
        return (self._bucket.flat_p.clone(), o._m.clone(), o._v.clone(), o._t_dev.clone(), o.t)

    def _restore(self, snap):
        o = self.optimizer
        self._bucket.flat_p.copy_(snap[0]); o._m.copy_(snap[1]); o._v.copy_(snap[2]); o._t_dev.copy_(snap[3])
        o.t = snap[4]

    def _update_device(self, obs, actions, rewards, states, dones, seq_len):
        """Everything of update() that runs on the GPU: forward, TD loss, backward, optimiser step.
        No host synchronisation; returns the float64[3] stats tensor (loss, mean q_tot, mean target)."""
        dev, f32 = self.device, torch.float32
        B, T, A, _ = obs.shape
        K = self.action_dim
        obs_tb = obs.permute(2, 1, 0, 3).contiguous()                                 # [A,T,B,obs] time-major per agent
        # The 2A forward chains (online and target network of every agent) and the A backward chains are independent of
        # each other and each keeps only a handful of SMs busy (the GRU time loop of B = 32 episodes is 8 thread blocks):
        # while the update is being captured they go to separate streams ("lanes"), i.e. parallel branches of the graph.
        cur = torch.cuda.current_stream(dev)
        multi = torch.cuda.is_current_stream_capturing()
        if multi and self._aux is None:
            self._aux = [torch.cuda.Stream(device=dev) for _ in range(3)]
        lanes = [None] + self._aux if multi else [None]
        L = len(lanes)
        on = lambda i: ops.side_branch(lanes[i % L], i % L) if lanes[i % L] is not None else contextlib.nullcontext()

        def fork():
            for st in lanes[1:]:
                st.wait_stream(cur)

        def join():
            for st in lanes[1:]:
                cur.wait_stream(st)

        fork()
        # online Q for every agent and timestep (:215-229)
        qs = [None] * A
        for a in range(A):
            with on(a):
                qs[a] = self.agent_networks[a].forward_seq(obs_tb[a])                 # each [T,B,K]
        # target networks (:244-253), no gradient
        tmax = [None] * A
        for a in range(A):
            with on(A + a):
                tq = self.agent_networks_target[a].forward_seq(obs_tb[a], save=False)     # [T,B,K]
                m, _ = ops.row_max(tq.reshape(T * B, K))
                tmax[a] = m.reshape(T, B)
        join()
        q_all = torch.stack(qs, 0).permute(2, 1, 0, 3).contiguous()                   # [B,T,A,K]
        idx = actions[:, :, :, 0]                                                     # [B,T,A]
        if self.strict_reference:
            flat = q_all.reshape(B, T, A * K)
            chosen = flat.gather(2, idx)                                              # :231-234 (agent-0 block)
        else:
            chosen = q_all.gather(3, idx.unsqueeze(-1)).squeeze(-1)
        chosen = chosen.contiguous()
        states2 = states.reshape(B * T, -1).contiguous()
        q_tot = self.mixer.forward(chosen.reshape(B * T, A), states2, save=True).reshape(B, T).contiguous()
        # targets (:254-268)
        target_agent_qs = torch.stack(tmax, 0).permute(2, 1, 0).contiguous()          # [B,T,A]
        target_q_tot = self.mixer_target.forward(target_agent_qs.reshape(B * T, A), states2).reshape(B, T).contiguous()
        # reward sum over agents: a [B*T, A] x ones GEMM (rewards.sum(dim=2), :267)
        ones = torch.ones((1, A), dtype=f32, device=dev)
        rsum = ops.linear(rewards.reshape(B * T, A).contiguous(), ones).reshape(B, T).contiguous()
        targets, dq_tot, stats = ops.qmix_td_loss(q_tot, target_q_tot, rsum, dones, seq_len, self.gamma)
        # backward (:280-285)
        self._bucket.flat_g.zero_()
        dchosen = self.mixer.backward(dq_tot.reshape(B * T)).reshape(B, T, A)
        dq_all = torch.zeros((B, T, A * K) if self.strict_reference else (B, T, A, K), dtype=f32, device=dev)
        if self.strict_reference:
            dq_all.scatter_add_(2, idx, dchosen)
            dq_all = dq_all.reshape(B, T, A, K)
        else:
            dq_all.scatter_add_(3, idx.unsqueeze(-1), dchosen.unsqueeze(-1))
        dq_tb = dq_all.permute(2, 1, 0, 3).contiguous()                               # [A,T,B,K]
        fork()
        for a in range(A):
            with on(a):                        # the lane that holds this agent's tape
                self.agent_networks[a].backward_seq(dq_tb[a])
        join()
        self.optimizer.step()                                                         # all-reduce, clip 10 (:284), Adam
        return stats

    def _finish_update(self, stats):
        A = self.num_agents
        self.total_updates += 1
        if self.total_updates % self.target_update_interval == 0:                     # :288-294
            for i in range(A):
                self.agent_networks_target[i].load_state_dict(self.agent_networks[i].state_dict())
            self.mixer_target.load_state_dict(self.mixer.state_dict())
        s = stats.cpu().numpy()
        out = {'loss': float(s[0]), 'q_tot': float(s[1]), 'target_q_tot': float(s[2])}
        for k, v in out.items():
            self.training_stats[k].append(v)
        return out

    # ------------------------------------------------------------------ checkpoints (qmix_agent.py:309-337)
    def save(self, filepath):
        filepath = Path(filepath)
        filepath.parent.mkdir(parents=True, exist_ok=True)
        torch.save({'agent_networks': [n.state_dict() for n in self.agent_networks],
                    'mixer': self.mixer.state_dict(), 'optimizer': self.optimizer.state_dict(),
                    'total_updates': self.total_updates}, filepath)
        print(f"QMIX agent saved to {filepath}")

    def load(self, filepath):
        ck = torch.load(filepath, map_location=self.device)
        for i, sd in enumerate(ck['agent_networks']):
            self.agent_networks[i].load_state_dict(sd)
            self.agent_networks_target[i].load_state_dict(sd)
        self.mixer.load_state_dict(ck['mixer'])
        self.mixer_target.load_state_dict(ck['mixer'])
        if isinstance(ck.get('optimizer'), dict):
            self.optimizer.load_state_dict(ck['optimizer'])       # torch.optim.Adam layout (qmix_agent.py:331)
        else:
            import warnings
            warnings.warn("QMIX checkpoint holds no optimizer state: Adam restarts from zero moments")
        self.total_updates = ck['total_updates']
        print(f"QMIX agent loaded from {filepath}")

    def get_stats(self):
        return {'total_updates': self.total_updates, 'buffer_size': len(self.episode_buffer),
                'training_stats': self.training_stats}
