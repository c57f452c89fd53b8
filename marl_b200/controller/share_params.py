"""Parameter-sharing multi-agent controller, drop-in for ``controller/share_params.py:8-182``.

Same surface as the reference's ``SharedMAC`` (``init_hidden``, ``get_current_q_values``,
``get_next_q_values``, ``choose_action``, ``parameters``, ``load_state``, ``save_models``,
``load_models``, ``cuda``) and the same stateful ``hidden_states`` semantics -- the hidden
state is carried between successive ``get_*_q_values`` calls until ``init_hidden`` -- but each
T-step unroll is ONE call into libmarl_b200 instead of a Python loop over timesteps, and the
input rows [obs | last_action | agent_id] (share_params.py:84-112; the last two blocks as args.last_action /
args.reuse_network select them) are never materialised.
"""
from __future__ import annotations

import ctypes as C
from typing import NamedTuple

import numpy as np
import torch as th

from .. import _lib as L
from ..network.q_network import RNNQNet, agent_param_struct


def _as_f32_cuda(x, device):
    if isinstance(x, np.ndarray):
        x = th.from_numpy(np.ascontiguousarray(x))
    if not th.is_tensor(x):
        x = th.as_tensor(x)
    return x.to(device=device, dtype=th.float32, non_blocking=True).contiguous()


class PhiloxDraws(NamedTuple):
    """Exploration drawn inside the act launch from Philox4x64-10 (include/marl_b200.h, marl_act_philox): agent n of
    instance e draws from key (seed, 0) and counter (episode_base + e, step, n, 0), so the draws depend on nothing but
    these numbers -- not on torch's or numpy's generator, nor on how the instances are split between calls or devices."""
    seed: int
    episode_base: int = 0
    step: int = 0


def _philox_struct(philox, eps_table):
    """The marl_act_philox descriptor of a PhiloxDraws and an optional device float64 epsilon table."""
    seed, base, step = (int(x) for x in philox)
    if not (0 <= seed < 1 << 64 and 0 <= base < 1 << 64 and 0 <= step < 1 << 31):
        raise ValueError(f"PhiloxDraws out of range: {philox}")
    if eps_table is not None and (eps_table.dtype != th.float64 or not eps_table.is_contiguous() or eps_table.dim() != 1):
        raise ValueError("eps_table must be a contiguous 1-D float64 device tensor")
    return L.ActPhilox(seed, base, step, L.ptr(eps_table), 0 if eps_table is None else eps_table.numel())


def _act(mac, fn, fn_philox, p, n, obs, last, avail, hidden, explore, random_action, explore_u, choice_u, eps, gate,
         actions, onehot, q, philox, eps_table):
    """The library call behind SharedMAC.act / SeparatedMAC.act: fn, or fn_philox when philox is given."""
    if actions is None:
        actions = th.empty(n, mac.n_agents, dtype=th.int64, device=mac.device)
    head = (n, mac.n_agents, mac.n_actions, mac.obs_shape, int(mac.args.last_action), int(mac.args.reuse_network), p,
            obs.data_ptr(), L.ptr(last), L.ptr(avail), hidden.data_ptr(), hidden.data_ptr())
    tail = (float(eps), L.ptr(gate), actions.data_ptr(), L.ptr(onehot), L.ptr(q), L.stream_ptr())
    if philox is None:
        if eps_table is not None:
            raise ValueError("eps_table belongs to the Philox form: pass philox= as well")
        L.call(fn, *head, L.ptr(explore), L.ptr(random_action), L.ptr(explore_u), L.ptr(choice_u), *tail)
    else:
        if any(x is not None for x in (explore, random_action, explore_u, choice_u)):
            raise ValueError("philox= replaces explore / random_action / explore_u / choice_u")
        L.call(fn_philox, *head, C.byref(_philox_struct(philox, eps_table)), *tail)
    return actions


def _input_shape(args):
    """Width of the agent's input [obs | last action if args.last_action | agent id if args.reuse_network]
    (share_params.py:114-123 and :497-506)."""
    return args.obs_shape + (args.n_actions if args.last_action else 0) + (args.n_agents if args.reuse_network else 0)


def _agent_row(args, obs, last_action, agent_num):
    """The reference's host-side input row of one agent for choose_action (share_params.py:40-48 and :421-429)."""
    inputs = np.asarray(obs, dtype=np.float64).copy()
    agent_id = np.zeros(args.n_agents)
    agent_id[agent_num] = 1.
    if args.last_action:
        inputs = np.hstack((inputs, last_action))
    if args.reuse_network:
        inputs = np.hstack((inputs, agent_id))
    return inputs


def _choose_actions(mac, obs, last_action, avail_actions, epsilon, evaluate, draws):
    """The body of ``SharedMAC.choose_actions`` / ``SeparatedMAC.choose_actions``: checks shapes, draws the exploration
    uniforms and calls ``mac.act`` on the carried hidden state.  ``last_action`` may be None when ``args.last_action``
    is False."""
    dev = mac.device
    if dev.type != "cuda":
        raise L.MarlLibraryError(f"{type(mac).__name__} needs a CUDA device: marl_b200 has no CPU path")
    N, A, O, H = mac.n_agents, mac.n_actions, mac.obs_shape, mac.args.rnn_hidden_dim
    obs = _as_f32_cuda(obs, dev)
    n = obs.shape[0]
    if last_action is None and mac.args.last_action:
        raise ValueError("last_action is required: the network reads the last action")
    last = None if last_action is None else _as_f32_cuda(last_action, dev)
    avail = None if avail_actions is None else _as_f32_cuda(avail_actions, dev)
    for name, t, want in (("obs", obs, (n, N, O)), ("last_action", last, (n, N, A)), ("avail_actions", avail, (n, N, A))):
        if t is not None and tuple(t.shape) != want:
            raise ValueError(f"{name} has shape {tuple(t.shape)}, expected {want}")
    h = mac.hidden_states
    if h is None or h.numel() != n * N * H:
        raise ValueError(f"hidden_states must hold {n} x {N} rows: call init_hidden({n}) first")
    work = h if (h.is_cuda and h.dtype == th.float32 and h.is_contiguous()) else h.to(dev, th.float32).contiguous()
    explore_u = choice_u = philox = None
    if not evaluate:
        if isinstance(draws, PhiloxDraws):
            philox = draws
        elif draws is None:
            explore_u = th.rand(n, N, dtype=th.float64, device=dev)
            choice_u = th.rand(n, N, dtype=th.float64, device=dev)
        else:
            explore_u, choice_u = (th.as_tensor(d, dtype=th.float64).to(dev).reshape(n, N).contiguous() for d in draws)
    with th.no_grad():
        actions = mac.act(n, obs, last, avail, work, explore_u=explore_u, choice_u=choice_u, eps=float(epsilon), philox=philox)
        if work is not h:
            h.copy_(work.view_as(h))
    return actions


class SharedMAC:
    """All agents share one RNNQNet; the agent id travels as a one-hot input."""

    def __init__(self, args):
        self.n_actions = args.n_actions
        self.n_agents = args.n_agents
        self.state_shape = args.state_shape
        self.obs_shape = args.obs_shape
        self.args = args
        self._build_agents(self._get_input_shape())
        self.hidden_states = None   # (n_episodes, n_agents, hidden_dim)

    # ---- construction -----------------------------------------------------------------------------
    def _get_input_shape(self):                   # share_params.py:114-123
        return _input_shape(self.args)

    def _blocks(self):
        return dict(last_action=bool(self.args.last_action), agent_id=bool(self.args.reuse_network))

    def _build_agents(self, input_shape):
        self.agent = RNNQNet(input_shape, self.args)

    @property
    def device(self):
        return self.agent.fc1.weight.device

    def cuda(self):
        self.agent.cuda()

    def parameters(self):
        return self.agent.parameters()

    def load_state(self, other_mac):
        self.agent.load_state_dict(other_mac.agent.state_dict())

    def save_models(self, path):
        th.save(self.agent.state_dict(), path)

    def load_models(self, path):
        self.agent.load_state_dict(th.load(path, map_location=self.device))

    # ---- hidden state -------------------------------------------------------------------------------
    def init_hidden(self, episode_num):
        self.hidden_states = th.zeros((episode_num, self.n_agents, self.args.rnn_hidden_dim), device=self.device)

    # ---- episode unrolls ------------------------------------------------------------------------------
    def _unroll(self, obs, onehot, max_episode_len, shift):
        dev = self.device
        if dev.type != "cuda":
            raise L.MarlLibraryError("SharedMAC needs a CUDA device: marl_b200 has no CPU path")
        obs = _as_f32_cuda(obs, dev)[:, :max_episode_len].contiguous()
        onehot = _as_f32_cuda(onehot, dev)[:, :max_episode_len].contiguous() if self.args.last_action else None
        h0 = self.hidden_states.reshape(-1, self.args.rnn_hidden_dim).to(dev).contiguous()
        q, hidden, h_last = self.agent.unroll(obs, onehot, h0, shift, **self._blocks())
        self.hidden_states = h_last            # [B*N, H], as left behind by the reference's loop
        return q, hidden

    def get_current_q_values(self, batch, max_episode_len):
        """Q-values of every transition's current observation (share_params.py:125-146):
        step t consumes [o_t | u_onehot_{t-1} (zeros at t=0) if last_action | agent id if reuse_network]."""
        return self._unroll(batch["o"], batch["u_onehot"], max_episode_len, shift=1)

    def get_next_q_values(self, batch, max_episode_len):
        """Q-values of every transition's next observation (share_params.py:148-168):
        step t consumes [o_next_t | u_onehot_t if last_action | agent id if reuse_network]."""
        return self._unroll(batch["o_next"], batch["u_onehot"], max_episode_len, shift=0)

    def forward(self, ep_batch, t):
        """pymarl-style alias named by the north star: Q-values of all agents at step t of the
        current-observation stream (one step of get_current_q_values), returns [B, N, A]."""
        sl = slice(max(t - 1, 0), t + 1)
        batch = {"o": ep_batch["o"][:, sl], "u_onehot": ep_batch["u_onehot"][:, sl]}
        if t == 0:
            q, _ = self._unroll(batch["o"], batch["u_onehot"], 1, shift=1)
            return q[:, 0]
        # step t needs u_onehot[t-1]: feed it unshifted alongside o_t
        dev = self.device
        obs = _as_f32_cuda(ep_batch["o"], dev)[:, t:t + 1].contiguous()
        oh = _as_f32_cuda(ep_batch["u_onehot"], dev)[:, t - 1:t].contiguous() if self.args.last_action else None
        h0 = self.hidden_states.reshape(-1, self.args.rnn_hidden_dim).to(dev).contiguous()
        q, _, h_last = self.agent.unroll(obs, oh, h0, 0, **self._blocks())
        self.hidden_states = h_last
        return q[:, 0]

    # ---- acting ---------------------------------------------------------------------------------------
    def choose_action(self, obs, last_action, agent_num, avail_actions, epsilon, evaluate=False):
        """Epsilon-greedy action of ONE agent (share_params.py:37-72); RNG order: one
        np.random.uniform(), then np.random.choice only when exploring."""
        inputs = _agent_row(self.args, obs, last_action, agent_num)
        avail_actions_ind = np.nonzero(avail_actions)[0]
        dev = self.device
        hidden_state = self.hidden_states[:, agent_num, :]
        inputs = th.tensor(inputs, dtype=th.float32).unsqueeze(0).to(dev)
        avail = th.tensor(np.asarray(avail_actions), dtype=th.float32).unsqueeze(0).to(dev)
        with th.no_grad():
            q_value, h = self.agent(inputs, hidden_state.to(dev))
            self.hidden_states[:, agent_num, :] = h
            q_value[avail == 0.0] = -float("inf")
        if np.random.uniform() < epsilon:
            action = np.random.choice(avail_actions_ind)
        else:
            action = th.argmax(q_value)
        return action

    def choose_actions(self, obs, last_action, avail_actions, epsilon, evaluate=False, draws=None):
        """Epsilon-greedy actions of every agent of every instance in ONE ``marl_agent_act_input`` launch: the batched
        counterpart of ``choose_action``.

        obs [n, N, O], last_action [n, N, A] (may be None when ``args.last_action`` is False), avail_actions [n, N, A] or
        None (all available); numpy arrays or tensors.
        Agent a of instance e explores iff explore_u[e, a] < epsilon and then takes the
        min(floor(choice_u[e, a] * cnt), cnt - 1)-th of its cnt available actions (action 0 when it has none);
        ``draws=(explore_u, choice_u)`` ([n, N] uniforms in [0, 1)) supplies them, None draws them on the device from
        torch's generator, and ``draws=PhiloxDraws(seed, episode_base, step)`` has the act launch draw them itself from
        Philox (instance e is episode episode_base + e; no draw buffer).  ``evaluate=True`` is greedy.  Advances ``self.hidden_states`` (n * N rows, e.g. after
        ``init_hidden(n)``) in place and keeps its shape.  Returns the int64 CUDA actions [n, N]; nothing waits for the GPU."""
        return _choose_actions(self, obs, last_action, avail_actions, epsilon, evaluate, draws)

    def act(self, n, obs, last, avail, hidden, explore=None, random_action=None, explore_u=None, choice_u=None, eps=0.0,
            gate=None, actions=None, onehot=None, q=None, philox=None, eps_table=None):
        """One ``marl_agent_act_input`` launch over n instances: contiguous device tensors, ``hidden`` [n * N, H] advanced
        in place, ``last`` may be None without a last-action input (include/marl_b200.h documents every argument).
        ``philox=PhiloxDraws(...)`` selects the Philox exploration form (``marl_agent_act_philox``) in place of the four
        exploration arrays, with ``eps_table`` (optional contiguous float64 device tensor) giving instance e the
        epsilon ``eps_table[min(e, len - 1)]`` instead of ``eps``.  Returns ``actions`` [n, N] int64."""
        p = C.byref(agent_param_struct(self.agent.param_addresses()))
        return _act(self, "marl_agent_act_input", "marl_agent_act_philox", p, n, obs, last, avail, hidden, explore,
                    random_action, explore_u, choice_u, eps, gate, actions, onehot, q, philox, eps_table)


class SeparatedMAC:
    """Every agent has its own RNNQNet, drop-in for ``controller/share_params.py:389-610`` (what ``runner.py:24-26``
    builds when ``reuse_network`` is False).

    Same surface and state semantics as the reference: ``agent`` is a LIST of networks, ``hidden_states`` is
    ``[episodes, n_agents, hidden]`` and is carried between successive ``get_*_q_values`` calls, the input of agent
    n at step t is ``[o_t[n] | u_onehot_{t-1}[n] (last_action) | eye(N)[n] (reuse_network)]`` (``:467-495``), and
    ``get_next_q_values`` returns the per-agent LIST of final hidden states as its second value like the reference
    does (``:590``).  Each agent's T-step unroll is one ``marl_agent_unroll_fwd`` call on its own [B, T, 1, I] input
    (N calls per unroll instead of N*T network forwards), differentiable through ``RNNQNet``'s autograd function.

    Two reference defects are NOT reproduced because they make the class unusable for training: ``load_state`` there
    calls ``other_mac.agent.state_dict()`` (an AttributeError on a list -> the first target sync raises), and its
    per-agent in-place ``hidden_states`` write-back breaks ``loss.backward()`` under current torch.  Here ``load_state``
    copies agent i to agent i (or one shared network into every agent), and the hidden state is re-assembled out of place.
    """

    def __init__(self, args):
        self.n_actions = args.n_actions
        self.n_agents = args.n_agents
        self.state_shape = args.state_shape
        self.obs_shape = args.obs_shape
        self.args = args
        self._build_agents(self._get_input_shape())
        self.hidden_states = None

    def _get_input_shape(self):                   # share_params.py:497-506
        return _input_shape(self.args)

    def _build_agents(self, input_shape):
        self.agent = [RNNQNet(input_shape, self.args) for _ in range(self.n_agents)]

    @property
    def device(self):
        return self.agent[0].fc1.weight.device

    def cuda(self):
        for a in self.agent:
            a.cuda()

    def parameters(self):
        params = []
        for a in self.agent:
            params += list(a.parameters())
        return params

    def load_state(self, other_mac):
        for i, a in enumerate(self.agent):
            src = other_mac.agent[i] if isinstance(other_mac.agent, (list, tuple)) else other_mac.agent
            a.load_state_dict(src.state_dict())

    def save_models(self, path):                  # share_params.py:603-605: every agent to the same path (the last one stays)
        for a in self.agent:
            th.save(a.state_dict(), path)

    def load_models(self, path):
        for a in self.agent:
            a.load_state_dict(th.load(path, map_location=self.device))

    def init_hidden(self, episode_num):
        self.hidden_states = th.zeros((episode_num, self.n_agents, self.args.rnn_hidden_dim), device=self.device)

    def _inputs(self, obs, onehot, L_, shift):
        """[B, L, N, I]: obs | last action (shifted by one step for the current-observation stream) | agent id."""
        dev = self.device
        obs = _as_f32_cuda(obs, dev)[:, :L_]
        parts = [obs]
        if self.args.last_action:
            oh = _as_f32_cuda(onehot, dev)[:, :L_]
            if shift:
                oh = th.cat([th.zeros_like(oh[:, :1]), oh[:, :-1]], dim=1)
            parts.append(oh)
        if self.args.reuse_network:
            B = obs.shape[0]
            parts.append(th.eye(self.n_agents, device=dev).view(1, 1, self.n_agents, self.n_agents).expand(B, L_, -1, -1))
        return th.cat(parts, dim=3)

    def _unroll(self, obs, onehot, max_episode_len, shift):
        if self.device.type != "cuda":
            raise L.MarlLibraryError("SeparatedMAC needs a CUDA device: marl_b200 has no CPU path")
        x = self._inputs(obs, onehot, max_episode_len, shift)
        B, L_, N, _ = x.shape
        h0 = self.hidden_states.reshape(B, N, -1).to(self.device)
        qs, hids, lasts = [], [], []
        for n, net in enumerate(self.agent):
            q, hid, h_last = net.unroll_full(x[:, :, n:n + 1].contiguous(), h0[:, n].contiguous())
            qs.append(q)
            hids.append(hid)
            lasts.append(h_last)
        self.hidden_states = th.stack(lasts, dim=1)                      # [B, N, H]
        return th.cat(qs, dim=2), th.cat(hids, dim=2), lasts

    def get_current_q_values(self, batch, max_episode_len):
        q, hid, _ = self._unroll(batch["o"], batch["u_onehot"], max_episode_len, shift=1)
        return q, hid

    def get_next_q_values(self, batch, max_episode_len):
        q, _, lasts = self._unroll(batch["o_next"], batch["u_onehot"], max_episode_len, shift=0)
        return q, lasts                                                  # the per-agent list, as share_params.py:590 returns

    def choose_action(self, obs, last_action, agent_num, avail_actions, epsilon, evaluate=False):
        """share_params.py:419-453 with the agent's own network; same RNG order as SharedMAC.choose_action."""
        inputs = _agent_row(self.args, obs, last_action, agent_num)
        avail_actions_ind = np.nonzero(avail_actions)[0]
        dev = self.device
        hidden_state = self.hidden_states[:, agent_num, :]
        inputs = th.tensor(inputs, dtype=th.float32).unsqueeze(0).to(dev)
        avail = th.tensor(np.asarray(avail_actions), dtype=th.float32).unsqueeze(0).to(dev)
        with th.no_grad():
            q_value, h = self.agent[agent_num](inputs, hidden_state.to(dev))
            self.hidden_states[:, agent_num, :] = h
            q_value[avail == 0.0] = -float("inf")
        if np.random.uniform() < epsilon:
            action = np.random.choice(avail_actions_ind)
        else:
            action = th.argmax(q_value)
        return action

    def choose_actions(self, obs, last_action, avail_actions, epsilon, evaluate=False, draws=None):
        """``SharedMAC.choose_actions`` with each agent's own network, in ONE ``marl_agent_act_separated`` launch: the
        batched counterpart of ``choose_action``.  Same arguments, exploration rule, hidden-state handling and result;
        ``last_action`` may be None when ``args.last_action`` is False."""
        return _choose_actions(self, obs, last_action, avail_actions, epsilon, evaluate, draws)

    def act(self, n, obs, last, avail, hidden, explore=None, random_action=None, explore_u=None, choice_u=None, eps=0.0,
            gate=None, actions=None, onehot=None, q=None, philox=None, eps_table=None):
        """``SharedMAC.act`` with each agent's own network: one ``marl_agent_act_separated`` launch over n instances
        (``marl_agent_act_separated_philox`` with ``philox=``), ``hidden`` [n * N, H] advanced in place, ``last`` may be
        None without a last-action input.  Returns ``actions`` [n, N] int64."""
        # rebuilt on every call: a learner's flat buffer or .cuda() re-packs the agents and moves their addresses
        p = (L.AgentParams * self.n_agents)(*(agent_param_struct(net.param_addresses()) for net in self.agent))
        return _act(self, "marl_agent_act_separated", "marl_agent_act_separated_philox", p, n, obs, last, avail, hidden,
                    explore, random_action, explore_u, choice_u, eps, gate, actions, onehot, q, philox, eps_table)
