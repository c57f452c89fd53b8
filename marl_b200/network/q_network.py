"""Shared recurrent agent network: fc1 -> ReLU -> GRUCell -> fc2 on sm_100a kernels.

Drop-in for the reference's ``network/q_network.py:6-21`` (``RNNQNet``): same constructor,
same submodule / state_dict names (``fc1.*``, ``rnn.weight_ih|weight_hh|bias_ih|bias_hh``,
``fc2.*``), same default initialisation (so a given torch seed yields the same weights), same
``forward(obs, hidden_state) -> (q, h)``.  The arithmetic runs in libmarl_b200
(``marl_agent_unroll_fwd`` / ``_bwd``); there is no PyTorch or CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn

from .. import _lib as L
from ..flat import FlatBuffer, FlatPackedMixin

HIDDEN_WIDTHS = (32, 64, 128)     # rnn_hidden_dim values the recurrence and acting kernels are built for

AGENT_FLAT_ORDER = ("fc1.weight", "fc1.bias", "rnn.weight_ih", "rnn.weight_hh", "rnn.bias_ih", "rnn.bias_hh",
                    "fc2.weight", "fc2.bias")


def check_hidden(hidden):
    """rnn_hidden_dim as the kernels take it; ValueError for any width they are not built for."""
    if hidden not in HIDDEN_WIDTHS:
        raise ValueError(f"libmarl_b200 supports rnn_hidden_dim in {HIDDEN_WIDTHS}, got {hidden}")
    return int(hidden)


def agent_param_struct(named, cls=L.AgentParams, hidden=64):
    """named: dict name -> device address, in AGENT_FLAT_ORDER naming; hidden = rnn_hidden_dim (parameter structs only)."""
    s = cls()
    for field, name in zip(L.AGENT_KEYS, AGENT_FLAT_ORDER):
        setattr(s, field, named[name])
    if cls is L.AgentParams:
        s.hidden = hidden
    return s


class _UnrollFn(torch.autograd.Function):
    """Differentiable T-step unroll (used by the drop-in module surface; the fused learner
    calls the same C entry points directly and bypasses autograd).  `blocks`: None for the default [obs | last action |
    agent id] input (or a full input), else the (last_action, agent_id) input blocks (marl_unroll_stream.input_flags)."""

    @staticmethod
    def forward(ctx, obs, onehot, h0, shift, full_input, dims, blocks, *params):
        B, Lq, N, A, O = dims
        H = params[0].shape[0]                       # fc1.weight [H, I]
        dev = obs.device
        rows = B * Lq * N
        d = L.Dims(B, Lq, N, A, O, 0)
        f32 = dict(dtype=torch.float32, device=dev)
        q = torch.empty(B, Lq, N, A, **f32)
        hidden = torch.empty(B, Lq, N, H, **f32)
        h_last = torch.empty(B * N, H, **f32)
        x = torch.empty(rows, H, **f32)
        gi = torch.empty(rows, 3 * H, **f32)
        gates = torch.empty(rows, 4 * H, **f32)
        w_ih_t = torch.empty(H, 3 * H, **f32)        # W_ih^T, produced by the forward for the backward's data gradient
        st = L.UnrollStream()
        st.obs, st.onehot = obs.data_ptr(), (None if onehot is None else onehot.data_ptr())
        st.shift_onehot, st.full_input, st.h0_from = int(shift), int(full_input), -1
        st.h0 = None if h0 is None else h0.data_ptr()
        st.params = agent_param_struct({n: p.data_ptr() for n, p in zip(AGENT_FLAT_ORDER, params)}, hidden=H)
        st.q, st.hidden, st.h_last = q.data_ptr(), hidden.data_ptr(), h_last.data_ptr()
        st.x, st.gi, st.gates = x.data_ptr(), gi.data_ptr(), gates.data_ptr()
        st.w_ih_t = w_ih_t.data_ptr()
        if blocks is not None:
            st.input_flags, st.last_action, st.agent_id = 1, int(blocks[0]), int(blocks[1])
        L.call("marl_agent_unroll_fwd", C.byref(d), C.byref(st), 1, L.stream_ptr())
        ctx.save_for_backward(obs, onehot if onehot is not None else obs, h0 if h0 is not None else obs,
                              hidden, x, gates, w_ih_t, *params)
        ctx.meta = (dims, int(shift), int(full_input), onehot is None, h0 is not None, blocks)
        ctx.mark_non_differentiable(h_last)
        return q, hidden, h_last

    @staticmethod
    def backward(ctx, dq, dhidden, _dh_last):
        dims, shift, full_input, no_onehot, had_h0, blocks = ctx.meta
        obs, onehot, h0, hidden, x, gates, w_ih_t, *params = ctx.saved_tensors
        B, Lq, N, A, O = dims
        H = params[0].shape[0]
        dev = obs.device
        rows = B * Lq * N
        f32 = dict(dtype=torch.float32, device=dev)
        gflat = [torch.zeros_like(p) for p in params]
        a = L.UnrollBwd()
        a.obs, a.onehot = obs.data_ptr(), (None if no_onehot else onehot.data_ptr())
        a.shift_onehot, a.full_input = shift, full_input
        a.params = agent_param_struct({n: p.data_ptr() for n, p in zip(AGENT_FLAT_ORDER, params)}, hidden=H)
        a.hidden, a.x, a.gates = hidden.data_ptr(), x.data_ptr(), gates.data_ptr()
        a.w_ih_t = w_ih_t.data_ptr()
        if blocks is not None:
            a.input_flags, a.last_action, a.agent_id = 1, int(blocks[0]), int(blocks[1])
        dq = None if dq is None else dq.contiguous()
        dhidden = None if dhidden is None else dhidden.contiguous()
        a.dq, a.dhidden = L.ptr(dq), L.ptr(dhidden)
        ws = [torch.empty(rows, k, **f32) for k in (H, 3 * H, 3 * H, H)]
        a.dhext, a.dgi, a.dgh, a.dx = (w.data_ptr() for w in ws)
        dh0 = torch.empty(B * N, H, **f32) if had_h0 else None
        a.h0, a.dh0 = (h0.data_ptr() if had_h0 else None), L.ptr(dh0)
        a.grads = agent_param_struct({n: g.data_ptr() for n, g in zip(AGENT_FLAT_ORDER, gflat)}, L.AgentGrads)
        d = L.Dims(B, Lq, N, A, O, 0)
        L.call("marl_agent_unroll_bwd", C.byref(d), C.byref(a), L.stream_ptr())
        return (None, None, dh0, None, None, None, None, *gflat)


class RNNQNet(FlatPackedMixin, nn.Module):
    # Because all the agents share the same network, input_shape = obs_shape + n_actions + n_agents
    def __init__(self, input_shape, args):
        super().__init__()
        self.args = args
        H = self.hidden = check_hidden(args.rnn_hidden_dim)
        self.input_shape = input_shape
        self.fc1 = nn.Linear(input_shape, H)
        self.rnn = nn.GRUCell(H, H)
        self.fc2 = nn.Linear(H, args.n_actions)
        self._flat = None
        self._pack(torch.device("cuda") if torch.cuda.is_available() else torch.device("cpu"))

    # ---- flat storage -------------------------------------------------------------------------
    def flat_named_parameters(self):
        table = dict(self.named_parameters())
        return [(n, table[n]) for n in AGENT_FLAT_ORDER]

    def _pack(self, device):
        self._flat = FlatBuffer(self.flat_named_parameters(), device=device, with_grad=False)

    def adopt(self, flat: FlatBuffer):
        """Called by a learner after it re-packed these parameters into its own flat buffer."""
        self._flat = flat

    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        self._pack(self.fc1.weight.device)
        return out

    def param_struct(self):
        """marl_agent_params of this network's parameters."""
        return agent_param_struct(self.param_addresses(), hidden=self.hidden)

    def param_addresses(self):
        return {n: p.data_ptr() for n, p in self.flat_named_parameters()}

    # ---- reference surface ----------------------------------------------------------------------
    def forward(self, obs, hidden_state):
        """obs [R, input_shape] (already [obs | last_action | agent_id]); hidden_state [..., H]."""
        H = self.hidden
        obs = L.require_cuda(obs, "obs").to(torch.float32).contiguous()
        h_in = hidden_state.reshape(-1, H).to(torch.float32).contiguous()
        R = obs.shape[0]
        A = self.args.n_actions
        dims = (R, 1, 1, A, self.input_shape - A - 1)
        params = [p for _, p in self.flat_named_parameters()]
        q, hidden, _ = _UnrollFn.apply(obs, None, h_in, 0, 1, dims, None, *params)
        return q.view(R, A), hidden.view(R, H)

    def unroll_full(self, x, h0):
        """x [B, T, 1, input_shape] (already the full network input) -> q [B,T,1,A], hidden [B,T,1,H], h_last [B,H]."""
        B, T, _, I = x.shape
        A = self.args.n_actions
        dims = (B, T, 1, A, I - A - 1)                 # only O + A + N = input_shape matters for a full input
        params = [p for _, p in self.flat_named_parameters()]
        return _UnrollFn.apply(x, None, h0, 0, 1, dims, None, *params)

    def unroll(self, obs, onehot, h0, shift, last_action=True, agent_id=True):
        """[B,T,N,O], [B,T,N,A] -> q [B,T,N,A], hidden [B,T,N,H], h_last [B*N,H].  The input row is
        [obs | onehot (if last_action) | eye(N)[n] (if agent_id)]; onehot may be None without last_action."""
        B, T, N, O = obs.shape
        dims = (B, T, N, self.args.n_actions, O)
        params = [p for _, p in self.flat_named_parameters()]
        return _UnrollFn.apply(obs, onehot, h0, int(shift), 0, dims, (bool(last_action), bool(agent_id)), *params)
