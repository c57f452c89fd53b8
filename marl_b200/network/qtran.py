"""QTRAN-base joint networks on sm_100a kernels, drop-in for ``QtranQBase`` / ``QtranV``
(reference ``network/mixer.py:355-418``): same constructors, state_dict keys
(``hidden_action_encoding.{0,2}``, ``q.{0,2,4}`` / ``hidden_encoding.{0,2}``, ``v.{0,2,4}``) and forwards.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn

from .. import _lib as L
from ..flat import FlatBuffer, FlatPackedMixin

from .q_network import check_hidden


def net_struct(addrs, cls=L.QtranNetParams, hidden=64):
    """addrs: the 10 device addresses in parameter order (we1, be1, we2, be2, w0, b0, w2, b2, w4, b4); hidden =
    rnn_hidden_dim (parameter structs only)."""
    s = cls()
    for f, a in zip(L.QTRAN_FIELDS, addrs):
        setattr(s, f, a)
    if cls is L.QtranNetParams:
        s.hidden = hidden
    return s


def net_workspace(M, N, D, qh, device):
    f = lambda *shape: torch.empty(*shape, dtype=torch.float32, device=device)
    return dict(e1=f(M * N, D), es=f(M, D), enc=f(M, D), a1=f(M, qh), a2=f(M, qh))


def net_ws_struct(ws):
    s = L.QtranNetWs()
    s.e1, s.es, s.enc, s.a1, s.a2 = (ws[k].data_ptr() for k in ("e1", "es", "enc", "a1", "a2"))
    return s


class _JointNetFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, s, hidden, actions, meta, *params):
        M, N, S, A_enc, qh, H = meta
        ws = net_workspace(M, N, H + A_enc, qh, s.device)
        out = torch.empty(M, 1, dtype=torch.float32, device=s.device)
        p = net_struct([t.data_ptr() for t in params], hidden=H)
        wss = net_ws_struct(ws)
        L.call("marl_qtran_net_fwd", M, N, S, A_enc, qh, C.byref(p), s.data_ptr(), hidden.data_ptr(), L.ptr(actions),
               C.byref(wss), out.data_ptr(), L.stream_ptr())
        ctx.save_for_backward(s, hidden, actions if actions is not None else s, *params)
        ctx.meta, ctx.ws = meta, ws
        return out

    @staticmethod
    def backward(ctx, dout):
        M, N, S, A_enc, qh, H = ctx.meta
        s, hidden, actions, *params = ctx.saved_tensors
        dev = s.device
        grads = [torch.zeros_like(t) for t in params]
        dws = net_workspace(M, N, H + A_enc, qh, dev)
        dhidden = torch.empty(M * N, H, dtype=torch.float32, device=dev)
        p = net_struct([t.data_ptr() for t in params], hidden=H)
        g = net_struct([t.data_ptr() for t in grads], L.QtranNetGrads)
        wss, dwss = net_ws_struct(ctx.ws), net_ws_struct(dws)
        L.call("marl_qtran_net_bwd", M, N, S, A_enc, qh, C.byref(p), s.data_ptr(), hidden.data_ptr(),
               actions.data_ptr() if A_enc else None, C.byref(wss), dout.contiguous().data_ptr(), C.byref(dwss),
               dhidden.data_ptr(), 0, C.byref(g), L.stream_ptr())
        return (None, dhidden.view(hidden.shape), None, None, *grads)


class _JointNet(FlatPackedMixin, nn.Module):
    def _finish(self):
        self._flat = None
        self._pack(torch.device("cuda") if torch.cuda.is_available() else torch.device("cpu"))

    def flat_named_parameters(self):
        return list(self.named_parameters())

    def _pack(self, device):
        self._flat = FlatBuffer(self.flat_named_parameters(), device=device, with_grad=False)

    def adopt(self, flat):
        self._flat = flat

    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        self._pack(next(self.parameters()).device)
        return out

    def _run(self, state, hidden, actions):
        B, T, N, _ = hidden.shape
        a = self.args
        H = a.rnn_hidden_dim
        s = L.require_cuda(state, "state").reshape(B * T, -1).to(torch.float32).contiguous()
        h = L.require_cuda(hidden, "hidden").reshape(B * T * N, H).to(torch.float32).contiguous()
        act = None if actions is None else actions.reshape(B * T * N, -1).to(torch.float32).contiguous()
        meta = (B * T, N, a.state_shape, 0 if act is None else a.n_actions, a.qtran_hidden_dim, H)
        return _JointNetFn.apply(s, h, act, meta, *[p for _, p in self.named_parameters()])


class QtranQBase(_JointNet):
    """Joint action-value network Q(s, [h_i | a_i]) (mixer.py:355-388) -> [B*T, 1]."""

    def __init__(self, args):
        super().__init__()
        self.args = args
        check_hidden(args.rnn_hidden_dim)
        ae_input = args.rnn_hidden_dim + args.n_actions
        qh = args.qtran_hidden_dim
        self.hidden_action_encoding = nn.Sequential(nn.Linear(ae_input, ae_input), nn.ReLU(), nn.Linear(ae_input, ae_input))
        q_input = args.state_shape + args.n_actions + args.rnn_hidden_dim
        self.q = nn.Sequential(nn.Linear(q_input, qh), nn.ReLU(), nn.Linear(qh, qh), nn.ReLU(), nn.Linear(qh, 1))
        self._finish()

    def forward(self, state, hidden_states, actions):
        return self._run(state, hidden_states, actions)


class QtranV(_JointNet):
    """State-value network V(s, [h_i]) (mixer.py:392-418) -> [B*T, 1]."""

    def __init__(self, args):
        super().__init__()
        self.args = args
        hd, qh = check_hidden(args.rnn_hidden_dim), args.qtran_hidden_dim
        self.hidden_encoding = nn.Sequential(nn.Linear(hd, hd), nn.ReLU(), nn.Linear(hd, hd))
        self.v = nn.Sequential(nn.Linear(args.state_shape + hd, qh), nn.ReLU(), nn.Linear(qh, qh), nn.ReLU(), nn.Linear(qh, 1))
        self._finish()

    def forward(self, state, hidden):
        return self._run(state, hidden, None)
