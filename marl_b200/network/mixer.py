"""Value-factorisation mixers on sm_100a kernels, drop-in for the reference's ``network/mixer.py``.

``VDNMixer`` (:9-16), ``QMixMixer`` (:21-80): same constructors, state_dict keys and forward
signatures.  The learner's fused train step calls the C entry points directly; the modules'
own ``forward`` wraps the same kernels in an autograd Function so they also work stand-alone.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn

from .. import _lib as L
from ..flat import FlatBuffer, FlatPackedMixin

MAX_EMBED = 128        # qmix_hidden_dim served by the mixing kernel (include/marl_b200.h: MARL_QMIX_MAX_EMBED)


def hy_cols(N, E):
    """Row pitch of the hyper-network outputs hy [M, C]: w1 (N E) | b1 | w2 | b2.0 (E each)."""
    return N * E + 3 * E


class VDNMixer(nn.Module):
    """Q_tot = sum_n Q_n (mixer.py:15-16)."""

    def __init__(self, args):
        super().__init__()
        self.args = args

    def forward(self, q_values, states=None):
        return torch.sum(q_values, dim=2, keepdim=True)

    def flat_named_parameters(self):
        return []


# flat layout: the four state-conditioned heads are contiguous so that one GEMM serves them all
QMIX_FLAT_ORDER = ("hyper_w1.weight", "hyper_b1.weight", "hyper_w2.weight", "hyper_b2.0.weight",
                   "hyper_w1.bias", "hyper_b1.bias", "hyper_w2.bias", "hyper_b2.0.bias",
                   "hyper_b2.2.weight", "hyper_b2.2.bias")
# ... packed tight behind hyper_w1: wcat [N*E + 3E, S] and bcat [N*E + 3E] stay one matrix / vector whatever E is
QMIX_TIGHT = frozenset(("hyper_b1.weight", "hyper_w2.weight", "hyper_b2.0.weight", "hyper_b1.bias", "hyper_w2.bias",
                        "hyper_b2.0.bias"))


def qmix_struct(addr, embed, cls=L.QmixParams):
    """addr: name -> device address for QMIX_FLAT_ORDER names (contiguity is guaranteed by FlatBuffer); embed: E."""
    s = cls()
    s.wcat, s.bcat = addr["hyper_w1.weight"], addr["hyper_w1.bias"]
    s.wb2, s.bb2 = addr["hyper_b2.2.weight"], addr["hyper_b2.2.bias"]
    s.embed = embed
    return s


# two_hyper_layers=True (mixer.py:36-43): the first layers of hyper_w1 / hyper_w2 are contiguous (one [2 hh, S] GEMM)
QMIX2_FLAT_ORDER = ("hyper_w1.0.weight", "hyper_w2.0.weight", "hyper_w1.0.bias", "hyper_w2.0.bias",
                    "hyper_w1.2.weight", "hyper_w1.2.bias", "hyper_w2.2.weight", "hyper_w2.2.bias",
                    "hyper_b1.weight", "hyper_b1.bias", "hyper_b2.0.weight", "hyper_b2.0.bias",
                    "hyper_b2.2.weight", "hyper_b2.2.bias")


def qmix2_struct(addr, embed, hh=None, cls=L.QmixHyper2):
    """addr: name -> device address for QMIX2_FLAT_ORDER names; embed: E (kept by the parameter struct only)."""
    s = cls()
    s.w_in, s.b_in = addr["hyper_w1.0.weight"], addr["hyper_w1.0.bias"]
    s.w1_out, s.b1_out = addr["hyper_w1.2.weight"], addr["hyper_w1.2.bias"]
    s.w2_out, s.b2_out = addr["hyper_w2.2.weight"], addr["hyper_w2.2.bias"]
    s.w_b1, s.b_b1 = addr["hyper_b1.weight"], addr["hyper_b1.bias"]
    s.w_b20, s.b_b20 = addr["hyper_b2.0.weight"], addr["hyper_b2.0.bias"]
    if hh is not None:
        s.hh, s.embed = hh, embed
    return s


def qmix_tail_struct(addr, embed, cls=L.QmixParams):
    """Only the last layer of hyper_b2 (what the mixing kernel itself reads); wcat / bcat stay null."""
    s = cls()
    s.wb2, s.bb2 = addr["hyper_b2.2.weight"], addr["hyper_b2.2.bias"]
    s.embed = embed
    return s


class _Qmix2Fn(torch.autograd.Function):
    """QMixMixer with two_hyper_layers=True: hyper2 GEMMs -> mixing kernel, and the reverse."""

    @staticmethod
    def forward(ctx, q, s, N, S, E, hh, *params):
        M, dev = q.shape[0], q.device
        h = torch.empty(M, 2 * hh, dtype=torch.float32, device=dev)
        hy = torch.empty(M, hy_cols(N, E), dtype=torch.float32, device=dev)
        q_tot = torch.empty(M, dtype=torch.float32, device=dev)
        addr = {n: t.data_ptr() for n, t in zip(QMIX2_FLAT_ORDER, params)}
        p2, pt = qmix2_struct(addr, E, hh), qmix_tail_struct(addr, E)
        L.call("marl_qmix_hyper2_fwd", M, N, S, C.byref(p2), s.data_ptr(), h.data_ptr(), hy.data_ptr(), L.stream_ptr())
        L.call("marl_qmix_mix_fwd", M, N, C.byref(pt), q.data_ptr(), hy.data_ptr(), q_tot.data_ptr(), L.stream_ptr())
        ctx.save_for_backward(q, s, h, hy, *params)
        ctx.meta = (N, S, E, hh)
        return q_tot

    @staticmethod
    def backward(ctx, dq_tot):
        N, S, E, hh = ctx.meta
        q, s, h, hy, *params = ctx.saved_tensors
        M, dev = q.shape[0], q.device
        sizes = [p.numel() for p in params]
        gbuf = torch.zeros(sum(sizes), dtype=torch.float32, device=dev)
        views, off = [], 0
        for p, n in zip(params, sizes):
            views.append(gbuf[off:off + n].view(p.shape))
            off += n
        addr = {n: t.data_ptr() for n, t in zip(QMIX2_FLAT_ORDER, params)}
        gaddr = {n: v.data_ptr() for n, v in zip(QMIX2_FLAT_ORDER, views)}
        p2, pt = qmix2_struct(addr, E, hh), qmix_tail_struct(addr, E)
        g2, gt = qmix2_struct(gaddr, E, None, L.QmixHyper2Grads), qmix_tail_struct(gaddr, E, L.QmixGrads)
        dhy = torch.empty_like(hy)
        dh = torch.empty_like(h)
        dq = torch.empty(M, N, dtype=torch.float32, device=dev)
        L.call("marl_qmix_mix_bwd", M, N, C.byref(pt), q.data_ptr(), hy.data_ptr(), dq_tot.contiguous().data_ptr(),
               dhy.data_ptr(), dq.data_ptr(), C.byref(gt), L.stream_ptr())
        L.call("marl_qmix_hyper2_bwd", M, N, S, C.byref(p2), s.data_ptr(), h.data_ptr(), dhy.data_ptr(), dh.data_ptr(),
               C.byref(g2), L.stream_ptr())
        return (dq, None, None, None, None, None, *views)


class _QmixFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, q, s, N, S, E, *params):
        M = q.shape[0]
        dev = q.device
        hy = torch.empty(M, hy_cols(N, E), dtype=torch.float32, device=dev)
        q_tot = torch.empty(M, dtype=torch.float32, device=dev)
        p = qmix_struct({n: t.data_ptr() for n, t in zip(QMIX_FLAT_ORDER, params)}, E)
        L.call("marl_qmix_fwd", M, N, S, C.byref(p), q.data_ptr(), s.data_ptr(), hy.data_ptr(), q_tot.data_ptr(),
               L.stream_ptr())
        ctx.save_for_backward(q, s, hy, *params)
        ctx.meta = (N, S, E)
        return q_tot

    @staticmethod
    def backward(ctx, dq_tot):
        N, S, E = ctx.meta
        q, s, hy, *params = ctx.saved_tensors
        M = q.shape[0]
        dev = q.device
        # gradient buffer with the same contiguous layout as the parameters
        sizes = [p.numel() for p in params]
        gbuf = torch.zeros(sum(sizes), dtype=torch.float32, device=dev)
        views, off = [], 0
        for p, n in zip(params, sizes):
            views.append(gbuf[off:off + n].view(p.shape))
            off += n
        addr = {n: v.data_ptr() for n, v in zip(QMIX_FLAT_ORDER, views)}
        g = qmix_struct(addr, E, L.QmixGrads)
        pst = qmix_struct({n: t.data_ptr() for n, t in zip(QMIX_FLAT_ORDER, params)}, E)
        dhy = torch.empty_like(hy)
        dq = torch.empty(M, N, dtype=torch.float32, device=dev)
        L.call("marl_qmix_bwd", M, N, S, C.byref(pst), q.data_ptr(), s.data_ptr(), hy.data_ptr(),
               dq_tot.contiguous().data_ptr(), dhy.data_ptr(), dq.data_ptr(), C.byref(g), L.stream_ptr())
        return (dq, None, None, None, None, *views)


class QMixMixer(FlatPackedMixin, nn.Module):
    """Monotonic mixing network with state-conditioned hyper-networks (mixer.py:21-80)."""

    def __init__(self, args):
        super().__init__()
        self.args = args
        E = args.qmix_hidden_dim
        if not 1 <= E <= MAX_EMBED:
            raise ValueError(f"qmix_hidden_dim must be an integer in 1..{MAX_EMBED}, got {E!r}")
        S, N = args.state_shape, args.n_agents
        self.two_hyper_layers = bool(getattr(args, "two_hyper_layers", False))
        if self.two_hyper_layers:                     # mixer.py:36-43
            hh = args.hyper_hidden_dim
            if hh % 4:
                raise ValueError("hyper_hidden_dim must be a multiple of 4 (128-bit operand loads)")
            self.hyper_w1 = nn.Sequential(nn.Linear(S, hh), nn.ReLU(), nn.Linear(hh, N * E))
            self.hyper_w2 = nn.Sequential(nn.Linear(S, hh), nn.ReLU(), nn.Linear(hh, E))
        else:
            self.hyper_w1 = nn.Linear(S, N * E)
            self.hyper_w2 = nn.Linear(S, E)
        self.hyper_b1 = nn.Linear(S, E)
        self.hyper_b2 = nn.Sequential(nn.Linear(S, E), nn.ReLU(), nn.Linear(E, 1))
        self._flat = None
        self._pack(torch.device("cuda") if torch.cuda.is_available() else torch.device("cpu"))

    def flat_named_parameters(self):
        table = dict(self.named_parameters())
        if self.two_hyper_layers:
            return [(n, table[n]) for n in QMIX2_FLAT_ORDER]
        return [(n, table[n], "tight") if n in QMIX_TIGHT else (n, table[n]) for n in QMIX_FLAT_ORDER]

    def _pack(self, device):
        self._flat = FlatBuffer(self.flat_named_parameters(), device=device, with_grad=False)

    def adopt(self, flat):
        self._flat = flat

    def _apply(self, fn, *a, **k):
        out = super()._apply(fn, *a, **k)
        self._pack(self.hyper_w1.weight.device)
        return out

    def param_addresses(self):
        return {e[0]: e[1].data_ptr() for e in self.flat_named_parameters()}

    def forward(self, q_values, states):
        # states (episode_num, max_episode_len, state_shape); q_values (episode_num, max_episode_len, n_agents)
        episode_num = q_values.size(0)
        self.ensure_packed()      # the kernels read the four heads as ONE matrix: a copied module is re-packed first
        N, S, E = self.args.n_agents, self.args.state_shape, self.args.qmix_hidden_dim
        q = L.require_cuda(q_values, "q_values").reshape(-1, N).to(torch.float32).contiguous()
        s = L.require_cuda(states, "states").reshape(-1, S).to(torch.float32).contiguous()
        params = [e[1] for e in self.flat_named_parameters()]
        if self.two_hyper_layers:
            q_tot = _Qmix2Fn.apply(q, s, N, S, E, self.args.hyper_hidden_dim, *params)
        else:
            q_tot = _QmixFn.apply(q, s, N, S, E, *params)
        return q_tot.view(episode_num, -1, 1)


# north_star alias (pymarl spelling): QMixer.forward(agent_qs, states)
QMixer = QMixMixer

from .qplex import DMAQ_SI_Weight, DMAQer  # noqa: E402,F401  (reference: network/mixer.py:85-288)
from .qtran import QtranQBase, QtranV  # noqa: E402,F401      (reference: network/mixer.py:355-418)
