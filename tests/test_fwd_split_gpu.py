"""The split forward of marl_agent_unroll_fwd (include/marl_b200.h: marl_agent_unroll_fwd_split): the input layers of the
eval/o stream and of the two o_next streams as two launches side by side, the eval/o chain (level 0) and the target chain on
disjoint SMs, then the eval/o_next chain (level 1) from level 0's h_last.  Every output must be bit-identical to the one-launch
plan (MARL_B200_FWD_SPLIT=0) in a raw call, graph-replayed learner steps must agree with it, and the plan that ran is visible in the library
profiler: three recurrence launches per step where the split applies, one everywhere else."""
import ctypes as C

import numpy as np
import pytest
import torch

from marl_b200 import _lib as L
from marl_b200.synthetic import synthetic_batch
from tests import parity_util as PU

pytestmark = pytest.mark.gpu

CFG2 = (5, 11, 80, 120, 120, 32)        # N, A, O, S, T, B: the 2s3z-like shape of bench.py's headline
SMALL = (3, 4, 8, 6, 8, 4)              # a tiny shape with a 4-aligned observation (the fused input layers' tensor maps)


class _Split:
    """marl_fwd_split_enable(on) for the duration of a with-block."""

    def __init__(self, on):
        self.on = on

    def __enter__(self):
        self.prev = L.load().marl_fwd_split_enable(self.on)

    def __exit__(self, *exc):
        L.load().marl_fwd_split_enable(self.prev)


def _unroll3(B, T, N, A, O, split, seed=0):
    """The learner's three streams (eval on o with gates and W_ih^T, target on o_next, eval on o_next continued from the first)
    in one marl_agent_unroll_fwd call; returns every output and whether the call took the split forward."""
    from marl_b200.network.q_network import RNNQNet
    H, I = 64, O + A + N
    torch.manual_seed(seed)
    args = PU.make_args("qmix", N, A, O, 4, T)
    ev, tg = RNNQNet(I, args), RNNQNet(I, args)
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    obs = torch.randn(B, T, N, O, device="cuda", generator=g)
    obs_next = torch.randn(B, T, N, O, device="cuda", generator=g)
    onehot = torch.nn.functional.one_hot(torch.randint(0, A, (B, T, N), device="cuda", generator=g), A).float()
    nan = lambda *s: torch.full(s, float("nan"), device="cuda")      # every element the call writes is compared
    outs = [dict(hidden=nan(B, T, N, H), h_last=nan(B * N, H), x=nan(B * T * N, H), gi=nan(B * T * N, 3 * H))
            for _ in range(3)]
    outs[0]["gates"] = nan(B, T, N, 4 * H)
    w_ih_t = nan(H, 3 * H)
    arr = (L.UnrollStream * 3)()
    for i, (net, o, shift, h0_from) in enumerate([(ev, obs, 1, -1), (tg, obs_next, 0, -1), (ev, obs_next, 0, 0)]):
        s = arr[i]
        s.obs, s.onehot, s.shift_onehot, s.full_input, s.h0_from, s.h0 = o.data_ptr(), onehot.data_ptr(), shift, 0, h0_from, None
        s.params = net.param_struct()
        s.q = None
        for k in ("hidden", "h_last", "x", "gi"):
            setattr(s, k, outs[i][k].data_ptr())
        s.gates = outs[i]["gates"].data_ptr() if i == 0 else None
        s.w_ih_t = w_ih_t.data_ptr() if i == 0 else None
        s.last_action, s.agent_id, s.input_flags = 1, 1, 1
    d = L.Dims(B, T, N, A, O, 0)
    with _Split(split):
        took = L.load().marl_agent_unroll_fwd_split(C.byref(d), arr, 3) == 1
        L.call("marl_agent_unroll_fwd", C.byref(d), arr, 3, L.stream_ptr())
    torch.cuda.synchronize()
    outs[0]["w_ih_t"] = w_ih_t
    return outs, took


def _same(a, b):
    """Bit-for-bit equality (NaN where neither plan writes counts as equal)."""
    return torch.equal(a.view(torch.int32), b.view(torch.int32))


@pytest.mark.parametrize("B,T,N,A,O,split_expected", [
    (32, 120, 5, 11, 80, True),        # cfg 2: 160 rows
    (3, 7, 3, 4, 8, True),             # tiny and ragged: 9 rows, one level CTA with a single row
    (34, 12, 5, 11, 80, True),         # 170 rows: just inside the gate (B*N <= 170)
    (35, 12, 5, 11, 80, False),        # 175 rows: just outside
])
def test_split_forward_is_bit_identical(B, T, N, A, O, split_expected):
    on, took_on = _unroll3(B, T, N, A, O, split=1)
    off, took_off = _unroll3(B, T, N, A, O, split=0)
    assert took_on == split_expected and not took_off
    for i in range(3):
        for k in on[i]:
            assert _same(on[i][k], off[i][k]), (i, k)
    # the outputs every stream must produce were written
    for i in range(3):
        assert not torch.isnan(on[i]["hidden"]).any() and not torch.isnan(on[i]["h_last"]).any(), i
    assert not torch.isnan(on[0]["w_ih_t"]).any() and not torch.isnan(on[0]["x"]).any()


def _steps(alg, split, shape=CFG2, steps=3):
    """`steps` graph-replayed learner steps in deterministic mode: losses, and after each step the agent's parameters and
    gradients and the whole flat parameter buffer."""
    N, A, O, S, T, B = shape
    batch = synthetic_batch(0, B, T, N, A, O, S)
    prev = L.load().marl_set_deterministic(1)
    try:
        with _Split(split):
            learner, _ = PU.build_pair(PU.make_args(alg, N, A, O, S, T))
            out = []
            for i in range(steps):
                loss = learner.train({k: v.copy() for k, v in batch.items()}, i)
                agent = PU.module_groups(learner)["agent"]
                out.append((loss, [p.detach().clone() for p in agent.parameters()],
                            [p.grad.clone() for p in agent.parameters()], learner._flat.data.clone()))
            torch.cuda.synchronize()
            assert learner._use_graph and learner._graphs
            return out
    finally:
        L.load().marl_set_deterministic(prev)


@pytest.mark.parametrize("alg", ["qmix", "vdn"])
def test_learner_steps_bit_identical(alg):
    """The forward is bit-identical (test above), so the first step's agent gradient and updated agent parameters are too.
    The mixer's loss and hyper-network gradient sums differ between runs of the SAME code in the last bits even in
    deterministic mode; every later quantity is held to 1e-6 of the one-launch plan."""
    on, off = _steps(alg, 1), _steps(alg, 0)
    (l1, p1, g1, _), (l0, p0, g0, _) = on[0], off[0]
    assert all(_same(a, b) for a, b in zip(g1, g0)) and all(_same(a, b) for a, b in zip(p1, p0))
    for (l1, _, _, f1), (l0, _, _, f0) in zip(on, off):
        assert abs(l1 - l0) <= 1e-6 * abs(l0)
        assert PU.rel_err(f1, f0) <= 1e-6


def _fwd_launches(args, shape, separated=False):
    """gru_unroll_fwd_kernel launches of one eager learner step (library profiler)."""
    from marl_b200.algorithm.q_learner import QLearner
    from marl_b200.controller.share_params import SeparatedMAC
    N, A, O, S, T, B = shape
    args.cuda_graph = False
    if separated:
        torch.manual_seed(0)
        learner = QLearner(SeparatedMAC(args), args)
        learner._update_targets()
    else:
        learner, _ = PU.build_pair(args)
    batch = synthetic_batch(0, B, T, N, A, O, S)
    learner.train({k: v.copy() for k, v in batch.items()}, 0)
    torch.cuda.synchronize()
    L.profile_collect()
    L.profile(True)
    try:
        learner.train({k: v.copy() for k, v in batch.items()}, 1)
        rows = L.profile_timeline()
        L.profile_collect()
    finally:
        L.profile(False)
    return sum(1 for name, _, _ in rows if name == "gru_unroll_fwd_kernel"), learner


@pytest.mark.parametrize("case,kw,shape,want", [
    ("qmix", dict(), SMALL, 3),
    ("vdn", dict(alg="vdn"), SMALL, 3),
    ("cfg2", dict(), CFG2[:4] + (16, 32), 3),
    ("no_double_q", dict(double_q=False), SMALL, 1),
    ("separated", dict(reuse_network=False), SMALL, 1),
    ("h32", dict(rnn_hidden_dim=32), SMALL, 1),
    ("h128", dict(rnn_hidden_dim=128), SMALL, 1),
    ("early_exit", dict(early_exit=True), SMALL, 1),
    ("large_rows", dict(), (5, 11, 80, 120, 8, 35), 1),      # B*N = 175
    ("qplex", dict(alg="qplex"), SMALL, 3),                   # the agent stage is shared: any mixer at a small shape
])
def test_plan_visible_in_profiler(case, kw, shape, want):
    kw = dict(kw)
    alg = kw.pop("alg", "qmix")
    N, A, O, S, T, B = shape
    args = PU.make_args(alg, N, A, O, S, T, **kw)
    n, learner = _fwd_launches(args, shape, separated=case == "separated")
    assert n == want, (case, n)
    with _Split(0):
        n_off, _ = _fwd_launches(PU.make_args(alg, N, A, O, S, T, **kw), shape, separated=case == "separated")
    assert n_off == 1, case
