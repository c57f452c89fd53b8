"""QLearner.train with one network per agent (SeparatedMAC) on the fused device step: per-agent W_hh in the recurrence
kernels, per-agent dense layers batched over z = agent (marl_unroll_stream.agent_stride)."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from marl_b200 import _lib as L
from marl_b200.synthetic import synthetic_batch
from oracle import marl_oracle as MO
from tests import parity_util as PU

pytestmark = pytest.mark.gpu
TOL = 1e-5
QPLEX_SMALL = dict(num_kernel=2, adv_hypernet_embed=8, hypernet_embed=8)


def _learner(args, seed=0):
    """A learner over a SeparatedMAC whose agents hold distinct weights (each RNNQNet draws its own initialisation)."""
    from marl_b200.controller.share_params import SeparatedMAC
    from marl_b200.algorithm.q_learner import QLearner
    from marl_b200.algorithm.qtran_learner import QTRANLearner
    torch.manual_seed(seed)
    mac = SeparatedMAC(args)
    learner = (QTRANLearner if args.alg == "qtran_base" else QLearner)(mac, args)
    learner._update_targets()
    return learner


def _groups(learner):
    g = {f"agent.{n}": net for n, net in enumerate(learner.eval_net.agent)}
    g["mixer"] = learner.mixer
    if hasattr(learner, "v"):
        g["v"], g["q_sum_mixer"] = learner.v, learner.q_sum_mixer
    return g


def _oracle(learner, args):
    cfg = PU.oracle_cfg(args)
    cfg.separated, cfg.last_action, cfg.reuse_network = True, args.last_action, args.reuse_network
    params = {g: {k: v.detach().cpu().clone() for k, v in m.state_dict().items()} for g, m in _groups(learner).items()}
    return MO.LearnerState(cfg, params)


def _args(alg, N, A, O, S, T, **kw):
    base = dict(reuse_network=False, last_action=True, target_update_cycle=2)
    base.update(QPLEX_SMALL if alg == "qplex" else {})
    base.update(kw)
    return PU.make_args(alg, N, A, O, S, T, **base)


def _pair_losses(args, batch, steps, **learner_kw):
    """(losses, flat gradient, learner) of the fused step and of the module path on identical learners."""
    out = {}
    for modules in (False, True):
        args.train_through_modules = modules
        for k, v in learner_kw.items():
            setattr(args, k, v)
        learner = _learner(args)
        losses = [learner.train({k: v.copy() for k, v in batch.items()}, i) for i in range(steps)]
        out[modules] = (losses, learner._flat.grad.clone(), learner)
    args.train_through_modules = False
    return out[False], out[True]


@pytest.mark.parametrize("optimizer", ["RMS", "Adam"])
@pytest.mark.parametrize("double_q", [True, False])
@pytest.mark.parametrize("alg", ["vdn", "qmix", "qmix2", "qplex", "qtran_base"])
def test_fused_separated_step_vs_oracle(alg, double_q, optimizer):
    """Three steps with a target sync after step 2 against the oracle's per-agent restatement: loss within 1e-5 at step 0,
    each agent's clipped gradients within 5e-5, eval and target parameters with params_close."""
    two = alg == "qmix2"
    alg = "qmix" if two else alg
    N, A, O, S, T, B = 3, 5, 7, 9, 10, 5
    args = _args(alg, N, A, O, S, T, double_q=double_q, optimizer=optimizer, two_hyper_layers=two)
    learner = _learner(args)
    assert learner._separated and not learner._fusion().heads
    st = _oracle(learner, args)
    batch = synthetic_batch(3, B, T, N, A, O, S)
    for step in range(3):
        loss = learner.train({k: v.copy() for k, v in batch.items()}, step)
        oloss, info = MO.train_step(st, batch, step)
        assert abs(loss - oloss) <= (TOL if step == 0 else 5e-5) * abs(oloss), (step, loss, oloss)
        if step == 0:
            for g, m in _groups(learner).items():
                for k, p in m.named_parameters():
                    want = info["clipped_grads"].get(f"{g}.{k}")
                    if want is not None:
                        assert PU.rel_err(p.grad, want) < 5e-5, (g, k)
    for g, m in _groups(learner).items():
        for k, p in m.named_parameters():
            if info["clipped_grads"].get(f"{g}.{k}") is not None:
                assert PU.params_close(p, st.params[g][k], args.lr, 3), (g, k)
    for n, tnet in enumerate(learner.target_net.agent):
        for k, p in tnet.named_parameters():
            assert PU.params_close(p, st.target[f"agent.{n}"][k], args.lr, 3), (n, k)


@pytest.mark.parametrize("last_action,reuse_network", [(True, False), (True, True), (False, False), (False, True)])
def test_fused_step_agrees_with_module_path(last_action, reuse_network):
    """All four input compositions [obs | last action? | agent id?]: the fused step and the same step through the modules'
    autograd Functions (each agent its own one-agent unroll) give the same losses and flat gradient."""
    N, A, O, S, T, B = 4, 6, 12, 10, 20, 8
    args = _args("qmix", N, A, O, S, T, last_action=last_action, reuse_network=reuse_network)
    batch = synthetic_batch(5, B, T, N, A, O, S)
    (lf, gf, fused), (lm, gm, mods) = _pair_losses(args, batch, 2)
    assert abs(lf[0] - lm[0]) <= 2e-6 * abs(lf[0]) and abs(lf[1] - lm[1]) <= 5e-5 * abs(lf[1]), (lf, lm)
    assert PU.rel_err(gm, gf) < 5e-5
    # hidden states as SeparatedMAC's module path leaves them: [B, N, H], equal values
    for net in ("eval_net", "target_net"):
        hf, hm = getattr(fused, net).hidden_states, getattr(mods, net).hidden_states
        assert tuple(hf.shape) == tuple(hm.shape) == (B, N, 64), (net, hf.shape, hm.shape)
    # (after step 1 the parameters differ by one update of rounding; compare the step-0 states on a fresh pair)
    args.target_update_cycle = 100
    hs = {}
    for modules in (False, True):
        args.train_through_modules = modules
        lr = _learner(args)
        lr.train({k: v.copy() for k, v in batch.items()}, 0)
        hs[modules] = (lr.eval_net.hidden_states.clone(), lr.target_net.hidden_states.clone())
    args.train_through_modules = False
    for i in range(2):
        assert PU.rel_err(hs[False][i], hs[True][i]) < TOL


@pytest.mark.parametrize("N,B,T", [
    (3, 7, 6),          # odd B: agent boundaries inside what one CTA gets
    (7, 9, 5),          # N = 7
    (7, 45, 4),         # 315 rows: more than 296, several rows per BPTT CTA
    (3, 401, 3),        # 1203 rows: more than 8 rows per recurrence CTA, several passes per CTA
    (150, 2, 2),        # more agents than CTAs: no group per agent, the kernels split a pass at each agent boundary
])
def test_row_deal_keeps_each_pass_on_one_agent(N, B, T):
    """Shapes where the index-order deal would put rows of two agents into one pass (the deal gives each agent its own
    group of CTAs, or splits the pass): the fused step matches the module path, which runs every agent in its own call."""
    A, O, S = 4, 6, 5
    # (the VDN kernel's fused selection takes at most 64 agents: beyond that the selection is its own launch)
    args = _args("vdn", N, A, O, S, T, double_q=True, fused_mixer_kernel=N <= 64)
    batch = synthetic_batch(11, B, T, N, A, O, S)
    (lf, gf, _), (lm, gm, _) = _pair_losses(args, batch, 1)
    assert abs(lf[0] - lm[0]) <= 2e-6 * abs(lm[0]), (lf, lm)
    assert PU.rel_err(gf, gm) < 5e-5


def test_graph_replay_is_bitwise_equal_to_eager_under_deterministic_mode():
    """Under marl_set_deterministic(1) the batched weight gradients reduce their splits in a fixed order, so the captured step
    leaves the same gradients and parameters as the eager one, bit for bit.  VDN: no mixer parameters, whose gradients the
    QMIX / QPLEX kernels sum with atomics; the loss itself is such a sum in every mixing kernel, hence compared to 1e-6."""
    N, A, O, S, T, B = 3, 5, 8, 6, 12, 6
    batch = synthetic_batch(2, B, T, N, A, O, S)
    prev = L.load().marl_set_deterministic(1)
    try:
        out = {}
        for graph in (False, True):
            args = _args("vdn", N, A, O, S, T, cuda_graph=graph)
            learner = _learner(args)
            losses = [learner.train({k: v.copy() for k, v in batch.items()}, i) for i in range(5)]   # capture at the third
            out[graph] = (losses, learner._flat.data.cpu().numpy(), learner._flat.grad.cpu().numpy())
    finally:
        L.load().marl_set_deterministic(prev)
    (le, pe, ge), (lg, pg, gg) = out[False], out[True]
    assert np.allclose(le, lg, rtol=1e-6, atol=0), (le, lg)
    assert np.array_equal(pe, pg) and np.array_equal(ge, gg)


def test_launch_count_of_the_separated_step():
    """The separated agent stage: per stream one fc1, one W_ih and one fc2 launch batched over the agents, one recurrence;
    the BPTT: the fc2 data gradient, the recurrence, the dx data gradient and four weight gradients."""
    N, A, O, S, T, B = 3, 5, 7, 9, 10, 4
    args = _args("vdn", N, A, O, S, T, cuda_graph=False)
    learner = _learner(args)
    batch = synthetic_batch(0, B, T, N, A, O, S)
    learner.train({k: v.copy() for k, v in batch.items()}, 0)
    streams = 3 if args.double_q else 2
    select = 0 if learner._fusion().select else 1           # marl_q_select unless the VDN kernel selects itself
    # zero-grad + (3 per stream + recurrence) + selection + VDN kernel + 7 BPTT + optimiser
    assert learner.launches_per_step == 1 + (3 * streams + 1) + select + 1 + 7 + 1


@pytest.mark.parametrize("alg", ["vdn", "qmix"])
def test_replay_batch_trains_like_the_host_batch(alg):
    from marl_b200.common.replaybuffer import ReplayBuffer
    N, A, O, S, T = 3, 4, 5, 6, 8
    args = _args(alg, N, A, O, S, T, buffer_size=10)
    la, lb = _learner(args), _learner(args)
    buf = ReplayBuffer(args)
    ep = synthetic_batch(4, 6, T, N, A, O, S, full_length_first=False, min_len=2)
    buf.store_episode({k: v.copy() for k, v in ep.items()})
    idx = [4, 0, 0, 2, 5]
    for step in range(3):
        a = la.train({k: v[idx].copy() for k, v in ep.items()}, step)
        b = lb.train(buf.sample_at(idx), step)
        assert lb.max_episode_len == la.max_episode_len
        assert abs(a - b) <= 1e-6 * abs(a), (step, a, b)


def test_unroll_entry_points_reject_invalid_agent_strides():
    """marl_agent_unroll_fwd / _bwd: MARL_EINVAL (ValueError) for a stride that is not a multiple of 4 floats, and for a
    stride together with a full input or with W_ih^T."""
    learner = _learner(_args("vdn", 2, 3, 4, 5, 3))
    B, T, N, A, O = 2, 3, 2, 3, 4
    f = lambda *shape: torch.zeros(*shape, device="cuda")
    obs, oh, hid, x, gi, wt = f(B, T, N, O), f(B, T, N, A), f(B, T, N, 64), f(B * T * N, 64), f(B * T * N, 192), f(64, 192)
    params, stride = learner._agent_structs(learner._flat)
    grads, _ = learner._agent_structs(learner._flat, grad=True)
    d = L.Dims(B, T, N, A, O, 0)

    def fwd(**kw):
        s = L.UnrollStream()
        s.obs, s.onehot, s.h0_from, s.params = obs.data_ptr(), oh.data_ptr(), -1, params
        s.hidden, s.x, s.gi, s.q = hid.data_ptr(), x.data_ptr(), gi.data_ptr(), None
        s.agent_stride, s.last_action, s.agent_id = stride, 1, 0
        for k, v in kw.items():
            setattr(s, k, v)
        L.call("marl_agent_unroll_fwd", C.byref(d), C.byref(s), 1, L.stream_ptr())

    def bwd(**kw):
        a = L.UnrollBwd()
        a.obs, a.onehot, a.shift_onehot, a.params, a.grads = obs.data_ptr(), oh.data_ptr(), 1, params, grads
        a.hidden, a.x, a.gates = hid.data_ptr(), x.data_ptr(), f(B * T * N, 256).data_ptr()
        a.dgi, a.dgh, a.dx = gi.data_ptr(), f(B * T * N, 192).data_ptr(), f(B * T * N, 64).data_ptr()
        a.agent_stride, a.last_action, a.agent_id = stride, 1, 0
        for k, v in kw.items():
            setattr(a, k, v)
        L.call("marl_agent_unroll_bwd", C.byref(d), C.byref(a), L.stream_ptr())

    fwd()                                                   # the valid call runs
    torch.cuda.synchronize()
    for call in (fwd, bwd):
        for bad in (dict(agent_stride=stride + 2), dict(agent_stride=-4), dict(full_input=1), dict(w_ih_t=wt.data_ptr())):
            with pytest.raises(ValueError):
                call(**bad)


# ---------------------------------------------------------------------------------------------------------- two GPUs
DP_SHAPE = dict(B=8, T=10, N=3, A=5, O=12, S=9)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _dp_learner(optimizer):
    args = _args("qmix", DP_SHAPE["N"], DP_SHAPE["A"], DP_SHAPE["O"], DP_SHAPE["S"], DP_SHAPE["T"], optimizer=optimizer,
                 target_update_cycle=200)
    return _learner(args)


def _dp_worker(rank, world, port, ret, peer, optimizer):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    os.environ["MARL_B200_PEER_ALLREDUCE"] = "1" if peer else "0"
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    learner = _dp_learner(optimizer)
    learner.enable_data_parallel()
    assert (learner._peer is not None) == peer
    batch = synthetic_batch(0, **DP_SHAPE)
    losses = [learner.train({k: v.copy() for k, v in batch.items()}, i) for i in range(4)]   # eager, capture, 2 replays
    ret[rank] = (losses, learner._flat.data.cpu().numpy())
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("peer,optimizer", [(True, "RMS"), (True, "Adam"), (False, "RMS")])
def test_two_gpu_separated_dp_matches_single_gpu(peer, optimizer):
    """Each rank trains its half of the episodes; peer-memory and NCCL exchanges both reproduce the single-GPU learner."""
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_dp_worker, args=(2, _free_port(), ret, peer, optimizer), nprocs=2, join=True)
    (l0, p0), (l1, p1) = ret[0], ret[1]
    assert l0 == l1 and np.array_equal(p0, p1)
    single = _dp_learner(optimizer)
    batch = synthetic_batch(0, **DP_SHAPE)
    ls = [single.train({k: v.copy() for k, v in batch.items()}, i) for i in range(4)]
    assert np.allclose(l0, ls, rtol=1e-5)
    ps = single._flat.data.cpu().numpy()
    assert np.max(np.abs(p0 - ps)) <= 1e-5 * np.max(np.abs(ps)) + 0.1 * 5e-4 * 4
