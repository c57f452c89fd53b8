"""rnn_hidden_dim = 32 and 128 on the device: the unroll and its backward against fp64 autograd of the oracle, the hidden
field of the C ABI, every acting entry point, the batched rollouts, and the learners against the fp64 oracle on their
routes (graphs, replay batches, SeparatedMAC, last_action, modules, the TMA back end, deterministic mode), checkpoints,
the matrix-game tables and data parallelism.

Tolerance: within 1e-5 of the fp32 oracle, or, failing that, as close to the fp64 oracle as the fp32 oracle is."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from marl_b200 import _lib as L
from marl_b200.controller.share_params import PhiloxDraws
from marl_b200.synthetic import synthetic_batch
from oracle import marl_oracle as MO
from tests import parity_util as PU
from tests import separated_rollout_oracle as SRO

pytestmark = pytest.mark.gpu
TOL = 1e-5
WIDTHS = (32, 128)
TINY = (3, 4, 5, 6, 8, 4)               # N, A, O, S, T, B
CFG2 = (5, 11, 80, 120, 120, 32)        # the 2s3z-like shape of bench.py's headline
ACT_SHAPES = [(64, 5, 11, 80), (32, 8, 14, 128), (16, 27, 36, 285)]      # cfg-2, 3, 4 acting shapes: n, N, A, O


def _close(mine, o32, o64):
    """The repository's rule: within TOL of the fp32 oracle, or as close to the fp64 oracle as the fp32 oracle is."""
    if PU.rel_err(mine, o32) < TOL:
        return True
    return PU.rel_err(mine, o64) <= max(PU.rel_err(o32, o64), 1e-7)


# ------------------------------------------------------------------------------------------ unroll and backward
def _unroll_case(H, B, T, N, A, O, last_action=True, reuse_network=True, seed=0):
    from marl_b200.network.q_network import RNNQNet
    args = PU.make_args("qmix", N, A, O, 4, T, rnn_hidden_dim=H, last_action=last_action, reuse_network=reuse_network)
    torch.manual_seed(seed)
    I = O + A * last_action + N * reuse_network
    net = RNNQNet(I, args)
    g = torch.Generator().manual_seed(seed + 1)
    obs = torch.randn(B, T, N, O, generator=g, dtype=torch.float64)
    onehot = torch.nn.functional.one_hot(torch.randint(0, A, (B, T, N), generator=g), A).double()
    h0 = 0.5 * torch.randn(B * N, H, generator=g, dtype=torch.float64)
    wq = torch.randn(B, T, N, A, generator=g, dtype=torch.float64)
    wh = torch.randn(B, T, N, H, generator=g, dtype=torch.float64)
    # device
    cu = lambda x: x.float().cuda().contiguous()
    h0d = cu(h0).requires_grad_(True)
    params = [p for _, p in net.flat_named_parameters()]
    q, hid, hl = net.unroll(cu(obs), cu(onehot) if last_action else None, h0d, 0, last_action, reuse_network)
    loss = (q * cu(wq)).sum() + (hid * cu(wh)).sum()
    grads = torch.autograd.grad(loss, [h0d] + params)
    mine = dict(q=q, hidden=hid, h_last=hl, dh0=grads[0])
    mine.update({n: gr for (n, _), gr in zip(net.flat_named_parameters(), grads[1:])})
    # oracle in fp32 and fp64
    cfg = MO.make_cfg(n_agents=N, n_actions=A, obs_shape=O, rnn_hidden_dim=H, last_action=last_action,
                      reuse_network=reuse_network)
    ref = {}
    for dt in (torch.float32, torch.float64):
        p = {k: v.detach().cpu().to(dt).requires_grad_(True) for k, v in net.state_dict().items()}
        hh = h0.to(dt).requires_grad_(True)
        oq, oh, ol = MO.unroll(p, obs.to(dt), onehot.to(dt), hh, cfg)
        ol_ = (oq * wq.to(dt)).sum() + (oh * wh.to(dt)).sum()
        keys = list(p)
        gr = torch.autograd.grad(ol_, [hh] + [p[k] for k in keys])
        r = dict(q=oq, hidden=oh, h_last=ol, dh0=gr[0])
        r.update({k: v for k, v in zip(keys, gr[1:])})
        ref[dt] = r
    bad = [k for k in mine if not _close(mine[k], ref[torch.float32][k], ref[torch.float64][k])]
    assert not bad, {k: (PU.rel_err(mine[k], ref[torch.float32][k]), PU.rel_err(mine[k], ref[torch.float64][k])) for k in bad}


@pytest.mark.parametrize("H", WIDTHS)
@pytest.mark.parametrize("B", [20, 50, 100, 200])       # 100 / 250 / 500 / 1000 rows: 1, 2, <= 4 and <= 8 rows per CTA
def test_unroll_fwd_bwd_vs_fp64_oracle_at_every_pass_size(H, B):
    _unroll_case(H, B, 6, 5, 11, 20, seed=B)


@pytest.mark.parametrize("H", WIDTHS)
@pytest.mark.parametrize("last_action,reuse_network", [(False, True), (True, False), (False, False)])
def test_unroll_input_flags(H, last_action, reuse_network):
    _unroll_case(H, 7, 9, 3, 5, 6, last_action, reuse_network, seed=3)


def _raw_unroll(hidden_fields, H=64, B=4, T=5, N=3, A=4, O=6):
    """marl_agent_unroll_fwd with one stream per entry of hidden_fields (the value written to params.hidden); returns the
    q and hidden outputs of every stream."""
    from marl_b200.network.q_network import RNNQNet, agent_param_struct
    torch.manual_seed(0)
    net = RNNQNet(O + A + N, PU.make_args("qmix", N, A, O, 4, T, rnn_hidden_dim=H))
    f = lambda *s: torch.zeros(*s, device="cuda")
    obs, onehot = torch.randn(B, T, N, O, device="cuda"), f(B, T, N, A)
    streams, outs = (L.UnrollStream * len(hidden_fields))(), []
    for i, hf in enumerate(hidden_fields):
        o = dict(q=f(B, T, N, A), hidden=f(B, T, N, H), x=f(B * T * N, H), gi=f(B * T * N, 3 * H))
        st = streams[i]
        st.obs, st.onehot, st.h0_from = obs.data_ptr(), onehot.data_ptr(), -1
        st.params = agent_param_struct(net.param_addresses(), hidden=hf)
        st.q, st.hidden, st.x, st.gi = (o[k].data_ptr() for k in ("q", "hidden", "x", "gi"))
        outs.append(o)
    L.call("marl_agent_unroll_fwd", C.byref(L.Dims(B, T, N, A, O, 0)), streams, len(hidden_fields), L.stream_ptr())
    torch.cuda.synchronize()
    return outs


def test_hidden_zero_means_64_bit_for_bit():
    (a,), (b,) = _raw_unroll([0]), _raw_unroll([64])
    assert torch.equal(a["q"], b["q"]) and torch.equal(a["hidden"], b["hidden"])


def test_unsupported_and_mismatched_widths_are_einval():
    for hf in (16, 48, 96, 256, -1):
        with pytest.raises(ValueError, match="MARL_EINVAL"):
            _raw_unroll([hf])
    with pytest.raises(ValueError, match="MARL_EINVAL"):
        _raw_unroll([64, 32])
    with pytest.raises(ValueError, match="MARL_EINVAL"):
        _raw_unroll([32, 128], H=128)
    # separated acting: the N parameter sets must carry one width
    mac = _mac("separated", 3, 4, 5, 32)
    sets = (L.AgentParams * 3)(*(net.param_struct() for net in mac.agent))
    sets[1].hidden = 64
    n, N, A, O = 2, 3, 4, 5
    t = lambda *s: torch.zeros(*s, device="cuda")
    obs, last, avail, h, q = t(n, N, O), t(n, N, A), t(n, N, A) + 1, t(n * N, 32), t(n, N, A)
    act = torch.empty(n, N, dtype=torch.int64, device="cuda")
    with pytest.raises(ValueError, match="MARL_EINVAL"):
        L.call("marl_agent_act_separated", n, N, A, O, 1, 0, sets, obs.data_ptr(), last.data_ptr(), avail.data_ptr(),
               h.data_ptr(), h.data_ptr(), None, None, None, None, 0.0, None, act.data_ptr(), None, q.data_ptr(),
               L.stream_ptr())


# ------------------------------------------------------------------------------------------ acting
def _mac(kind, N, A, O, H, last_action=True, reuse_network=True, seed=0):
    from marl_b200.controller.share_params import SeparatedMAC, SharedMAC
    torch.manual_seed(seed)
    cls = SharedMAC if kind == "shared" else SeparatedMAC
    return cls(PU.make_args("qmix", N, A, O, 4, 10, last_action=last_action, reuse_network=reuse_network,
                            rnn_hidden_dim=H))


def _act_inputs(n, N, A, O, H, seed):
    rng = np.random.RandomState(seed)
    t = lambda x: torch.as_tensor(x, dtype=torch.float32, device="cuda").contiguous()
    avail = (rng.rand(n, N, A) < 0.6).astype(np.float32)
    avail[::5, 0, :] = 0.0
    return (t(rng.randn(n, N, O)), t(np.eye(A)[rng.randint(0, A, (n, N))]), t(avail), t(0.5 * rng.randn(n * N, H)),
            rng.rand(n, N), rng.rand(n, N))


def _oracle_step(mac, kind, obs, last, h, dt):
    N = mac.n_agents
    n = obs.shape[0]
    cfg = MO.make_cfg(n_agents=N, n_actions=mac.n_actions, obs_shape=obs.shape[2], rnn_hidden_dim=h.shape[1],
                      last_action=mac.args.last_action, reuse_network=mac.args.reuse_network)
    nets = mac.agent if kind == "separated" else [mac.agent]
    p = [{k: v.detach().cpu().to(dt) for k, v in net.state_dict().items()} for net in nets]
    q, hh, _ = MO.unroll(p if kind == "separated" else p[0], obs.cpu().to(dt)[:, None], last.cpu().to(dt)[:, None],
                         h.cpu().to(dt), cfg)
    return q[:, 0], hh[:, 0].reshape(n * N, -1)


def _want_actions(q64, avail, eu=None, cu=None, eps=0.0):
    """Masked first maximum (0 when nothing is available), then the uniform exploration rule of include/marl_b200.h."""
    av = avail.cpu().numpy()
    q = np.where(av != 0, q64.numpy(), -np.inf)
    best = np.where(av.any(-1), q.argmax(-1), 0)
    if eu is not None:
        for e, a in zip(*np.nonzero(eu < eps)):
            idx = np.nonzero(av[e, a])[0]
            best[e, a] = idx[min(int(np.floor(cu[e, a] * len(idx))), len(idx) - 1)] if len(idx) else 0
    return best


@pytest.mark.parametrize("H", WIDTHS)
@pytest.mark.parametrize("kind", ["shared", "separated"])
@pytest.mark.parametrize("n,N,A,O", ACT_SHAPES)
def test_act_entry_points_vs_oracle(H, kind, n, N, A, O):
    """marl_agent_act_input / _separated (greedy and exploring with fed uniforms), their Philox forms against the uniform
    form fed the same Philox uniforms, and (shared) the plain marl_agent_act: q and h' within tolerance of the oracle, the
    actions exact wherever the fp64 top-2 gap leaves the greedy choice unambiguous."""
    from tests.test_philox_rollout_gpu import np_uniforms
    mac = _mac(kind, N, A, O, H, seed=n + H)
    obs, last, avail, h0, eu, cu = _act_inputs(n, N, A, O, H, n + N)
    q64, h64 = _oracle_step(mac, kind, obs, last, h0, torch.float64)
    q32, h32 = _oracle_step(mac, kind, obs, last, h0, torch.float32)
    srt = np.sort(np.where(avail.cpu().numpy() != 0, q64.numpy(), -np.inf), -1)
    clear = ~((srt[..., -1] - srt[..., -2]) < 1e-5)
    runs = {}
    for form in ("greedy", "explore"):
        h, q = h0.clone(), torch.empty(n, N, A, device="cuda")
        kw = {} if form == "greedy" else dict(explore_u=torch.as_tensor(eu, device="cuda"),
                                              choice_u=torch.as_tensor(cu, device="cuda"), eps=0.4)
        act = mac.act(n, obs, last, avail, h, q=q, **kw).cpu().numpy()
        assert _close(q, q32, q64) and _close(h, h32, h64), form
        want = _want_actions(q64, avail, *((eu, cu, 0.4) if form == "explore" else ()))
        keep = clear | ((eu < 0.4) if form == "explore" else False)
        assert np.array_equal(act[keep], want[keep]), form
        runs[form] = (act, q, h)
    draws = PhiloxDraws(seed=7 + n, episode_base=3, step=2)
    out = []
    for philox in (True, False):
        h, q, oh = h0.clone(), torch.empty(n, N, A, device="cuda"), torch.empty(n, N, A, device="cuda")
        if philox:
            act = mac.act(n, obs, last, avail, h, eps=0.5, q=q, onehot=oh, philox=draws)
        else:
            pe, pc = (torch.as_tensor(x, device="cuda").contiguous() for x in np_uniforms(7 + n, 3, 2, n, N))
            act = mac.act(n, obs, last, avail, h, explore_u=pe, choice_u=pc, eps=0.5, q=q, onehot=oh)
        out.append((act, oh, q, h))
    assert all(torch.equal(x, y) for x, y in zip(*out))
    if kind == "shared":
        h, q = h0.clone(), torch.empty(n, N, A, device="cuda")
        act = torch.empty(n, N, dtype=torch.int64, device="cuda")
        L.call("marl_agent_act", n, N, A, O, C.byref(mac.agent.param_struct()), obs.data_ptr(), last.data_ptr(),
               avail.data_ptr(), h.data_ptr(), h.data_ptr(), None, None, None, None, 0.0, None, act.data_ptr(), None,
               q.data_ptr(), L.stream_ptr())
        ga, gq, gh = runs["greedy"]
        assert np.array_equal(act.cpu().numpy(), ga) and torch.equal(q, gq) and torch.equal(h, gh)


# ------------------------------------------------------------------------------------------ rollouts
PAYOFF1 = [[8, -12, -12], [-12, 0, 0], [-12, 0, 0]]
KEYS11 = ("o", "s", "u", "r", "avail_u", "o_next", "s_next", "avail_u_next", "u_onehot", "padded", "terminated")


@pytest.mark.parametrize("epsilon", [0.3, 0.0])
def test_matrix_game_rollout_at_128(epsilon):
    from marl_b200.env.single_state_matrix_game import BatchedMatrixGame
    from marl_b200.rollout import BatchedRolloutWorker
    n = 4096

    def worker():
        from marl_b200.controller.share_params import SharedMAC
        torch.manual_seed(5)
        mac = SharedMAC(PU.make_args("qmix", 2, 3, 1, 1, 1, rnn_hidden_dim=128))
        mac.args.epsilon, mac.args.anneal_epsilon = epsilon, 0.01
        env = BatchedMatrixGame(PAYOFF1, n, keep_r64=True)
        return BatchedRolloutWorker(env, mac, mac.args), env, mac
    w, env, mac = worker()
    np.random.seed(7)
    episodes, _, _, steps = w.generate_episodes(rng="numpy")
    np.random.seed(7)
    agent = {k: v.detach().cpu() for k, v in mac.agent.state_dict().items()}
    want_u, want_r, want_eps = SRO.generate_episodes(agent, PAYOFF1, n, epsilon, 0.01, mac.args.min_epsilon, "step",
                                                    hidden=128)
    assert np.array_equal(episodes["u"].reshape(n, 2).cpu().numpy(), want_u)
    assert np.array_equal(env.r64.cpu().numpy(), want_r) and w.epsilon == want_eps and steps == n
    runs = [worker()[0].generate_episodes(rng="philox")[0]["u"] for _ in range(2)]
    assert torch.equal(runs[0], runs[1])


def test_multistep_rollout_at_128():
    from marl_b200.rollout import BatchedRolloutWorker
    from tests.envs import CountdownGameBatched, CountdownGameHost
    N, A, O, S, T, n = 3, 5, 4, 3, 12, 64

    def worker():
        mac = _mac("shared", N, A, O, 128, seed=8)
        a = mac.args
        a.state_shape, a.episode_limit = S, T
        a.epsilon, a.anneal_epsilon, a.min_epsilon, a.epsilon_anneal_scale = 0.5, 0.01, 0.02, "step"
        return BatchedRolloutWorker(CountdownGameBatched(n, n_agents=N, n_actions=A, episode_limit=T), mac, a), mac
    w, mac = worker()
    rng = np.random.RandomState(3)
    draws = (rng.rand(n, T, N), rng.rand(n, T, N))
    ep, rewards, _, steps = w.generate_episodes(draws=draws)
    agent = {k: v.detach().cpu() for k, v in mac.agent.state_dict().items()}
    oep, orew, osteps = SRO.rollout_multistep(agent, CountdownGameHost(n_agents=N, n_actions=A, episode_limit=T), n, 0.5,
                                              0.01, 0.02, "step", draws=draws, hidden=128)
    for k in KEYS11:
        assert np.array_equal(ep[k].cpu().numpy().astype(np.float64), oep[k]), k
    assert np.array_equal(rewards.cpu().numpy(), np.array(orew)) and steps == osteps
    runs = [worker()[0].generate_episodes(rng="philox")[0] for _ in range(2)]
    assert all(torch.equal(runs[0][k], runs[1][k]) for k in KEYS11)


# ------------------------------------------------------------------------------------------ learners against the fp64 oracle
def _args(shape, H, alg="qmix", **kw):
    N, A, O, S, T, _ = shape
    return PU.make_args(alg, N, A, O, S, T, rnn_hidden_dim=H, **kw)


def _batch(shape, seed=0, **kw):
    N, A, O, S, T, B = shape
    return synthetic_batch(seed, B, T, N, A, O, S, **kw)


def _train_vs_fp64(args, batch, steps=3):
    """Per step, on the learner's current weights: the loss against the fp64 oracle, the clipped gradients against the fp32
    oracle with the fp64 oracle as the arbiter (PU.compare_grads)."""
    learner, _ = PU.build_pair(args)
    cfg = PU.oracle_cfg(args)
    params = lambda: PU.export_params(learner)
    st32, st64 = (MO.LearnerState(cfg, params(), dtype=dt) for dt in (torch.float32, torch.float64))
    report = []
    for step in range(steps):
        for st in (st32, st64):
            for g, sd in params().items():
                for k, v in sd.items():
                    st.params[g][k] = v.to(st.dtype).requires_grad_(True)
        loss = learner.train({k: v.copy() for k, v in batch.items()}, step)
        oloss, info = MO.train_step(st64, batch, step)
        info32 = MO.train_step(st32, batch, step)[1]
        if abs(loss - oloss) > TOL * abs(oloss):
            report.append(f"step {step}: loss {loss} vs {oloss}")
        mine = {f"{g}.{k}": p.grad for g, m in PU.module_groups(learner).items() for k, p in m.named_parameters()}
        before = len(report)
        PU.compare_grads(mine, info32["clipped_grads"], TOL, report, info["clipped_grads"], whole_tol=5 * TOL)
        report[before:] = [f"step {step}: {r}" for r in report[before:]]
    assert not report, "\n".join(report)
    return learner


def _groups(learner):
    if isinstance(learner.eval_net.agent, list):
        g = {f"agent.{n}": net for n, net in enumerate(learner.eval_net.agent)}
        g["mixer"] = learner.mixer
        return g
    return PU.module_groups(learner)


CASES = {"rms": {}, "adam": dict(optimizer="Adam"), "no_double_q": dict(double_q=False)}
ALGS = ("vdn", "qmix", "qplex", "qtran_base")


@pytest.mark.parametrize("H", WIDTHS)
@pytest.mark.parametrize("alg", ALGS)
@pytest.mark.parametrize("case", list(CASES))
def test_learner_tiny_shape(H, alg, case):
    _train_vs_fp64(_args(TINY, H, alg, **CASES[case]), _batch(TINY))


@pytest.mark.parametrize("H", WIDTHS)
@pytest.mark.parametrize("alg", ALGS)
def test_learner_cfg2_shape(H, alg):
    _train_vs_fp64(_args(CFG2, H, alg), _batch(CFG2), steps=1)


@pytest.mark.parametrize("H", WIDTHS)
def test_learner_ten_steps(H):
    _train_vs_fp64(_args(TINY, H, optimizer="Adam"), _batch(TINY), steps=10)


@pytest.mark.parametrize("H", WIDTHS)
def test_early_exit_with_row_order(H):
    """640 rows (B = 128, N = 5) of ragged episodes: the recurrences stop at each episode's length and the rows are dealt
    length-sorted (row_order) in the forward and the BPTT."""
    shape = (5, 4, 6, 6, 20, 128)
    args = _args(shape, H)
    learner = _train_vs_fp64(args, _batch(shape, full_length_first=False, min_len=3), steps=2)
    assert learner._agent_plan(128, 20)[1]


def _losses(args, batches, make=None):
    learner = make(args) if make else PU.build_pair(args)[0]
    return [learner.train(b if not isinstance(b, dict) else {k: v.copy() for k, v in b.items()}, i)
            for i, b in enumerate(batches)], learner


@pytest.mark.parametrize("H", WIDTHS)
def test_graphs_replay_modules(H):
    from marl_b200.common.replaybuffer import ReplayBuffer
    N, A, O, S, T, _ = TINY
    b1, b2 = synthetic_batch(0, 4, T, N, A, O, S), synthetic_batch(1, 6, T, N, A, O, S, full_length_first=False, min_len=3)
    seq = [b1, b2, b1, b2, b1, b2]
    lg, learner = _losses(_args(TINY, H), seq)
    assert sum(1 for v in learner._graphs.values() if isinstance(v, tuple)) == 2
    le, _ = _losses(_args(TINY, H, cuda_graph=False), seq)
    assert np.allclose(lg, le, rtol=TOL, atol=0), (lg, le)
    lm, _ = _losses(_args(TINY, H, train_through_modules=True), seq)
    assert np.allclose(lm, le, rtol=TOL, atol=0), (lm, le)
    from oracle.replay_oracle import OracleReplayBuffer
    args = _args(TINY, H, buffer_size=10)
    la, st = PU.build_pair(args)
    lb, _ = PU.build_pair(args)
    buf, orc = ReplayBuffer(args), OracleReplayBuffer(10, T, N, A, O, S)
    for seed in range(3):
        ep = synthetic_batch(seed, 4, T, N, A, O, S, full_length_first=False, min_len=2)
        buf.store_episode({k: v.copy() for k, v in ep.items()})
        orc.store(ep)
    for step in range(3):
        np.random.seed(10 + step)
        host_batch, _ = orc.sample(6)
        np.random.seed(10 + step)
        view = buf.sample(6)
        a = la.train({k: v.copy() for k, v in host_batch.items()}, step)
        b = lb.train(view, step)
        assert abs(a - b) <= 1e-6 * abs(a)
        oloss, _ = MO.train_step(st, host_batch, step)
        assert abs(b - oloss) <= TOL * abs(oloss)


@pytest.mark.parametrize("H", WIDTHS)
@pytest.mark.parametrize("alg", ["vdn", "qmix"])
def test_separated_mac(H, alg):
    from marl_b200.controller.share_params import SeparatedMAC
    from marl_b200.algorithm.q_learner import QLearner
    args = _args(TINY, H, alg, reuse_network=False)
    torch.manual_seed(0)
    learner = QLearner(SeparatedMAC(args), args)
    learner._update_targets()
    cfg = PU.oracle_cfg(args)
    cfg.separated, cfg.reuse_network = True, False
    batch = _batch(TINY)

    st = MO.LearnerState(cfg, {g: {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
                               for g, m in _groups(learner).items()})
    for step in range(2):
        loss = learner.train({k: v.copy() for k, v in batch.items()}, step)
        oloss, _ = MO.train_step(st, batch, step)
        assert abs(loss - oloss) <= TOL * abs(oloss), step


@pytest.mark.parametrize("H", WIDTHS)
def test_last_action_off(H):
    args = _args(TINY, H, last_action=False)
    learner, st = PU.build_pair(args)
    st.cfg.last_action = False
    batch = _batch(TINY)
    for step in range(3):
        loss = learner.train({k: v.copy() for k, v in batch.items()}, step)
        oloss, _ = MO.train_step(st, batch, step)
        assert abs(loss - oloss) <= TOL * abs(oloss), step


@pytest.mark.parametrize("H", WIDTHS)
@pytest.mark.parametrize("switch", ["tgemm", "deterministic"])
def test_tma_back_end_and_deterministic_mode(H, switch):
    fn = "marl_tgemm_enable" if switch == "tgemm" else "marl_set_deterministic"
    prev = getattr(L.load(), fn)(1)
    try:
        args = _args(TINY, H, cuda_graph=False)
        learner, st = PU.build_pair(args)
        batch = _batch(TINY)
        for step in range(2):
            loss = learner.train({k: v.copy() for k, v in batch.items()}, step)
            oloss, _ = MO.train_step(st, batch, step)
            assert abs(loss - oloss) <= TOL * abs(oloss), step
    finally:
        getattr(L.load(), fn)(prev)


@pytest.mark.parametrize("H", WIDTHS)
def test_checkpoint_round_trip(H, tmp_path):
    args = _args(TINY, H)
    args.model_dir = str(tmp_path)
    src, _ = PU.build_pair(args, seed=0)
    batch = _batch(TINY)
    src.train({k: v.copy() for k, v in batch.items()}, 0)
    src.save_models(0)
    for k in ("rnn_net_params", "mixer_net_params"):
        os.replace(os.path.join(src.model_dir, f"0_{k}.pkl"), os.path.join(src.model_dir, f"{k}.pkl"))
    dst, _ = PU.build_pair(args, seed=1)
    dst.load_models()
    sa, sb = src.eval_net.agent.state_dict(), dst.eval_net.agent.state_dict()
    assert sa.keys() == sb.keys() and all(torch.equal(sa[k], sb[k]) for k in sa)
    assert tuple(sb["rnn.weight_hh"].shape) == (3 * H, H)
    src._update_targets()
    dst._update_targets()
    a = src.train({k: v.copy() for k, v in batch.items()}, 1)
    b = dst.train({k: v.copy() for k, v in batch.items()}, 1)
    assert abs(a - b) <= 1e-6 * abs(a)


@pytest.mark.parametrize("H", WIDTHS)
def test_matrix_game_q_tables(H):
    args = PU.make_args("qmix", 2, 3, 1, 1, 1, rnn_hidden_dim=H)
    learner, st = PU.build_pair(args)
    qt, qi, qj = learner.get_q_and_q_tot_table()
    P = {g: {k: v.detach().double() for k, v in sd.items()} for g, sd in st.params.items()}
    x = torch.cat([torch.ones(2, 1), torch.zeros(2, 3), torch.eye(2)], dim=1).double()
    q, _ = MO.agent_step(P["agent"], x, torch.zeros(2, H, dtype=torch.float64))
    assert PU.rel_err(qi, q[0]) < TOL and PU.rel_err(qj, q[1]) < TOL
    want = np.zeros((3, 3))
    for i in range(3):
        for j in range(3):
            chosen = torch.stack([q[0, i], q[1, j]]).view(1, 1, 2)
            want[i, j] = float(MO.qmix_mix(P["mixer"], chosen, torch.ones(1, 1, 1, dtype=torch.float64), st.cfg))
    assert PU.rel_err(qt, want) < TOL


def _dp_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    learner, _ = PU.build_pair(_args(TINY, 128))
    learner.enable_data_parallel()
    batch = _batch(TINY)
    ret[rank] = ([learner.train({k: v.copy() for k, v in batch.items()}, i) for i in range(4)],
                 learner._flat.data.cpu().numpy())
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_data_parallel():
    import socket
    import torch.multiprocessing as mp
    sock = socket.socket()
    sock.bind(("127.0.0.1", 0))
    port = sock.getsockname()[1]
    sock.close()
    ret = mp.Manager().dict()
    mp.spawn(_dp_worker, args=(2, port, ret), nprocs=2, join=True)
    (l0, p0), (l1, p1) = ret[0], ret[1]
    assert l0 == l1 and np.array_equal(p0, p1)
