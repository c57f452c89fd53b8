"""Batched on-device acting with one network per agent (SeparatedMAC.choose_actions / act, marl_agent_act_separated) and
the batched rollout driven by it: parity with the per-agent call and the fp64 oracle for every input composition, each
row on its own agent's weights, the exploration contract, the matrix game and the multi-step game against the sequential
restatement with per-agent networks, and the episodes going on through the replay buffer into QLearner.train."""
import warnings

import numpy as np
import pytest
import torch

from marl_b200 import _lib as L
from oracle import marl_oracle as MO
from tests import golden_util as GU
from tests import parity_util as PU
from tests import separated_rollout_oracle as SRO

pytestmark = pytest.mark.gpu
H = 64
FLAGS = [(True, True), (True, False), (False, True), (False, False)]      # (last_action, reuse_network)


def _sep(N, A, O, last_action=True, reuse_network=False, seed=0, S=4, T=10):
    from marl_b200.controller.share_params import SeparatedMAC
    torch.manual_seed(seed)                        # the N networks are built one after another: distinct weights
    return SeparatedMAC(PU.make_args("qmix", N, A, O, S, T, last_action=last_action, reuse_network=reuse_network))


def _f64_params(mac):
    return [{k: v.detach().cpu().double() for k, v in net.state_dict().items()} for net in mac.agent]


@pytest.mark.parametrize("last_action,reuse_network", FLAGS)
def test_greedy_choose_actions_matches_choose_action_loop(last_action, reuse_network):
    """The reference's literal 3s5z inputs (golden choose_action_3s5z) on distinct seeded per-agent weights: one
    choose_actions call per step gives the actions of choose_action looped over the agents, greedy, and the same carried
    hidden state, for every (last_action, reuse_network) input composition."""
    z = GU.load("choose_action_3s5z")
    N, A, O = (int(x) for x in z["meta/dims"])
    one = _sep(N, A, O, last_action, reuse_network, seed=1)
    batched = _sep(N, A, O, last_action, reuse_network, seed=2)
    batched.load_state(one)
    assert not torch.equal(one.agent[0].fc1.weight, one.agent[1].fc1.weight)
    for m in (one, batched):
        m.init_hidden(1)
    last = np.zeros((N, A))
    for t in range(z["obs"].shape[0]):
        want = np.array([int(one.choose_action(z["obs"][t, a], last[a], a, z["avail"][t, a], 0.0)) for a in range(N)])
        got = batched.choose_actions(z["obs"][t][None], last[None] if last_action else None, z["avail"][t][None], 0.0,
                                     evaluate=True)
        assert tuple(got.shape) == (1, N) and got.dtype == torch.int64
        assert np.array_equal(got[0].cpu().numpy(), want), t
        assert tuple(batched.hidden_states.shape) == (1, N, H)
        assert PU.rel_err(batched.hidden_states, one.hidden_states) < 1e-5, t
        last = np.eye(A)[want]


@pytest.mark.parametrize("reuse_network", [True, False])
@pytest.mark.parametrize("n,N,A,O", [(64, 5, 11, 80), (32, 8, 14, 128), (16, 27, 36, 285), (7, 3, 5, 4), (257, 3, 5, 4),
                                     (7, 2, 3, 1), (1, 27, 36, 285)])
def test_act_matches_fp64_oracle_over_five_steps(n, N, A, O, reuse_network):
    """q and h' within 1e-5 of the fp64 oracle's unroll with the per-agent parameter list, carried over 5 consecutive
    calls; greedy actions exact except where the fp64 top-2 gap is below 1e-5; random availability masks, agent 0 with
    nothing available (action 0)."""
    mac = _sep(N, A, O, reuse_network=reuse_network, seed=n + N)
    p = _f64_params(mac)
    cfg = MO.make_cfg(n_agents=N, n_actions=A, obs_shape=O, last_action=True, reuse_network=reuse_network, separated=True)
    rng = np.random.RandomState(n * 31 + A)
    T = 5
    obs = rng.randn(n, T, N, O)
    last = rng.rand(n, T, N, A)                            # any float vector is accepted where the last action goes
    avail = (rng.rand(n, T, N, A) < 0.6).astype(np.float64)
    avail[:, :, 0, :] = 0.0
    oq, oh, _ = MO.unroll(p, torch.as_tensor(obs), torch.as_tensor(last), torch.zeros(n * N, H, dtype=torch.float64), cfg)
    dev = "cuda"
    hidden = torch.zeros(n * N, H, device=dev)
    for t in range(T):
        q = torch.empty(n, N, A, device=dev)
        t32 = lambda x: torch.as_tensor(x[:, t], dtype=torch.float32, device=dev).contiguous()
        act = mac.act(n, t32(obs), t32(last), t32(avail), hidden, q=q)
        assert PU.rel_err(q, oq[:, t]) < 1e-5, t
        assert PU.rel_err(hidden.view(n, N, H), oh[:, t]) < 1e-5, t
        masked = np.where(avail[:, t] == 0, -np.inf, oq[:, t].numpy()).reshape(n * N, A)
        _, hard = PU.argmax_mismatches(act, masked, masked.argmax(1))
        assert hard == 0, t
        assert np.all(act[:, 0].cpu().numpy() == 0)


def _inputs(n, N, A, O, seed):
    rng = np.random.RandomState(seed)
    dev = "cuda"
    t = lambda x: torch.as_tensor(x, dtype=torch.float32, device=dev).contiguous()
    avail = (rng.rand(n, N, A) < 0.5).astype(np.float32)
    avail[::5, 0, :] = 0.0
    return t(rng.randn(n, N, O)), t(np.eye(A)[rng.randint(0, A, (n, N))]), t(avail), avail, rng


def test_each_row_uses_its_own_agents_weights():
    """Reversing the agents' weights and the agent axis of every input reverses the outputs (reuse_network=False: no
    agent-id input tells the rows apart); all agents on one shared network's weights reproduce SharedMAC.act."""
    from marl_b200.controller.share_params import SharedMAC
    n, N, A, O = 100, 6, 9, 20
    fwd = _sep(N, A, O, seed=3)
    rev = _sep(N, A, O, seed=4)
    for i, net in enumerate(rev.agent):
        net.load_state_dict(fwd.agent[N - 1 - i].state_dict())
    obs, last, avail_d, _, _ = _inputs(n, N, A, O, 3)
    h0 = torch.randn(n, N, H, device="cuda") * 0.5
    outs = []
    for mac, flip in ((fwd, False), (rev, True)):
        f = (lambda x: x.flip(1).contiguous()) if flip else (lambda x: x)
        q = torch.empty(n, N, A, device="cuda")
        h = f(h0).reshape(n * N, H).clone()
        act = mac.act(n, f(obs), f(last), f(avail_d), h, q=q)
        outs.append((f(act), f(q), f(h.view(n, N, H))))
    for x, y in zip(*outs):
        assert torch.equal(x, y)
    # identical weights in every agent, agent-id input on: the shared controller's launch
    torch.manual_seed(5)
    shared = SharedMAC(PU.make_args("qmix", N, A, O, 4, 10))
    same = _sep(N, A, O, reuse_network=True, seed=6)
    same.load_state(shared)
    res = []
    for mac in (shared, same):
        q = torch.empty(n, N, A, device="cuda")
        h = h0.reshape(n * N, H).clone()
        res.append((mac.act(n, obs, last, avail_d, h, q=q), q, h))
    assert torch.equal(res[0][0], res[1][0])
    assert PU.rel_err(res[1][1], res[0][1]) < 1e-6 and PU.rel_err(res[1][2], res[0][2]) < 1e-6


def test_uniform_exploration_follows_the_floor_rule():
    n, N, A, O = 300, 4, 9, 6
    mac = _sep(N, A, O)
    obs, last, avail_d, avail, rng = _inputs(n, N, A, O, 1)
    eu, cu = rng.rand(n, N), rng.rand(n, N)
    eps = 0.5
    h0 = torch.randn(n * N, H, device="cuda") * 0.5
    greedy = mac.act(n, obs, last, avail_d, h0.clone()).cpu().numpy()
    mac.init_hidden(n)
    mac.hidden_states.copy_(h0.view(n, N, H))
    got = mac.choose_actions(obs, last, avail_d, eps, draws=(eu, cu)).cpu().numpy()
    assert tuple(mac.hidden_states.shape) == (n, N, H)
    cnt = avail.sum(-1)
    kth = np.minimum(np.floor(cu * cnt), cnt - 1)
    want = np.where(cnt > 0, ((np.cumsum(avail, -1) == (kth + 1)[..., None]) & (avail > 0)).argmax(-1), 0)
    explored = eu < eps
    assert explored.mean() > 0.3 and (~explored).mean() > 0.3
    assert np.array_equal(got[explored], want[explored])
    assert np.array_equal(got[~explored], greedy[~explored])
    taken = np.take_along_axis(avail, got[..., None], -1)[..., 0]
    assert np.all(taken[cnt > 0] == 1)
    assert np.all(got[cnt == 0] == 0) and (cnt == 0).sum() >= n // 5
    outs = []
    for _ in range(2):
        mac.hidden_states.copy_(h0.view(n, N, H))
        torch.manual_seed(5)
        outs.append(mac.choose_actions(obs, last, avail_d, eps).cpu().numpy())
    assert np.array_equal(outs[0], outs[1])


def test_flag_exploration_reproduces_epsgreedy_select():
    n, N, A, O = 129, 3, 7, 5
    mac = _sep(N, A, O)
    obs, last, avail_d, avail, rng = _inputs(n, N, A, O, 2)
    dev = "cuda"
    explore = torch.as_tensor((rng.rand(n, N) < 0.4).astype(np.uint8), device=dev)
    rand_a = torch.as_tensor(rng.randint(0, A, (n, N)), dtype=torch.int64, device=dev)
    q = torch.empty(n, N, A, device=dev)
    onehot = torch.empty(n, N, A, device=dev)
    hidden = torch.zeros(n * N, H, device=dev)
    got = mac.act(n, obs, last, avail_d, hidden, explore=explore, random_action=rand_a, q=q, onehot=onehot)
    want = torch.empty(n * N, dtype=torch.int64, device=dev)
    want_oh = torch.empty(n * N, A, device=dev)
    L.call("marl_epsgreedy_select", n * N, A, q.data_ptr(), avail_d.data_ptr(), explore.data_ptr(), rand_a.data_ptr(),
           want.data_ptr(), want_oh.data_ptr(), L.stream_ptr())
    assert torch.equal(got.view(-1), want) and torch.equal(onehot.view(-1, A), want_oh)


def test_bad_calls_raise():
    n, N, A, O = 9, 3, 7, 5
    mac = _sep(N, A, O)
    obs, last, avail_d, _, _ = _inputs(n, N, A, O, 4)
    hidden = torch.zeros(n * N, H, device="cuda")
    u = torch.rand(n, N, dtype=torch.float64, device="cuda")
    flags = torch.zeros(n, N, dtype=torch.uint8, device="cuda")
    with pytest.raises(ValueError):                        # both exploration forms at once
        mac.act(n, obs, last, avail_d, hidden, explore=flags, random_action=u.long(), explore_u=u, choice_u=u, eps=0.5)
    with pytest.raises(ValueError):                        # last_action is on: the last action is required
        mac.act(n, obs, None, avail_d, hidden)
    mac.init_hidden(n)
    for bad in ((obs[:, :2], last, avail_d), (obs, last[..., :3], avail_d), (obs, last, avail_d[:2]), (obs, None, avail_d)):
        with pytest.raises(ValueError):
            mac.choose_actions(*bad, 0.5)
    mac.init_hidden(n + 1)
    with pytest.raises(ValueError):                        # hidden state of another instance count
        mac.choose_actions(obs, last, avail_d, 0.5)
    # one agent's 64 x (O + A) fc1 weights beyond one block's shared memory: MARL_EINVAL, as marl_agent_act refuses it
    big = _sep(2, 4, 1000)
    with pytest.raises(ValueError):
        big.act(1, torch.zeros(1, 2, 1000, device="cuda"), torch.zeros(1, 2, 4, device="cuda"), None,
                torch.zeros(2, H, device="cuda"))


# ------------------------------------------------------------------------------------------ the batched rollout
PAYOFF1 = [[8, -12, -12], [-12, 0, 0], [-12, 0, 0]]


@pytest.mark.parametrize("last_action", [True, False])
@pytest.mark.parametrize("epsilon", [1.0, 0.3, 0.0])
def test_matrix_game_matches_sequential_oracle(epsilon, last_action):
    """BatchedRolloutWorker with a SeparatedMAC (reuse_network=False, runner.py:24-26) against the sequential rollout with
    per-agent networks under the same numpy seed: actions, float64 rewards and the epsilon left behind, bit for bit."""
    from marl_b200.env.single_state_matrix_game import BatchedMatrixGame
    from marl_b200.rollout import BatchedRolloutWorker
    n = 257
    mac = _sep(2, 3, 1, last_action=last_action, seed=7, S=1, T=1)
    args = mac.args
    args.epsilon, args.anneal_epsilon = epsilon, 0.01
    env = BatchedMatrixGame(PAYOFF1, n, keep_r64=True)
    worker = BatchedRolloutWorker(env, mac, args)
    np.random.seed(7)
    episodes, rewards, _, steps = worker.generate_episodes()
    np.random.seed(7)
    agents = [{k: v.detach().cpu() for k, v in net.state_dict().items()} for net in mac.agent]
    want_u, want_r, want_eps = SRO.generate_episodes(agents, PAYOFF1, n, epsilon, 0.01, args.min_epsilon, "step",
                                                    last_action=last_action, reuse_network=False)
    assert np.array_equal(episodes["u"].reshape(n, 2).cpu().numpy(), want_u)
    assert np.array_equal(env.r64.cpu().numpy(), want_r)
    assert worker.epsilon == want_eps and steps == n


KEYS11 = ("o", "s", "u", "r", "avail_u", "o_next", "s_next", "avail_u_next", "u_onehot", "padded", "terminated")


def _multistep_worker(T, n, seed=8):
    from marl_b200.rollout import BatchedRolloutWorker
    from tests.envs import CountdownGameBatched
    N, A, O, S = 3, 5, 4, 3
    mac = _sep(N, A, O, seed=seed, S=S, T=T)
    args = mac.args
    args.epsilon, args.anneal_epsilon, args.min_epsilon, args.epsilon_anneal_scale = 0.5, 0.01, 0.02, "step"
    return BatchedRolloutWorker(CountdownGameBatched(n, n_agents=N, n_actions=A, episode_limit=T), mac, args)


def _oracle_rollout(worker, n, draws):
    from tests.envs import CountdownGameHost
    a = worker.args
    agents = [{k: v.detach().cpu() for k, v in net.state_dict().items()} for net in worker.mac.agent]
    return SRO.rollout_multistep(agents, CountdownGameHost(n_agents=a.n_agents, n_actions=a.n_actions,
                                                          episode_limit=a.episode_limit),
                                n, 0.5, 0.01, 0.02, "step", draws=draws, last_action=True, reuse_network=False)


def _check_against_oracle(worker, n, seed):
    N, T = worker.n_agents, worker.episode_limit
    rng = np.random.RandomState(seed)
    draws = (rng.rand(n, T, N), rng.rand(n, T, N))
    worker.epsilon = 0.5
    ep, rewards, _, steps = worker.generate_episodes(draws=draws)
    oep, orew, osteps = _oracle_rollout(worker, n, draws)
    for k in KEYS11:
        assert np.array_equal(ep[k].cpu().numpy().astype(np.float64), oep[k]), k
    assert np.array_equal(rewards.cpu().numpy(), np.array(orew)) and steps == osteps
    explored = (draws[0] < 0.5)[oep["padded"][:, :, 0] == 0].mean()
    assert explored > 0.2
    return ep


def test_multistep_rollout_to_buffer_to_learner_matches_oracle():
    """Exploring multi-step episodes under host draws: all 11 keys, rewards and the step count equal the sequential
    rollout with per-agent networks; they go through store_episode -> sample -> QLearner(SeparatedMAC).train, whose loss
    matches the oracle's separated train step (1e-5 on the first step, 5e-5 after, like the separated learner test); a
    rollout after training acts on the trained weights the learner re-packed into its flat buffer."""
    from marl_b200.algorithm.q_learner import QLearner
    from marl_b200.common.replaybuffer import ReplayBuffer
    n = 64
    worker = _multistep_worker(6, n)
    args = worker.args
    ep = _check_against_oracle(worker, n, 1)
    args.buffer_size = 256
    buf = ReplayBuffer(args)
    buf.store_episode(ep)
    learner = QLearner(worker.mac, args)
    cfg = PU.oracle_cfg(args)
    cfg.separated, cfg.last_action, cfg.reuse_network = True, True, False
    params = {f"agent.{i}": {k: v.detach().cpu() for k, v in net.state_dict().items()} for i, net in enumerate(worker.mac.agent)}
    params["mixer"] = {k: v.detach().cpu() for k, v in learner.mixer.state_dict().items()}
    st = MO.LearnerState(cfg, params)
    host = {k: v.cpu().numpy().astype(np.float64) for k, v in buf.buffers.items()}
    np.random.seed(0)
    for step in range(3):
        view = buf.sample(32)
        batch = {k: host[k][view.idx_host] for k in host}
        loss = learner.train(view, step)
        oloss, _ = MO.train_step(st, batch, step)
        assert abs(loss - oloss) <= (1e-5 if step == 0 else 5e-5) * abs(oloss), (step, loss, oloss)
    _check_against_oracle(worker, n, 2)                    # the learner's trained, re-packed weights


def _syncs(worker, draws):
    worker.epsilon = 0.5
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        torch.cuda.set_sync_debug_mode("warn")
        try:
            worker.generate_episodes(draws=draws)
        finally:
            torch.cuda.set_sync_debug_mode("default")
    return sum("called a synchronizing" in str(x.message) for x in w)


def test_multistep_step_loop_does_not_synchronise_per_step():
    counts = []
    for T in (6, 60):
        worker = _multistep_worker(T, 64)
        rng = np.random.RandomState(T)
        draws = tuple(torch.as_tensor(rng.rand(64, T, worker.n_agents), device="cuda") for _ in range(2))
        worker.generate_episodes(draws=draws)                # first call: one-time allocations
        counts.append(_syncs(worker, draws))
    assert counts[0] == counts[1] == 1, counts                 # the final read of the step counter


def test_multistep_launches_separated_act_once_per_step_and_one_other_kernel():
    worker = _multistep_worker(6, 64)
    env_steps = []
    step = worker.env.step
    worker.env.step = lambda a, act: env_steps.append(1) or step(a, act)
    worker.generate_episodes()
    torch.cuda.synchronize()
    L.profile(True)
    try:
        L.profile_collect()
        env_steps.clear()
        worker.generate_episodes()
        torch.cuda.synchronize()
        launches = L.profile_collect()
    finally:
        L.profile(False)
    k = len(env_steps)
    assert 1 <= k <= 6 and launches["agent_act_separated_kernel"][0] == k, (k, launches)
    assert "agent_act_kernel" not in launches, launches
    assert sum(c for name, (c, _) in launches.items() if name != "agent_act_separated_kernel") <= k, launches
