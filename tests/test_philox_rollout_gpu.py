"""Philox exploration drawn inside the act launch (marl_agent_act_philox / marl_agent_act_separated_philox,
PhiloxDraws, BatchedRolloutWorker rng="philox"): the generator against numpy's np.random.Philox bit for bit, the act
launch against the uniform form fed the same numbers, the matrix game and the multi-step game against the host-drawn
forms and the sequential restatement, episode ids that make a sharded run draw what one call draws, the launch and
memory footprint of the rollout, the statistics of the draws at 2^20 rows, and the argument checks."""
import ctypes

import numpy as np
import pytest
import torch
from scipy import stats

from marl_b200 import _lib as L
from marl_b200.controller.share_params import PhiloxDraws
from tests import golden_util as GU
from tests import parity_util as PU

pytestmark = pytest.mark.gpu
H = 64
M64 = (1 << 64) - 1
FLAGS = [(True, True), (True, False), (False, True), (False, False)]      # (last_action, reuse_network)
SHAPES = [(64, 5, 11, 80), (32, 8, 14, 128), (16, 27, 36, 285), (7, 3, 5, 4), (33, 2, 3, 1)]


def np_pair(seed, episode, step, n):
    """numpy's Philox for counter (episode, step, n, 0), key (seed, 0): (explore_u, choice_u) by Generator.random()."""
    c = (episode & M64) | (step << 64) | (n << 128)
    return np.random.Generator(np.random.Philox(counter=(c - 1) % (1 << 256), key=seed)).random(2)


def np_uniforms(seed, base, step, n_envs, N):
    u = np.array([[np_pair(seed, base + e, step, a) for a in range(N)] for e in range(n_envs)])
    return u[..., 0], u[..., 1]


def dev_uniforms(seed, base, step, n_envs, N):
    out = torch.empty(n_envs * N, 2, dtype=torch.float64, device="cuda")
    L.call("marl_philox_uniforms", seed, base, step, n_envs, N, out.data_ptr(), L.stream_ptr())
    return out.view(n_envs, N, 2)


@pytest.mark.parametrize("seed,base,step,n_envs,N", [
    (0, 0, 0, 64, 5), (123, 0, 7, 16, 128), (7, (1 << 32) - 5, 999, 11, 3), (2 ** 63 + 1, M64 - 4, 1000, 9, 4),
    (M64, (1 << 64) - 2, 1, 4, 37), (5, 2 ** 40, 0, 1, 1)])
def test_uniforms_equal_numpy_philox_bit_for_bit(seed, base, step, n_envs, N):
    """Episode ids around 2^32 and 2^64 - 1 (word 0 wraps; numpy's counter - 1 borrows across words), steps up to
    1000, up to 128 agents."""
    got = dev_uniforms(seed, base, step, n_envs, N).cpu().numpy()
    eu, cu = np_uniforms(seed, base, step, n_envs, N)
    assert np.array_equal(got[..., 0].view(np.int64), eu.view(np.int64))
    assert np.array_equal(got[..., 1].view(np.int64), cu.view(np.int64))


# ------------------------------------------------------------------------------------------------------- acting
def _mac(kind, N, A, O, last_action=True, reuse_network=True, seed=0):
    from marl_b200.controller.share_params import SeparatedMAC, SharedMAC
    torch.manual_seed(seed)
    cls = SharedMAC if kind == "shared" else SeparatedMAC
    return cls(PU.make_args("qmix", N, A, O, 4, 10, last_action=last_action, reuse_network=reuse_network))


def _inputs(n, N, A, O, seed):
    rng = np.random.RandomState(seed)
    t = lambda x: torch.as_tensor(x, dtype=torch.float32, device="cuda").contiguous()
    avail = (rng.rand(n, N, A) < 0.5).astype(np.float32)
    avail[::5, 0, :] = 0.0                                 # rows with nothing available
    return t(rng.randn(n, N, O)), t(np.eye(A)[rng.randint(0, A, (n, N))]), t(avail)


def _act_both(mac, n, obs, last, avail, draws, eps, eps_table=None):
    """(actions, onehot, q, h') of the Philox form, then of the uniform form fed numpy-Philox uniforms, from the same
    seeded hidden state."""
    N, A = mac.n_agents, mac.n_actions
    h0 = torch.randn(n * N, H, device="cuda", generator=torch.Generator(device="cuda").manual_seed(n * N)) * 0.5
    last = last if mac.args.last_action else None
    outs = []
    for philox in (True, False):
        hidden, q, oh = h0.clone(), torch.empty(n, N, A, device="cuda"), torch.empty(n, N, A, device="cuda")
        if philox:
            act = mac.act(n, obs, last, avail, hidden, eps=eps, q=q, onehot=oh, philox=draws, eps_table=eps_table)
        else:
            eu, cu = (torch.as_tensor(x, device="cuda").contiguous() for x in np_uniforms(*draws, n, N))
            act = mac.act(n, obs, last, avail, hidden, explore_u=eu, choice_u=cu, eps=eps, q=q, onehot=oh)
        outs.append((act, oh, q, hidden))
    return outs


@pytest.mark.parametrize("kind", ["shared", "separated"])
@pytest.mark.parametrize("last_action,reuse_network", FLAGS)
@pytest.mark.parametrize("n,N,A,O", SHAPES)
def test_act_philox_equals_uniform_form_fed_numpy_philox(kind, last_action, reuse_network, n, N, A, O):
    mac = _mac(kind, N, A, O, last_action, reuse_network, seed=n + A)
    obs, last, avail = _inputs(n, N, A, O, n * 7 + N)
    draws = PhiloxDraws(seed=1000 + n, episode_base=(1 << 32) - n // 2, step=N)
    (pa, po, pq, ph), (ua, uo, uq, uh) = _act_both(mac, n, obs, last, avail, draws, 0.5)
    assert torch.equal(pa, ua) and torch.equal(po, uo) and torch.equal(pq, uq) and torch.equal(ph, uh)
    explored = np_uniforms(*draws, n, N)[0] < 0.5
    assert 0.3 < explored.mean() < 0.7


@pytest.mark.parametrize("kind", ["shared", "separated"])
def test_act_philox_eps_table_gives_each_instance_its_epsilon(kind):
    """Instance e explores with eps_table[min(e, len - 1)]: for every value v of the table, the instances that use v act
    as the uniform form at eps = v does."""
    n, N, A, O = 40, 3, 5, 4
    mac = _mac(kind, N, A, O, seed=3)
    obs, last, avail = _inputs(n, N, A, O, 9)
    draws = PhiloxDraws(seed=77, episode_base=5, step=0)
    table = np.array([1.0, 0.9, 0.6, 0.3, 0.0])            # instances 4 .. n - 1 use 0.0: greedy
    eps_e = table[np.minimum(np.arange(n), len(table) - 1)]
    got = _act_both(mac, n, obs, last, avail, draws, 0.5, eps_table=torch.as_tensor(table, device="cuda"))[0]
    for v in table:
        want = _act_both(mac, n, obs, last, avail, draws, float(v))[1]
        rows = torch.as_tensor(eps_e == v, device="cuda")
        for x, y in zip(got, want):                        # actions, onehot, q, h': instance-major rows
            assert torch.equal(x.view(n, -1)[rows], y.view(n, -1)[rows]), v


@pytest.mark.parametrize("kind", ["shared", "separated"])
@pytest.mark.parametrize("last_action,reuse_network", FLAGS)
def test_choose_actions_philox_on_3s5z_masks(kind, last_action, reuse_network):
    """The reference's literal 3s5z observations and availability masks (golden choose_action_3s5z), one instance per
    recorded step: choose_actions with PhiloxDraws equals choose_actions with draws= from numpy Philox, and the carried
    hidden states agree bit for bit."""
    z = GU.load("choose_action_3s5z")
    N, A, O = (int(x) for x in z["meta/dims"])
    n = z["obs"].shape[0]
    macs = [_mac(kind, N, A, O, last_action, reuse_network, seed=4) for _ in range(2)]
    rng = np.random.RandomState(5)
    last = np.eye(A)[rng.randint(0, A, (n, N))] if last_action else None
    for m in macs:
        m.init_hidden(n)
    for step in range(3):
        draws = PhiloxDraws(seed=int(z["meta/seed"]), episode_base=1 << 20, step=step)
        got = macs[0].choose_actions(z["obs"], last, z["avail"], 0.6, draws=draws)
        want = macs[1].choose_actions(z["obs"], last, z["avail"], 0.6, draws=np_uniforms(*draws, n, N))
        assert torch.equal(got, want), step
        assert torch.equal(macs[0].hidden_states, macs[1].hidden_states), step
        taken = np.take_along_axis(z["avail"], got.cpu().numpy()[..., None], -1)[..., 0]
        assert np.all(taken[z["avail"].sum(-1) > 0] == 1)


@pytest.mark.parametrize("last_action,reuse_network", FLAGS)
def test_separated_with_equal_weights_reproduces_shared_philox_actions(last_action, reuse_network):
    n, N, A, O = 97, 5, 11, 80
    shared = _mac("shared", N, A, O, last_action, reuse_network, seed=8)
    sep = _mac("separated", N, A, O, last_action, reuse_network, seed=9)
    sep.load_state(shared)                                 # one network copied into every agent
    obs, last, avail = _inputs(n, N, A, O, 12)
    draws = PhiloxDraws(seed=31, episode_base=M64 - 40, step=3)
    a, b = (_act_both(m, n, obs, last, avail, draws, 0.4)[0] for m in (shared, sep))
    for x, y in zip(a, b):
        assert torch.equal(x, y)


# ------------------------------------------------------------------------------------------------- the matrix game
PAYOFF1 = [[8, -12, -12], [-12, 0, 0], [-12, 0, 0]]


def _matrix(n, **kw):
    from marl_b200.env.single_state_matrix_game import BatchedMatrixGame
    from marl_b200.rollout import BatchedRolloutWorker
    args = PU.make_args("qmix", 2, 3, 1, 1, 1, **kw)
    learner, _ = PU.build_pair(args)
    return BatchedRolloutWorker(BatchedMatrixGame(PAYOFF1, n, keep_r64=True), learner.eval_net, args), learner


def _matrix_want(worker, greedy, n, base):
    """Actions from the greedy joint action, numpy-Philox uniforms and _epsilons (every action of the game available)."""
    eps, after = worker._epsilons(n, False)
    eu, cu = np_uniforms(worker.args.seed, base, 0, n, 2)
    rand = np.minimum(np.floor(cu * 3), 2).astype(np.int64)
    return np.where(eu < eps[:, None], rand, greedy[None, :]), after


@pytest.mark.parametrize("scale", ["step", "episode"])
@pytest.mark.parametrize("epsilon,anneal,min_eps", [(0.6, 0.0, 0.05), (0.3, 0.01, 0.05)])   # the second crosses min
def test_matrix_game_philox_actions(scale, epsilon, anneal, min_eps):
    n = 257
    worker, learner = _matrix(n, epsilon=epsilon, epsilon_anneal_scale=scale)
    worker.anneal_epsilon, worker.min_epsilon = anneal, min_eps
    g, _, _, _ = worker.generate_episodes(evaluate=True)
    greedy = g["u"].reshape(n, 2)[0].cpu().numpy()
    worker.episode_base = 0
    for call in range(2):                                  # the second call plays episodes n .. 2n - 1
        want, after = _matrix_want(worker, greedy, n, call * n)
        ep, rewards, _, steps = worker.generate_episodes(rng="philox")
        got = ep["u"].reshape(n, 2).cpu().numpy()
        assert np.array_equal(got, want), call
        assert worker.epsilon == after and worker.episode_base == (call + 1) * n and steps == n
        assert np.array_equal(rewards.cpu().numpy(), np.array(PAYOFF1, dtype=np.float32)[got[:, 0], got[:, 1]])
    assert (worker.epsilon <= min_eps) == (anneal > 0)


def test_matrix_game_philox_two_shards_reproduce_one_worker():
    n = 512
    one, learner = _matrix(n, epsilon=0.5)
    halves = []
    for g in range(2):
        w, _ = _matrix(n // 2, epsilon=0.5)
        w.mac.load_state(one.mac)
        halves.append(w)
    for w in (one, *halves):
        w.anneal_epsilon = 0.0
    for rnd in range(2):
        for g, w in enumerate(halves):
            w.episode_base = rnd * n + g * (n // 2)        # global episodes so far + g * n_local
        full = one.generate_episodes(rng="philox")[0]["u"].reshape(n, 2)
        parts = torch.cat([w.generate_episodes(rng="philox")[0]["u"].reshape(n // 2, 2) for w in halves])
        assert torch.equal(full, parts), rnd


def test_matrix_game_philox_evaluate_is_greedy_and_keeps_epsilon():
    worker, _ = _matrix(64, epsilon=0.9)
    ep, _, _, _ = worker.generate_episodes(evaluate=True, rng="philox")
    u = ep["u"].reshape(64, 2)
    assert bool((u == u[0]).all()) and worker.epsilon == 0.9


def test_rng_argument_errors():
    worker, _ = _matrix(8, epsilon=0.5)
    with pytest.raises(ValueError):
        worker.generate_episodes(rng="philox", draws=(np.zeros((8, 1, 2)), np.zeros((8, 1, 2))))
    with pytest.raises(ValueError):
        worker.generate_episodes(rng="Philox")
    ms, _ = _multistep(7)
    with pytest.raises(ValueError):
        ms.generate_episodes(rng="philox", draws=(np.zeros((7, 6, 3)), np.zeros((7, 6, 3))))
    with pytest.raises(ValueError):
        ms.generate_episodes(rng="counter")


def test_null_descriptor_and_bad_eps_len_are_einval():
    n, N, A, O = 4, 3, 5, 4
    mac = _mac("shared", N, A, O)
    obs, last, avail = _inputs(n, N, A, O, 1)
    hidden, act = torch.zeros(n * N, H, device="cuda"), torch.empty(n, N, dtype=torch.int64, device="cuda")
    from marl_b200.network.q_network import agent_param_struct
    p = agent_param_struct(mac.agent.param_addresses())
    table = torch.ones(3, dtype=torch.float64, device="cuda")
    bad = [None, ctypes.byref(L.ActPhilox(1, 0, 0, table.data_ptr(), 0)), ctypes.byref(L.ActPhilox(1, 0, -1, None, 0))]
    for fn, params in (("marl_agent_act_philox", ctypes.byref(p)), ("marl_agent_act_separated_philox", (L.AgentParams * N)(p, p, p))):
        for d in bad:
            with pytest.raises(ValueError):
                L.call(fn, n, N, A, O, 1, 1, params, obs.data_ptr(), last.data_ptr(), avail.data_ptr(), hidden.data_ptr(),
                       hidden.data_ptr(), d, 0.5, None, act.data_ptr(), None, None, L.stream_ptr())
        good = ctypes.byref(L.ActPhilox(1, 0, 0, table.data_ptr(), 3))
        L.call(fn, n, N, A, O, 1, 1, params, obs.data_ptr(), last.data_ptr(), avail.data_ptr(), hidden.data_ptr(),
               hidden.data_ptr(), good, 0.5, None, act.data_ptr(), None, None, L.stream_ptr())
    with pytest.raises(ValueError):                        # the flag / uniform arrays do not go with philox=
        mac.act(n, obs, last, avail, hidden, explore_u=table, choice_u=table, philox=PhiloxDraws(1))
    with pytest.raises(ValueError):
        mac.act(n, obs, last, avail, hidden, eps_table=table)


# ------------------------------------------------------------------------------------------------- multi-step
KEYS11 = ("o", "s", "u", "r", "avail_u", "o_next", "s_next", "avail_u_next", "u_onehot", "padded", "terminated")


def _multistep(n):
    from marl_b200.controller.share_params import SharedMAC
    from marl_b200.rollout import BatchedRolloutWorker
    from tests.envs import CountdownGameBatched
    z = GU.load("rollout_multistep")
    N, A, O, S, T = (int(x) for x in z["meta/dims"])
    args = PU.make_args("qmix", N, A, O, S, T)
    args.epsilon, args.anneal_epsilon, args.min_epsilon, args.epsilon_anneal_scale = 0.5, 0.01, 0.02, "step"
    mac = SharedMAC(args)
    mac.agent.load_state_dict(GU.group(z, "init/agent"))
    return BatchedRolloutWorker(CountdownGameBatched(n, n_agents=N, n_actions=A, episode_limit=T), mac, args), args


def _np_draws(seed, base, n, T, N):
    per_t = [np_uniforms(seed, base, t, n, N) for t in range(T)]
    return tuple(np.stack([u[i] for u in per_t], 1) for i in range(2))       # [n, T, N] each


@pytest.mark.parametrize("n", [7, 64])
def test_multistep_philox_equals_draws_form_and_sequential_oracle(n):
    from oracle import rollout_oracle as RO
    from tests.envs import CountdownGameHost
    z = GU.load("rollout_multistep")
    px, args = _multistep(n)
    ref, _ = _multistep(n)
    N, A, T = args.n_agents, args.n_actions, args.episode_limit
    for call in range(2):                                  # the second call draws episodes n .. 2n - 1
        draws = _np_draws(args.seed, call * n, n, T, N)
        ep, rewards, _, steps = px.generate_episodes(rng="philox")
        rep, rrewards, _, rsteps = ref.generate_episodes(draws=draws)
        for k in KEYS11:
            assert torch.equal(ep[k], rep[k]), (call, k)
        assert torch.equal(rewards, rrewards) and steps == rsteps and px.epsilon == ref.epsilon
        assert px.episode_base == (call + 1) * n
    oep, orew, osteps = RO.rollout_multistep(GU.group(z, "init/agent"), CountdownGameHost(n_agents=N, n_actions=A, episode_limit=T),
                                             n, ref.epsilon, 0.01, 0.02, "step", draws=_np_draws(args.seed, 2 * n, n, T, N))
    ep, rewards, _, steps = px.generate_episodes(rng="philox")
    for k in KEYS11:
        assert np.array_equal(ep[k].cpu().numpy().astype(np.float64), oep[k]), k
    assert np.array_equal(rewards.cpu().numpy(), np.array(orew)) and steps == osteps


def test_multistep_philox_one_act_launch_per_step_and_no_draw_arrays():
    worker, args = _multistep(4096)
    env_steps = []
    step = worker.env.step
    worker.env.step = lambda a, act: env_steps.append(1) or step(a, act)
    peaks = {}
    for rng in ("device", "philox", "device", "philox"):    # the second round is the measured one
        worker.epsilon = 0.5
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        if rng == "philox":
            L.profile(True)
            L.profile_collect()
            env_steps.clear()
        try:
            worker.generate_episodes(rng=rng)
            torch.cuda.synchronize()
            launches = L.profile_collect() if rng == "philox" else None
        finally:
            L.profile(False)
        peaks[rng] = torch.cuda.max_memory_allocated() - before
    k = len(env_steps)
    assert 1 <= k <= args.episode_limit and launches["agent_act_kernel"][0] == k, (k, launches)
    assert sum(c for name, (c, _) in launches.items() if name != "agent_act_kernel") <= k, launches
    draw_bytes = 2 * 8 * 4096 * args.episode_limit * args.n_agents    # one [n, T, N] float64 pair
    assert peaks["philox"] + draw_bytes <= peaks["device"], peaks


# ------------------------------------------------------------------------------------------------- statistics
def test_statistics_at_2_pow_20_rows():
    """Exploration rate within 0.005 of epsilon (about 11 standard deviations at 0.25) and the random action uniform over
    the available ones (chi-square per number of available actions), at 2^20 rows; the kernel explores exactly the rows
    whose generator pair says so."""
    n, N, A, O = 1 << 18, 4, 9, 6
    mac = _mac("shared", N, A, O, seed=2)
    rng = np.random.RandomState(3)
    cnt = rng.randint(1, A + 1, (n, N))                    # 1 .. A available actions, at random positions
    avail = (np.argsort(rng.rand(n, N, A), -1) < cnt[..., None]).astype(np.float32)
    t = lambda x: torch.as_tensor(x, dtype=torch.float32, device="cuda").contiguous()
    obs, last, avail_d = t(rng.randn(n, N, O)), t(np.zeros((n, N, A))), t(avail)
    h0 = torch.zeros(n * N, H, device="cuda")
    greedy = mac.act(n, obs, last, avail_d, h0.clone()).cpu().numpy()
    draws = PhiloxDraws(seed=2024, episode_base=3 << 30, step=17)
    got = mac.act(n, obs, last, avail_d, h0.clone(), eps=0.25, philox=draws).cpu().numpy()
    u = dev_uniforms(*draws, n, N).cpu().numpy()
    explored = u[..., 0] < 0.25
    assert abs(explored.mean() - 0.25) < 0.005
    assert np.array_equal(got[~explored], greedy[~explored])
    rank = (np.cumsum(avail, -1) - 1)[np.arange(n)[:, None], np.arange(N)[None, :], got]   # position among the available
    assert np.all(np.take_along_axis(avail, got[..., None], -1)[..., 0] == 1)
    assert np.array_equal(rank[explored], np.minimum(np.floor(u[..., 1] * cnt), cnt - 1)[explored])
    for c in range(2, A + 1):
        r = rank[explored & (cnt == c)]
        observed = np.bincount(r.astype(np.int64), minlength=c)
        assert stats.chisquare(observed).pvalue > 1e-4, (c, observed)
