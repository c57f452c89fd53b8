"""Batched on-device acting (SharedMAC.choose_actions / marl_agent_act) and the multi-step rollout built on it
(marl_rollout_record): parity with the single-agent call and the fp64 oracle, the exploration contract, and a step
loop that neither synchronises with the host per step nor launches more than two library kernels per step."""
import warnings

import numpy as np
import pytest
import torch

from marl_b200 import _lib as L
from oracle import marl_oracle as MO
from tests import golden_util as GU
from tests import parity_util as PU

pytestmark = pytest.mark.gpu
H = 64


def _mac(N, A, O, seed=0, T=10):
    from marl_b200.controller.share_params import SharedMAC
    torch.manual_seed(seed)
    return SharedMAC(PU.make_args("qmix", N, A, O, 4, T))


def _f64_params(mac):
    return {k: v.detach().cpu().double() for k, v in mac.agent.state_dict().items()}


def test_greedy_choose_actions_matches_choose_action_loop():
    """The reference's literal 3s5z inputs (golden choose_action_3s5z): one choose_actions call per step gives the actions
    of choose_action looped over the agents, greedy, and the same carried hidden state."""
    z = GU.load("choose_action_3s5z")
    N, A, O = (int(x) for x in z["meta/dims"])
    macs = [_mac(N, A, O) for _ in range(2)]
    for m in macs:
        m.agent.load_state_dict(GU.group(z, "init/agent"))
        m.init_hidden(1)
    one, batched = macs
    last = np.zeros((N, A))
    for t in range(z["obs"].shape[0]):
        want = np.array([int(one.choose_action(z["obs"][t, a], last[a], a, z["avail"][t, a], 0.0)) for a in range(N)])
        got = batched.choose_actions(z["obs"][t][None], last[None], z["avail"][t][None], 0.0, evaluate=True)
        assert tuple(got.shape) == (1, N) and got.dtype == torch.int64
        assert np.array_equal(got[0].cpu().numpy(), want), t
        assert tuple(batched.hidden_states.shape) == (1, N, H)
        assert PU.rel_err(batched.hidden_states, one.hidden_states) < 1e-5, t
        last = np.eye(A)[want]


@pytest.mark.parametrize("n,N,A,O", [(64, 5, 11, 80), (32, 8, 14, 128), (16, 27, 36, 285), (7, 3, 5, 4), (257, 3, 5, 4),
                                     (7, 2, 3, 1)])
def test_act_matches_fp64_oracle_over_five_steps(n, N, A, O):
    """q and h' within 1e-5 of the fp64 oracle's unroll, carried over 5 consecutive calls; greedy actions exact except
    where the fp64 top-2 gap is below 1e-5; random availability masks including rows with nothing available."""
    mac = _mac(N, A, O, seed=n + N)
    p = _f64_params(mac)
    rng = np.random.RandomState(n * 31 + A)
    T = 5
    obs = rng.randn(n, T, N, O)
    last = rng.rand(n, T, N, A)                            # any float vector is accepted where the last action goes
    avail = (rng.rand(n, T, N, A) < 0.6).astype(np.float64)
    avail[:, :, 0, :] = 0.0                               # agent 0 never has an available action
    oq, _, _ = MO.unroll(p, torch.as_tensor(obs), torch.as_tensor(last), torch.zeros(n * N, H, dtype=torch.float64), None)
    dev = "cuda"
    hidden = torch.zeros(n * N, H, device=dev)
    h64 = torch.zeros(n * N, H, dtype=torch.float64)
    for t in range(T):
        q = torch.empty(n, N, A, device=dev)
        o_t = torch.as_tensor(obs[:, t], dtype=torch.float32, device=dev).contiguous()
        l_t = torch.as_tensor(last[:, t], dtype=torch.float32, device=dev).contiguous()
        a_t = torch.as_tensor(avail[:, t], dtype=torch.float32, device=dev).contiguous()
        act = mac.act(n, o_t, l_t, a_t, hidden, q=q)
        x = torch.cat([torch.as_tensor(obs[:, t]).reshape(n * N, O), torch.as_tensor(last[:, t]).reshape(n * N, A),
                       torch.eye(N, dtype=torch.float64).repeat(n, 1)], 1)
        q64, h64 = MO.agent_step(p, x, h64)
        assert PU.rel_err(q, oq[:, t]) < 1e-5 and PU.rel_err(q, q64.view(n, N, A)) < 1e-5, t
        assert PU.rel_err(hidden, h64) < 1e-5, t
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


def test_uniform_exploration_follows_the_floor_rule():
    n, N, A, O = 300, 4, 9, 6
    mac = _mac(N, A, O)
    obs, last, avail_d, avail, rng = _inputs(n, N, A, O, 1)
    eu, cu = rng.rand(n, N), rng.rand(n, N)
    eps = 0.5
    h0 = torch.randn(n * N, H, device="cuda") * 0.5
    greedy = mac.act(n, obs, last, avail_d, h0.clone()).cpu().numpy()
    mac.init_hidden(n)
    mac.hidden_states.copy_(h0.view(n, N, H))
    got = mac.choose_actions(obs, last, avail_d, eps, draws=(eu, cu)).cpu().numpy()
    cnt = avail.sum(-1)
    kth = np.minimum(np.floor(cu * cnt), cnt - 1)
    want = np.where(cnt > 0, ((np.cumsum(avail, -1) == (kth + 1)[..., None]) & (avail > 0)).argmax(-1), 0)
    explored = eu < eps
    assert explored.mean() > 0.3 and (~explored).mean() > 0.3
    assert np.array_equal(got[explored], want[explored])
    assert np.array_equal(got[~explored], greedy[~explored])
    taken = np.take_along_axis(avail, got[..., None], -1)[..., 0]
    assert np.all(taken[cnt > 0] == 1)                     # never an unavailable action
    assert np.all(got[cnt == 0] == 0) and (cnt == 0).sum() >= n // 5
    # device draws: torch.manual_seed governs them
    outs = []
    for _ in range(2):
        mac.hidden_states.copy_(h0.view(n, N, H))
        torch.manual_seed(5)
        outs.append(mac.choose_actions(obs, last, avail_d, eps).cpu().numpy())
    assert np.array_equal(outs[0], outs[1])


def test_flag_exploration_reproduces_epsgreedy_select_and_bad_calls_raise():
    n, N, A, O = 129, 3, 7, 5
    mac = _mac(N, A, O)
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
    u = torch.rand(n, N, dtype=torch.float64, device=dev)
    with pytest.raises(ValueError):                        # both exploration forms at once
        mac.act(n, obs, last, avail_d, hidden, explore=explore, random_action=rand_a, explore_u=u, choice_u=u, eps=0.5)
    with pytest.raises(ValueError):
        mac.choose_actions(obs[:, :2], last, avail_d, 0.5)


# ------------------------------------------------------------------------------------------ the multi-step rollout
def _worker(T, n=64):
    from marl_b200.rollout import BatchedRolloutWorker
    from tests.envs import CountdownGameBatched
    z = GU.load("rollout_multistep")
    N, A, O, S, _ = (int(x) for x in z["meta/dims"])
    args = PU.make_args("qmix", N, A, O, S, T)
    args.epsilon, args.anneal_epsilon, args.min_epsilon, args.epsilon_anneal_scale = 0.5, 0.01, 0.02, "step"
    from marl_b200.controller.share_params import SharedMAC
    mac = SharedMAC(args)
    mac.agent.load_state_dict(GU.group(z, "init/agent"))
    return BatchedRolloutWorker(CountdownGameBatched(n, n_agents=N, n_actions=A, episode_limit=T), mac, args)


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
        worker = _worker(T)
        rng = np.random.RandomState(T)
        draws = tuple(torch.as_tensor(rng.rand(64, T, worker.n_agents), device="cuda") for _ in range(2))
        worker.generate_episodes(draws=draws)                # first call: one-time allocations
        counts.append(_syncs(worker, draws))
    assert counts[0] == counts[1] == 1, counts                 # the final read of the step counter


def test_multistep_launches_act_once_per_step_and_one_other_kernel():
    worker = _worker(6)
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
    assert 1 <= k <= 6 and launches["agent_act_kernel"][0] == k, (k, launches)
    assert sum(c for name, (c, _) in launches.items() if name != "agent_act_kernel") <= k, launches


def _pre_change_loop(worker, draws):
    """The multi-step loop as it stood before marl_agent_act: mac.agent.unroll + torch exploration + marl_epsgreedy_select,
    with a host synchronisation per step.  Returns the final hidden state and the actions."""
    env, mac, dev = worker.env, worker.mac, "cuda"
    n, N, A, T = env.n_envs, worker.n_agents, worker.n_actions, worker.episode_limit
    explore_u, choice_u = (torch.as_tensor(d, dtype=torch.float64, device=dev) for d in draws)
    eps = float(worker.epsilon)
    env.reset()
    hidden = torch.zeros(n * N, H, device=dev)
    last = torch.zeros(n, N, A, device=dev)
    active = torch.ones(n, dtype=torch.bool, device=dev)
    us = torch.zeros(n, T, N, dtype=torch.int64, device=dev)
    with torch.no_grad():
        for t in range(T):
            obs, avail = env.get_obs(), env.get_avail_actions()
            if int(active.sum().item()) == 0:
                break
            q, _, hidden = mac.agent.unroll(obs.unsqueeze(1).contiguous(), last.unsqueeze(1).contiguous(), hidden, 0)
            explore = (explore_u[:, t] < eps).to(torch.uint8).contiguous()
            cnt = avail.sum(-1).to(torch.float64)
            kth = torch.minimum((choice_u[:, t] * cnt).floor(), cnt - 1)
            rand_a = ((avail.cumsum(-1).to(torch.float64) == (kth + 1).unsqueeze(-1)) & (avail > 0)).to(torch.uint8).argmax(-1)
            actions = torch.empty(n, N, dtype=torch.int64, device=dev)
            onehot = torch.empty(n, N, A, device=dev)
            L.call("marl_epsgreedy_select", n * N, A, q.reshape(n * N, A).contiguous().data_ptr(), avail.contiguous().data_ptr(),
                   explore.data_ptr(), rand_a.contiguous().data_ptr(), actions.data_ptr(), onehot.data_ptr(), L.stream_ptr())
            _, term = env.step(actions, active)
            us[:, t] = torch.where(active.view(n, 1), actions, us[:, t])
            last = torch.where(active.view(n, 1, 1), onehot, last)
            active = active & ~term
            eps = eps - worker.anneal_epsilon if eps > worker.min_epsilon else eps
    return hidden, us


@pytest.mark.parametrize("T", [6, 40])
def test_multistep_hidden_state_matches_pre_change_loop(T):
    worker = _worker(T, n=97)
    rng = np.random.RandomState(11)
    draws = (rng.rand(97, T, worker.n_agents), rng.rand(97, T, worker.n_agents))
    h_old, u_old = _pre_change_loop(worker, draws)
    worker.epsilon = 0.5
    ep, _, _, _ = worker.generate_episodes(draws=draws)
    assert tuple(worker.mac.hidden_states.shape) == (97 * worker.n_agents, H)
    assert PU.rel_err(worker.mac.hidden_states, h_old) < 1e-5
    assert torch.equal(ep["u"][..., 0], u_old)
