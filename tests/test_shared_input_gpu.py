"""The shared controller (SharedMAC) with the input blocks the reference's args.last_action / args.reuse_network select
(share_params.py:84-123): the fused learner step against the fp64 oracle and the module path, every route of the input
layers, early exit and graph replay, batched acting, the batched rollout, checkpoints, and the unroll ABI's default input
when a caller leaves marl_unroll_stream.input_flags at 0.  The main case is last_action=False, reuse_network=True."""
import ctypes as C

import numpy as np
import pytest
import torch

from marl_b200 import _lib as L
from marl_b200.synthetic import synthetic_batch
from oracle import marl_oracle as MO
from tests import golden_util as GU
from tests import parity_util as PU
from tests import separated_rollout_oracle as SRO

pytestmark = pytest.mark.gpu
H = 64
TOL = 1e-5
QPLEX_SMALL = dict(num_kernel=2, adv_hypernet_embed=8, hypernet_embed=8)
FLAGS = [(False, True), (True, False), (False, False)]       # (last_action, reuse_network); (True, True) is the default


def _args(alg, N, A, O, S, T, last_action=False, reuse_network=True, **kw):
    base = dict(last_action=last_action, reuse_network=reuse_network, target_update_cycle=2)
    base.update(QPLEX_SMALL if alg == "qplex" else {})
    base.update(kw)
    return PU.make_args(alg, N, A, O, S, T, **base)


def _mac(args, seed=0):
    from marl_b200.controller.share_params import SharedMAC
    torch.manual_seed(seed)
    return SharedMAC(args)


def _learner(args, seed=0):
    from marl_b200.algorithm.q_learner import QLearner
    from marl_b200.algorithm.qtran_learner import QTRANLearner
    learner = (QTRANLearner if args.alg == "qtran_base" else QLearner)(_mac(args, seed), args)
    learner._update_targets()
    return learner


def _oracle(learner, args):
    cfg = PU.oracle_cfg(args)
    cfg.last_action, cfg.reuse_network = args.last_action, args.reuse_network
    return MO.LearnerState(cfg, PU.export_params(learner))


def _width(args):
    return args.obs_shape + args.n_actions * bool(args.last_action) + args.n_agents * bool(args.reuse_network)


# ------------------------------------------------------------------------------------------ the fused learner step
STEP_CASES = [(alg, dq, opt, False, True) for alg in ("vdn", "qmix", "qmix2", "qplex", "qtran_base")
              for dq in (True, False) for opt in ("RMS", "Adam")]
STEP_CASES += [("qmix", True, "RMS", la, rn) for la, rn in ((True, False), (False, False))]


@pytest.mark.parametrize("alg,double_q,optimizer,last_action,reuse_network", STEP_CASES)
def test_fused_step_vs_oracle(alg, double_q, optimizer, last_action, reuse_network):
    """Three steps with a target sync after step 2 against the fp64-checked oracle: loss within 1e-5 at step 0, clipped
    gradients within 5e-5, eval and target parameters with params_close.  O = 8: the obs rows go through the fused input-layer
    kernel's tensor map, and the input width (O + 5 or O + 3 or O) is not a multiple of 4."""
    two = alg == "qmix2"
    alg = "qmix" if two else alg
    N, A, O, S, T, B = 3, 5, 8, 9, 10, 5
    args = _args(alg, N, A, O, S, T, last_action, reuse_network, double_q=double_q, optimizer=optimizer, two_hyper_layers=two)
    learner = _learner(args)
    assert not learner._separated and tuple(learner.eval_net.agent.fc1.weight.shape) == (H, _width(args))
    st = _oracle(learner, args)
    batch = synthetic_batch(3, B, T, N, A, O, S)
    groups = PU.module_groups(learner)
    for step in range(3):
        loss = learner.train({k: v.copy() for k, v in batch.items()}, step)
        oloss, info = MO.train_step(st, batch, step)
        assert abs(loss - oloss) <= (TOL if step == 0 else 5e-5) * abs(oloss), (step, loss, oloss)
        if step == 0:
            for g, m in groups.items():
                for k, p in m.named_parameters():
                    want = info["clipped_grads"].get(f"{g}.{k}")
                    if want is not None:
                        assert PU.rel_err(p.grad, want) < 5e-5, (g, k)
    for g, m in groups.items():
        for k, p in m.named_parameters():
            if info["clipped_grads"].get(f"{g}.{k}") is not None:
                assert PU.params_close(p, st.params[g][k], args.lr, 3), (g, k)
    for k, p in learner.target_net.agent.named_parameters():
        assert PU.params_close(p, st.target["agent"][k], args.lr, 3), k


@pytest.mark.parametrize("last_action,reuse_network", FLAGS)
def test_fused_step_agrees_with_module_path(last_action, reuse_network):
    """The fused step and the same step through RNNQNet.unroll's autograd Function give the same losses and flat gradient."""
    N, A, O, S, T, B = 4, 6, 12, 10, 20, 8
    args = _args("qmix", N, A, O, S, T, last_action, reuse_network)
    batch = synthetic_batch(5, B, T, N, A, O, S)
    out = {}
    for modules in (False, True):
        args.train_through_modules = modules
        learner = _learner(args)
        out[modules] = ([learner.train({k: v.copy() for k, v in batch.items()}, i) for i in range(2)], learner._flat.grad.clone())
    args.train_through_modules = False
    (lf, gf), (lm, gm) = out[False], out[True]
    assert abs(lf[0] - lm[0]) <= 2e-6 * abs(lf[0]) and abs(lf[1] - lm[1]) <= 5e-5 * abs(lf[1]), (lf, lm)
    assert PU.rel_err(gm, gf) < 5e-5


def test_forward_step_matches_the_unroll():
    """SharedMAC.forward(ep_batch, t), step by step, gives the Q-values of get_current_q_values."""
    N, A, O, S, T, B = 3, 5, 8, 4, 6, 4
    mac = _mac(_args("qmix", N, A, O, S, T))
    batch = synthetic_batch(1, B, T, N, A, O, S)
    mac.init_hidden(B)
    q_all, _ = mac.get_current_q_values(batch, T)
    mac.init_hidden(B)
    for t in range(T):
        assert PU.rel_err(mac.forward(batch, t), q_all[:, t]) < 1e-6, t


def _kernels(fn):
    torch.cuda.synchronize()
    L.profile(True)
    try:
        L.profile_collect()
        out = fn()
        torch.cuda.synchronize()
        return out, L.profile_collect()
    finally:
        L.profile(False)


def test_every_input_layer_route_gives_the_same_loss():
    """cfg-2 shape (O = 80, N = 5, no last action: input width 85, not a multiple of 4): the fused input-layer kernel
    (scalar W1 loads) and the separate linear.cu launches (marl_front_enable(0)) give one loss within 1e-6, with the TMA GEMM
    switch off and on.  The switch moves the agent's other dense layers (W_ih, fc2, their gradients) to tgemm.cu, so across
    it the losses agree within that back end's GEMM tolerance (3e-6, tests/test_gemm_gpu.py); all of them match the oracle."""
    N, A, O, S, T, B = 5, 11, 80, 120, 30, 32
    args = _args("qmix", N, A, O, S, T, cuda_graph=False, target_update_cycle=200)
    batch = synthetic_batch(7, B, T, N, A, O, S)
    lib = L.load()
    losses, launches = {}, {}
    for front in (1, 0):
        for tg in (0, 1):
            prev_f, prev_t = lib.marl_front_enable(front), lib.marl_tgemm_enable(tg)
            try:
                learner = _learner(args)
                losses[front, tg], launches[front, tg] = _kernels(lambda: learner.train({k: v.copy() for k, v in batch.items()}, 0))
            finally:
                lib.marl_front_enable(prev_f)
                lib.marl_tgemm_enable(prev_t)
    for tg in (0, 1):
        assert abs(losses[0, tg] - losses[1, tg]) <= 1e-6 * abs(losses[1, tg]), (tg, losses)
    ref = losses[1, 0]
    for key, loss in losses.items():
        assert abs(loss - ref) <= 3e-6 * abs(ref), (key, losses)
    assert "agent_front_kernel" in launches[1, 0] and "agent_front_kernel" in launches[1, 1]
    assert "agent_front_kernel" not in launches[0, 0] and "agent_front_kernel" not in launches[0, 1]
    oloss, _ = MO.train_step(_oracle(_learner(args), args), batch, 0)
    for key, loss in losses.items():
        assert abs(loss - oloss) <= TOL * abs(oloss), (key, loss, oloss)


def test_tgemm_falls_back_for_the_agent_id_only_input():
    """marl_tgemm_enable(1) with the [obs | agent id] composition: the TMA GEMM back end takes no one-hot column without
    the last-action block, so fc1 (forward) and its weight gradient (backward) run on linear.cu, while the plain layers still
    go to tgemm.cu; results as with the switch off.  Widths 84 ([obs | agent id]) and 96 (the default input) are both
    TMA-addressable: under the same switch the default input's fc1 does take the TMA path."""
    N, A, O, S, T, B = 4, 12, 80, 120, 8, 16
    mac = _mac(_args("vdn", N, A, O, S, T))
    default = _mac(_args("vdn", N, A, O, S, T, last_action=True))
    batch = synthetic_batch(2, B, T, N, A, O, S)
    obs = torch.as_tensor(batch["o"], dtype=torch.float32, device="cuda").contiguous()
    oh = torch.as_tensor(batch["u_onehot"], dtype=torch.float32, device="cuda").contiguous()
    lib = L.load()
    prev_f, prev_t = lib.marl_front_enable(0), lib.marl_tgemm_enable(1)
    try:
        _, launches = _kernels(lambda: default.agent.unroll(obs, oh, None, 1))
        assert "tgemm_kernel" in launches and "linear_fwd_kernel" not in launches, launches
        (q, _, _), launches = _kernels(lambda: mac.agent.unroll(obs, None, None, 1, last_action=False, agent_id=True))
        assert "tgemm_kernel" in launches and launches["linear_fwd_kernel"][0] == 1, launches      # fc1 alone
        (_, grads), launches = _kernels(lambda: (q.square().sum().backward(), [p.grad.clone() for p in mac.parameters()]))
        assert "linear_wgrad_kernel" in launches, launches
    finally:
        lib.marl_front_enable(prev_f)
        lib.marl_tgemm_enable(prev_t)
    for p in mac.parameters():
        p.grad = None
    q2, _, _ = mac.agent.unroll(obs, None, None, 1, last_action=False, agent_id=True)
    q2.square().sum().backward()
    assert PU.rel_err(q, q2) < 1e-6
    for g, p in zip(grads, mac.parameters()):
        assert PU.rel_err(g, p.grad) < 1e-5


def test_early_exit_and_graph_replay_at_two_batch_shapes():
    """B * N = 640 rows (B = 128, N = 5): early exit on and off give the same losses, on two batch shapes with different
    max_episode_len, alternating so that each shape is captured into its own CUDA graph and replayed."""
    N, A, O, S, T = 5, 11, 80, 120, 20
    b1 = synthetic_batch(1, 128, T, N, A, O, S, full_length_first=True, min_len=2)
    b2 = {}
    for k, v in synthetic_batch(2, 128, 12, N, A, O, S, full_length_first=True, min_len=2).items():   # padded to T as
        pad = np.ones if k in ("padded", "terminated") else np.zeros                               # rollout.py:122-133 pads
        b2[k] = np.concatenate([v, pad((v.shape[0], T - 12) + v.shape[2:])], axis=1)
    seq = [b1, b2] * 4
    out = {}
    for early in (False, True):
        args = _args("qmix", N, A, O, S, T, early_exit=early, cuda_graph=True, target_update_cycle=200)
        learner = _learner(args)
        out[early] = [learner.train({k: v.copy() for k, v in b.items()}, i) for i, b in enumerate(seq)]
        assert len([k for k, v in learner._graphs.items() if isinstance(v, tuple)]) == 2
    lf, le = out[False], out[True]
    assert abs(lf[0] - le[0]) <= 1e-6 * abs(lf[0]) and abs(lf[1] - le[1]) <= 1e-6 * abs(lf[1]), (lf, le)
    assert all(abs(a - b) <= 2e-5 * abs(a) for a, b in zip(lf, le)), (lf, le)


# ------------------------------------------------------------------------------------------ acting
@pytest.mark.parametrize("last_action,reuse_network", FLAGS)
def test_greedy_choose_actions_matches_choose_action_loop(last_action, reuse_network):
    """The reference's literal 3s5z inputs (golden choose_action_3s5z; the last-action input dropped where it is off) on
    seeded weights: one choose_actions call per step gives the actions and the carried hidden state of choose_action
    looped over the agents."""
    z = GU.load("choose_action_3s5z")
    N, A, O = (int(x) for x in z["meta/dims"])
    args = _args("qmix", N, A, O, 4, 10, last_action, reuse_network)
    one, batched = _mac(args, 1), _mac(args, 2)
    batched.load_state(one)
    for m in (one, batched):
        m.init_hidden(1)
    last = np.zeros((N, A))
    for t in range(z["obs"].shape[0]):
        want = np.array([int(one.choose_action(z["obs"][t, a], last[a], a, z["avail"][t, a], 0.0)) for a in range(N)])
        got = batched.choose_actions(z["obs"][t][None], last[None] if last_action else None, z["avail"][t][None], 0.0,
                                     evaluate=True)
        assert tuple(got.shape) == (1, N) and got.dtype == torch.int64
        assert np.array_equal(got[0].cpu().numpy(), want), t
        assert PU.rel_err(batched.hidden_states, one.hidden_states) < 1e-5, t
        last = np.eye(A)[want]


@pytest.mark.parametrize("last_action,reuse_network", FLAGS)
@pytest.mark.parametrize("n,N,A,O", [(64, 5, 11, 80), (32, 8, 14, 128), (16, 27, 36, 285), (7, 3, 5, 4), (257, 3, 5, 4),
                                     (7, 2, 3, 1)])
def test_act_matches_fp64_oracle_over_five_steps(n, N, A, O, last_action, reuse_network):
    """q and h' within 1e-5 of the fp64 oracle's unroll, carried over 5 consecutive calls; greedy actions exact except where
    the fp64 top-2 gap is below 1e-5; agent 0 with nothing available takes action 0."""
    mac = _mac(_args("qmix", N, A, O, 4, 10, last_action, reuse_network), seed=n + N)
    p = {k: v.detach().cpu().double() for k, v in mac.agent.state_dict().items()}
    cfg = MO.make_cfg(n_agents=N, n_actions=A, obs_shape=O, last_action=last_action, reuse_network=reuse_network)
    rng = np.random.RandomState(n * 31 + A)
    T = 5
    obs, last = rng.randn(n, T, N, O), rng.rand(n, T, N, A)
    avail = (rng.rand(n, T, N, A) < 0.6).astype(np.float64)
    avail[:, :, 0, :] = 0.0
    oq, oh, _ = MO.unroll(p, torch.as_tensor(obs), torch.as_tensor(last), torch.zeros(n * N, H, dtype=torch.float64), cfg)
    hidden = torch.zeros(n * N, H, device="cuda")
    for t in range(T):
        q = torch.empty(n, N, A, device="cuda")
        t32 = lambda x: torch.as_tensor(x[:, t], dtype=torch.float32, device="cuda").contiguous()
        act = mac.act(n, t32(obs), t32(last) if last_action else None, t32(avail), hidden, q=q)
        assert PU.rel_err(q, oq[:, t]) < 1e-5, t
        assert PU.rel_err(hidden.view(n, N, H), oh[:, t]) < 1e-5, t
        masked = np.where(avail[:, t] == 0, -np.inf, oq[:, t].numpy()).reshape(n * N, A)
        _, hard = PU.argmax_mismatches(act, masked, masked.argmax(1))
        assert hard == 0, t
        assert np.all(act[:, 0].cpu().numpy() == 0)


def _act_inputs(n, N, A, O, seed):
    rng = np.random.RandomState(seed)
    t = lambda x: torch.as_tensor(x, dtype=torch.float32, device="cuda").contiguous()
    avail = (rng.rand(n, N, A) < 0.5).astype(np.float32)
    avail[::5, 0, :] = 0.0
    return t(rng.randn(n, N, O)), t(avail), avail, rng


def test_exploration_contract_and_one_launch_per_call():
    """Uniform form: explore iff explore_u < eps, then the floor(choice_u * cnt)-th available action, else greedy; torch's
    seed governs device draws.  Flag form: what marl_epsgreedy_select makes of the same q.  Each call is one launch."""
    n, N, A, O = 300, 4, 9, 6
    mac = _mac(_args("qmix", N, A, O, 4, 10))
    obs, avail_d, avail, rng = _act_inputs(n, N, A, O, 1)
    eu, cu = rng.rand(n, N), rng.rand(n, N)
    eps = 0.5
    h0 = torch.randn(n * N, H, device="cuda") * 0.5
    greedy, launches = _kernels(lambda: mac.act(n, obs, None, avail_d, h0.clone()).cpu().numpy())
    assert {k: v[0] for k, v in launches.items()} == {"agent_act_kernel": 1}, launches
    mac.init_hidden(n)
    mac.hidden_states.copy_(h0.view(n, N, H))
    got, launches = _kernels(lambda: mac.choose_actions(obs, None, avail_d, eps, draws=(eu, cu)).cpu().numpy())
    assert {k: v[0] for k, v in launches.items()} == {"agent_act_kernel": 1}, launches
    cnt = avail.sum(-1)
    kth = np.minimum(np.floor(cu * cnt), cnt - 1)
    want = np.where(cnt > 0, ((np.cumsum(avail, -1) == (kth + 1)[..., None]) & (avail > 0)).argmax(-1), 0)
    explored = eu < eps
    assert explored.mean() > 0.3 and (~explored).mean() > 0.3
    assert np.array_equal(got[explored], want[explored]) and np.array_equal(got[~explored], greedy[~explored])
    assert np.all(got[cnt == 0] == 0)
    outs = []
    for _ in range(2):
        mac.hidden_states.copy_(h0.view(n, N, H))
        torch.manual_seed(5)
        outs.append(mac.choose_actions(obs, None, avail_d, eps).cpu().numpy())
    assert np.array_equal(outs[0], outs[1])
    explore = torch.as_tensor((rng.rand(n, N) < 0.4).astype(np.uint8), device="cuda")
    rand_a = torch.as_tensor(rng.randint(0, A, (n, N)), dtype=torch.int64, device="cuda")
    q, onehot = torch.empty(n, N, A, device="cuda"), torch.empty(n, N, A, device="cuda")
    got = mac.act(n, obs, None, avail_d, h0.clone(), explore=explore, random_action=rand_a, q=q, onehot=onehot)
    want, want_oh = torch.empty(n * N, dtype=torch.int64, device="cuda"), torch.empty(n * N, A, device="cuda")
    L.call("marl_epsgreedy_select", n * N, A, q.data_ptr(), avail_d.data_ptr(), explore.data_ptr(), rand_a.data_ptr(),
           want.data_ptr(), want_oh.data_ptr(), L.stream_ptr())
    assert torch.equal(got.view(-1), want) and torch.equal(onehot.view(-1, A), want_oh)


def test_bad_acting_calls_raise():
    n, N, A, O = 9, 3, 7, 5
    mac = _mac(_args("qmix", N, A, O, 4, 10))
    obs, avail_d, _, _ = _act_inputs(n, N, A, O, 4)
    hidden = torch.zeros(n * N, H, device="cuda")
    from marl_b200.network.q_network import agent_param_struct
    ps = agent_param_struct(mac.agent.param_addresses())
    action = torch.empty(n, N, dtype=torch.int64, device="cuda")
    with pytest.raises(ValueError):                        # last_action set, no last_onehot: MARL_EINVAL
        L.call("marl_agent_act_input", n, N, A, O, 1, 1, C.byref(ps), obs.data_ptr(), None, avail_d.data_ptr(),
               hidden.data_ptr(), hidden.data_ptr(), None, None, None, None, 0.0, None, action.data_ptr(), None, None,
               L.stream_ptr())
    with_last = _mac(_args("qmix", N, A, O, 4, 10, last_action=True))
    with pytest.raises(ValueError):                        # the network reads the last action: it is required
        with_last.act(n, obs, None, avail_d, hidden)
    mac.init_hidden(n)
    with pytest.raises(ValueError):
        mac.choose_actions(obs[:, :2], None, avail_d, 0.5)


# ------------------------------------------------------------------------------------------ the batched rollout
PAYOFF1 = [[8, -12, -12], [-12, 0, 0], [-12, 0, 0]]


@pytest.mark.parametrize("epsilon", [1.0, 0.3, 0.0])
def test_matrix_game_matches_sequential_oracle(epsilon):
    """BatchedRolloutWorker on the matrix game with a SharedMAC without the last-action input, against the sequential rollout
    with every agent on the shared network's parameters, under one numpy seed: actions, float64 rewards, epsilon, bit for bit."""
    from marl_b200.env.single_state_matrix_game import BatchedMatrixGame
    from marl_b200.rollout import BatchedRolloutWorker
    n = 257
    args = _args("qmix", 2, 3, 1, 1, 1)
    mac = _mac(args, 7)
    args.epsilon, args.anneal_epsilon = epsilon, 0.01
    env = BatchedMatrixGame(PAYOFF1, n, keep_r64=True)
    worker = BatchedRolloutWorker(env, mac, args)
    np.random.seed(7)
    episodes, _, _, steps = worker.generate_episodes()
    np.random.seed(7)
    sd = {k: v.detach().cpu() for k, v in mac.agent.state_dict().items()}
    want_u, want_r, want_eps = SRO.generate_episodes([sd, sd], PAYOFF1, n, epsilon, 0.01, args.min_epsilon, "step",
                                                    last_action=False, reuse_network=True)
    assert np.array_equal(episodes["u"].reshape(n, 2).cpu().numpy(), want_u)
    assert np.array_equal(env.r64.cpu().numpy(), want_r)
    assert worker.epsilon == want_eps and steps == n


KEYS11 = ("o", "s", "u", "r", "avail_u", "o_next", "s_next", "avail_u_next", "u_onehot", "padded", "terminated")


def _multistep_worker(T, n, seed=8):
    from marl_b200.rollout import BatchedRolloutWorker
    from tests.envs import CountdownGameBatched
    N, A, O, S = 3, 5, 4, 3
    args = _args("qmix", N, A, O, S, T)
    mac = _mac(args, seed)
    args.epsilon, args.anneal_epsilon, args.min_epsilon, args.epsilon_anneal_scale = 0.5, 0.01, 0.02, "step"
    return BatchedRolloutWorker(CountdownGameBatched(n, n_agents=N, n_actions=A, episode_limit=T), mac, args)


def _check_against_oracle(worker, n, seed):
    from tests.envs import CountdownGameHost
    a, N, T = worker.args, worker.n_agents, worker.episode_limit
    rng = np.random.RandomState(seed)
    draws = (rng.rand(n, T, N), rng.rand(n, T, N))
    worker.epsilon = 0.5
    ep, rewards, _, steps = worker.generate_episodes(draws=draws)
    sd = {k: v.detach().cpu() for k, v in worker.mac.agent.state_dict().items()}
    oep, orew, osteps = SRO.rollout_multistep([sd] * N, CountdownGameHost(n_agents=N, n_actions=a.n_actions, episode_limit=T),
                                              n, 0.5, 0.01, 0.02, "step", draws=draws, last_action=False, reuse_network=True)
    for k in KEYS11:
        assert np.array_equal(ep[k].cpu().numpy().astype(np.float64), oep[k]), k
    assert np.array_equal(rewards.cpu().numpy(), np.array(orew)) and steps == osteps
    assert (draws[0] < 0.5)[oep["padded"][:, :, 0] == 0].mean() > 0.2
    return ep


def test_multistep_rollout_to_buffer_to_learner_matches_oracle():
    """Exploring multi-step episodes under host draws equal the sequential rollout bit for bit; they go through
    store_episode -> sample -> QLearner.train, whose loss matches the oracle (1e-5 on the first step, 5e-5 after); a rollout
    after training acts on the weights the learner re-packed into its flat buffer."""
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
    st = _oracle(learner, args)
    host = {k: v.cpu().numpy().astype(np.float64) for k, v in buf.buffers.items()}
    np.random.seed(0)
    for step in range(3):
        view = buf.sample(32)
        batch = {k: host[k][view.idx_host] for k in host}
        loss = learner.train(view, step)
        oloss, _ = MO.train_step(st, batch, step)
        assert abs(loss - oloss) <= (1e-5 if step == 0 else 5e-5) * abs(oloss), (step, loss, oloss)
    _check_against_oracle(worker, n, 2)


# ------------------------------------------------------------------------------------------ checkpoints and the ABI default
def test_checkpoint_round_trip(tmp_path):
    N, A, O = 5, 11, 80
    args = _args("qmix", N, A, O, 4, 10)
    src, dst = _mac(args, 1), _mac(args, 2)
    sd = src.agent.state_dict()
    assert tuple(sd["fc1.weight"].shape) == (H, O + N)
    assert list(sd) == ["fc1.weight", "fc1.bias", "rnn.weight_ih", "rnn.weight_hh", "rnn.bias_ih", "rnn.bias_hh",
                        "fc2.weight", "fc2.bias"]
    path = str(tmp_path / "rnn_net_params.pkl")
    src.save_models(path)
    dst.load_models(path)
    for k, v in dst.agent.state_dict().items():
        assert torch.equal(v, sd[k]), k
    n = 20
    obs, avail_d, _, _ = _act_inputs(n, N, A, O, 3)
    outs = []
    for m in (src, dst):
        q, h = torch.empty(n, N, A, device="cuda"), torch.zeros(n * N, H, device="cuda")
        outs.append((m.act(n, obs, None, avail_d, h, q=q), q, h))
    for x, y in zip(*outs):
        assert torch.equal(x, y)


def test_default_input_when_input_flags_is_zero():
    """A shared stream that leaves input_flags at 0 reads [obs | last action | agent id] whatever last_action / agent_id
    hold (what callers written before the field existed rely on): with both at 0 its outputs equal, bit for bit, those of
    the same call with input_flags = last_action = agent_id = 1."""
    B, T, N, A, O = 4, 7, 3, 5, 8
    mac = _mac(_args("qmix", N, A, O, 4, T, last_action=True, reuse_network=True))
    from marl_b200.network.q_network import agent_param_struct
    params = agent_param_struct(mac.agent.param_addresses())
    rng = np.random.RandomState(0)
    t = lambda x: torch.as_tensor(x, dtype=torch.float32, device="cuda").contiguous()
    obs, oh = t(rng.randn(B, T, N, O)), t(np.eye(A)[rng.randint(0, A, (B, T, N))])
    d = L.Dims(B, T, N, A, O, 0)
    res = []
    for flags in (0, 1):
        f = lambda *shape: torch.zeros(*shape, device="cuda")
        q, hid, hl, x, gi = f(B, T, N, A), f(B, T, N, H), f(B * N, H), f(B * T * N, H), f(B * T * N, 3 * H)
        s = L.UnrollStream()
        s.obs, s.onehot, s.shift_onehot, s.h0_from, s.params = obs.data_ptr(), oh.data_ptr(), 1, -1, params
        s.q, s.hidden, s.h_last, s.x, s.gi = q.data_ptr(), hid.data_ptr(), hl.data_ptr(), x.data_ptr(), gi.data_ptr()
        s.input_flags, s.last_action, s.agent_id = flags, flags, flags
        L.call("marl_agent_unroll_fwd", C.byref(d), C.byref(s), 1, L.stream_ptr())
        res.append((q, hid, hl))
    for a, b in zip(*res):
        assert torch.equal(a, b)
    mac.init_hidden(B)
    q_mac, _ = mac.get_current_q_values({"o": obs, "u_onehot": oh}, T)
    assert PU.rel_err(res[0][0], q_mac) < 1e-6
    # the opt-in with a full input, and a last-action block without its one-hot, are refused
    for bad in (dict(input_flags=1, full_input=1, last_action=1, agent_id=1), dict(input_flags=1, last_action=1, onehot=None)):
        s = L.UnrollStream()
        s.obs, s.onehot, s.shift_onehot, s.h0_from, s.params = obs.data_ptr(), oh.data_ptr(), 1, -1, params
        s.hidden, s.x, s.gi = hid.data_ptr(), x.data_ptr(), gi.data_ptr()
        for k, v in bad.items():
            setattr(s, k, v)
        with pytest.raises(ValueError):
            L.call("marl_agent_unroll_fwd", C.byref(d), C.byref(s), 1, L.stream_ptr())
