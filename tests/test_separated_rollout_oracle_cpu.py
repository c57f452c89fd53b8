"""The per-agent sequential rollout of tests/separated_rollout_oracle.py (one parameter dict per agent, input blocks
chosen by last_action / reuse_network): equal to oracle/rollout_oracle.py when every agent holds the same network, and
pinned against the UNMODIFIED reference (RolloutWorker driving its own SeparatedMAC.choose_action,
share_params.py:419-453, on the matrix game) when it is staged in oracle/_ref (oracle/fetch_ref.py)."""
import sys
import types
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import fetch_ref as FR
from oracle import marl_oracle as MO
from oracle import rollout_oracle as RO
from tests import separated_rollout_oracle as SRO

PAYOFF1 = [[8, -12, -12], [-12, 0, 0], [-12, 0, 0]]
REF_PACKAGES = ("common", "controller", "network", "env", "rollout", "algorithm")


def test_list_form_with_one_network_everywhere_equals_shared_form():
    from tests import golden_util as GU
    from tests.envs import CountdownGameHost
    torch.manual_seed(0)
    p = MO.init_agent(MO.make_cfg(n_agents=2, n_actions=3, obs_shape=1))
    outs = []
    for run in (lambda: RO.generate_episodes(p, PAYOFF1, 30, 0.5, 0.01, 0.05, "step"),
                lambda: SRO.generate_episodes([p, p], PAYOFF1, 30, 0.5, 0.01, 0.05, "step")):
        np.random.seed(1)
        outs.append(run())
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1]) and outs[0][2] == outs[1][2]
    z = GU.load("rollout_multistep")
    q = GU.group(z, "init/agent")
    N, A, _, _, T = (int(x) for x in z["meta/dims"])
    rng = np.random.RandomState(2)
    draws = (rng.rand(9, T, N), rng.rand(9, T, N))
    outs = [f(x, CountdownGameHost(n_agents=N, n_actions=A, episode_limit=T), 9, 0.5, 0.01, 0.02, "step", draws=draws)
            for f, x in ((RO.rollout_multistep, q), (SRO.rollout_multistep, [q] * N))]
    for k in outs[0][0]:
        assert np.array_equal(outs[0][0][k], outs[1][0][k]), k
    assert outs[0][1:] == outs[1][1:]


@pytest.mark.skipif(not FR.available(), reason="reference not staged in oracle/_ref")
@pytest.mark.parametrize("last_action", [True, False])
def test_separated_rollout_oracle_matches_reference(last_action):
    sys.path.insert(0, FR.DST)
    saved_gym = sys.modules.get("gym")
    sys.modules["gym"] = types.SimpleNamespace(Env=object)          # env/single_state_matrix_game.py:3,123
    if not hasattr(np, "float"):
        np.float = float                                             # numpy >= 1.24 removed the aliases the reference uses
        np.long = np.int64
    try:
        for m in [k for k in sys.modules if k.split(".")[0] in REF_PACKAGES]:
            del sys.modules[m]
        from common.arguments import get_mixer_args
        from controller.share_params import SeparatedMAC
        from env.single_state_matrix_game import TwoAgentsMatrixGame
        from rollout import RolloutWorker
        args = SimpleNamespace(RTW=False, alg="qmix", map="matrix", last_action=last_action, reuse_network=False,
                               gamma=0.99, optimizer="RMS", model_dir="/tmp/m", result_dir="/tmp/r", cuda=False,
                               load_model=False, evaluate=False, evaluate_epoch=0, replay_dir="", n_episodes=1)
        get_mixer_args(args)
        env = TwoAgentsMatrixGame(np.array(PAYOFF1, dtype=np.float64))
        info = env.get_env_info()
        args.n_actions, args.n_agents, args.state_shape = info["n_actions"], info["n_agents"], info["state_shape"]
        args.obs_shape, args.episode_limit = info["obs_shape"], info["episode_limit"]
        args.epsilon, args.anneal_epsilon, args.min_epsilon, args.epsilon_anneal_scale = 0.5, 0.01, 0.05, "step"
        torch.manual_seed(0)
        mac = SeparatedMAC(args)                                     # what runner.py:24-26 builds when reuse_network is False
        worker = RolloutWorker(env, mac, args)
        np.random.seed(11)
        episodes, rewards, wins, steps = worker.generate_episodes(n_episodes=40)
        np.random.seed(11)
        params = [{k: v.detach().clone() for k, v in net.state_dict().items()} for net in mac.agent]
        u, r, eps = SRO.generate_episodes(params, PAYOFF1, 40, 0.5, 0.01, 0.05, "step", last_action=last_action,
                                          reuse_network=False)
    finally:
        sys.path.remove(FR.DST)
        if saved_gym is not None:
            sys.modules["gym"] = saved_gym
        else:
            sys.modules.pop("gym", None)
        for m in [k for k in sys.modules if k.split(".")[0] in REF_PACKAGES]:
            del sys.modules[m]
    assert not torch.equal(params[0]["fc1.weight"], params[1]["fc1.weight"])
    assert np.array_equal(np.asarray(episodes["u"]).reshape(40, 2).astype(np.int64), u)
    assert np.array_equal(np.asarray(rewards, dtype=np.float64), r)
    assert worker.epsilon == eps and steps == 40
