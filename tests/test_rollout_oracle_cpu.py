"""Pins oracle/rollout_oracle.py against the UNMODIFIED reference (RolloutWorker + SharedMAC.choose_action +
TwoAgentsMatrixGame) when it is staged in oracle/_ref (oracle/fetch_ref.py); the GPU tests then hold the batched
rollout to the oracle."""
import sys
import types
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import fetch_ref as FR
from oracle import rollout_oracle as RO

PAYOFF1 = [[8, -12, -12], [-12, 0, 0], [-12, 0, 0]]


@pytest.mark.skipif(not FR.available(), reason="reference not staged in oracle/_ref")
@pytest.mark.parametrize("scale", ["step", "episode"])
def test_rollout_oracle_matches_reference(scale, capsys):
    sys.path.insert(0, FR.DST)
    saved_gym = sys.modules.get("gym")
    sys.modules["gym"] = types.SimpleNamespace(Env=object)          # env/single_state_matrix_game.py:3,123
    if not hasattr(np, "float"):
        np.float = float                                             # numpy >= 1.24 removed the aliases the reference uses
        np.long = np.int64
    try:
        for m in [k for k in sys.modules if k.split(".")[0] in ("common", "controller", "network", "env", "rollout", "algorithm")]:
            del sys.modules[m]
        from common.arguments import get_mixer_args
        from controller.share_params import SharedMAC
        from env.single_state_matrix_game import TwoAgentsMatrixGame
        from rollout import RolloutWorker
        args = SimpleNamespace(RTW=False, alg="qmix", map="matrix", last_action=True, reuse_network=True, gamma=0.99,
                               optimizer="RMS", model_dir="/tmp/m", result_dir="/tmp/r", cuda=False, load_model=False,
                               evaluate=False, evaluate_epoch=0, replay_dir="", n_episodes=1)
        get_mixer_args(args)
        env = TwoAgentsMatrixGame(np.array(PAYOFF1, dtype=np.float64))
        info = env.get_env_info()
        args.n_actions, args.n_agents, args.state_shape = info["n_actions"], info["n_agents"], info["state_shape"]
        args.obs_shape, args.episode_limit = info["obs_shape"], info["episode_limit"]
        args.epsilon, args.anneal_epsilon, args.min_epsilon, args.epsilon_anneal_scale = 0.5, 0.01, 0.05, scale
        torch.manual_seed(0)
        mac = SharedMAC(args)
        worker = RolloutWorker(env, mac, args)
        np.random.seed(11)
        episodes, rewards, wins, steps = worker.generate_episodes(n_episodes=40)
        np.random.seed(11)
        params = {k: v.detach().clone() for k, v in mac.agent.state_dict().items()}
        u, r, eps = RO.generate_episodes(params, PAYOFF1, 40, 0.5, 0.01, 0.05, scale)
    finally:
        sys.path.remove(FR.DST)
        if saved_gym is not None:
            sys.modules["gym"] = saved_gym
        else:
            sys.modules.pop("gym", None)
        for m in [k for k in sys.modules if k.split(".")[0] in ("common", "controller", "network", "env", "rollout", "algorithm")]:
            del sys.modules[m]
    assert np.array_equal(np.asarray(episodes["u"]).reshape(40, 2).astype(np.int64), u)
    assert np.array_equal(np.asarray(rewards, dtype=np.float64), r)
    assert worker.epsilon == eps and steps == 40


def test_multistep_rollout_oracle_matches_reference_worker_golden():
    """oracle.rollout_oracle.rollout_multistep against the UNMODIFIED reference RolloutWorker on the ragged multi-step
    test game (tests/golden/rollout_multistep.npz, made by oracle/make_golden.py rollout): every key of the padded
    episode batch, the episode rewards and the step count, bit for bit."""
    from tests import golden_util as GU
    from tests.envs import CountdownGameHost
    z = GU.load("rollout_multistep")
    n = int(z["meta/n"])
    np.random.seed(3)
    eps, rewards, steps = RO.rollout_multistep(GU.group(z, "init/agent"), CountdownGameHost(), n, 0.5, 0.01, 0.02, "step", evaluate=True)
    for k in ("o", "s", "u", "r", "avail_u", "o_next", "s_next", "avail_u_next", "u_onehot", "padded", "terminated"):
        assert np.array_equal(eps[k], z[f"episodes/{k}"]), k
    assert np.array_equal(np.array(rewards), z["rewards"]) and steps == int(z["steps"])
    lens = (1 - eps["padded"][:, :, 0]).sum(1)
    assert lens.min() < lens.max() == 6            # the fixture really is ragged and reaches the limit
