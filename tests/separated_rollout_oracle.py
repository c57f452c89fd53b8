"""TEST INFRASTRUCTURE ONLY -- the sequential rollout of ``oracle/rollout_oracle.py`` with one network per agent.

``SeparatedMAC.choose_action`` (``controller/share_params.py:419-453``) driven by ``RolloutWorker``
(``rollout.py:30-173``): agent a acts with its own network on ``[obs | last_action (if last_action) | agent id (if
reuse_network)]`` (``share_params.py:467-506``); the episode loop, epsilon schedule, RNG order, masking and episode
layout are those of ``oracle/rollout_oracle.py``.  ``agent_params`` is a list of one state dict per agent (a single
dict is every agent's network, with the default flags that is exactly ``oracle/rollout_oracle.py``, which
tests/test_separated_rollout_oracle_cpu.py checks).  Only tests import this module.
"""
import numpy as np
import torch

from oracle import marl_oracle as MO


def _detach(agent_params):
    if isinstance(agent_params, (list, tuple)):
        return [{k: v.detach() for k, v in p.items()} for p in agent_params]
    return {k: v.detach() for k, v in agent_params.items()}


def _act_step(p, a, obs, last, n_agents, h, last_action, reuse_network):
    """Agent a's forward on [obs | last action (last_action) | agent id (reuse_network)]; advances h[:, a] in place."""
    parts = [obs]
    if last_action:
        parts.append(last)
    if reuse_network:
        agent_id = np.zeros(n_agents)
        agent_id[a] = 1.0
        parts.append(agent_id)
    x = torch.tensor(np.hstack(parts), dtype=torch.float32).unsqueeze(0)
    q, hn = MO.agent_step(p[a] if isinstance(p, list) else p, x, h[:, a, :])
    h[:, a, :] = hn
    return q


def generate_episodes(agent_params, payoff, n_episodes, epsilon, anneal_epsilon, min_epsilon, anneal_scale="step",
                      evaluate=False, n_agents=2, n_actions=3, obs_shape=1, hidden=64, last_action=True, reuse_network=True):
    payoff = np.asarray(payoff, dtype=np.float64).reshape(3, 3)
    p = _detach(agent_params)
    actions = np.zeros((n_episodes, n_agents), dtype=np.int64)
    rewards = np.zeros(n_episodes, dtype=np.float64)
    cur = epsilon
    with torch.no_grad():
        for e in range(n_episodes):
            h = torch.zeros(1, n_agents, hidden)                       # mac.init_hidden(1), rollout.py:45
            eps = 0 if evaluate else cur
            if anneal_scale == "episode":
                eps = eps - anneal_epsilon if eps > min_epsilon else eps
            obs = [np.zeros(obs_shape) for _ in range(n_agents)]       # env.get_obs(), single_state_matrix_game.py:42-45
            last = np.zeros((n_agents, n_actions))
            for a in range(n_agents):
                q = _act_step(p, a, obs[a], last[a], n_agents, h, last_action, reuse_network)
                avail = np.ones(n_actions)
                q[torch.tensor(avail).unsqueeze(0) == 0.0] = -float("inf")
                if np.random.uniform() < eps:                          # share_params.py:67-70
                    act = int(np.random.choice(np.nonzero(avail)[0]))
                else:
                    act = int(torch.argmax(q))
                actions[e, a] = act
                last[a] = np.eye(n_actions)[act]
            rewards[e] = payoff[actions[e, 0], actions[e, 1]]
            if anneal_scale == "step":
                eps = eps - anneal_epsilon if eps > min_epsilon else eps
            if not evaluate:
                cur = eps
    return actions, rewards, cur


def rollout_multistep(agent_params, env, n_episodes, epsilon, anneal_epsilon, min_epsilon, anneal_scale="step", evaluate=False,
                      draws=None, hidden=64, last_action=True, reuse_network=True):
    """``RolloutWorker.generate_episodes`` (rollout.py:30-173) on a multi-step SMAC-style host environment: per-step
    epsilon (``:47-49, 103-104``), availability masking in ``choose_action``, the trailing observation / state /
    availability read after the last step (``:106-120``), zero padding to ``episode_limit`` with ``padded = 1`` and
    ``terminated = 1`` (``:122-133``), the episode layout (``:135-149``).

    ``draws=None`` consumes numpy's global RNG in the reference's order.  ``draws=(explore_u, choice_u)`` (arrays
    [n_episodes, episode_limit, n_agents] of uniforms in [0, 1)) is the batched worker's RNG contract: agent a of
    episode e explores at step t iff explore_u[e, t, a] < epsilon_t and then takes the floor(choice_u * n_available)-th
    available action; every episode starts from the same epsilon (the instances run side by side)."""
    info = env.get_env_info()
    N, A, O, S, T = (info[k] for k in ("n_agents", "n_actions", "obs_shape", "state_shape", "episode_limit"))
    p = _detach(agent_params)
    keys = ("o", "s", "u", "r", "avail_u", "o_next", "s_next", "avail_u_next", "u_onehot", "padded", "terminated")
    out = {k: [] for k in keys}
    rewards, steps_tot, cur = [], 0, epsilon
    with torch.no_grad():
        for e in range(n_episodes):
            env.reset()
            h = torch.zeros(1, N, hidden)
            eps = 0 if evaluate else (cur if draws is None else epsilon)
            if anneal_scale == "episode":
                eps = eps - anneal_epsilon if eps > min_epsilon else eps
            last = np.zeros((N, A))
            o, u, r, s, avail_u, u_onehot, terminate, padded = [], [], [], [], [], [], [], []
            terminated, step, ep_reward = False, 0, 0.0
            while not terminated and step < T:
                obs, state, avail = env.get_obs(), env.get_state(), env.get_avail_actions()
                actions, onehots = [], []
                for a in range(N):
                    q = _act_step(p, a, obs[a], last[a], N, h, last_action, reuse_network)
                    av = np.asarray(avail[a])
                    q[torch.tensor(av, dtype=torch.float32).unsqueeze(0) == 0.0] = -float("inf")
                    idx = np.nonzero(av)[0]
                    if draws is None:
                        act = int(np.random.choice(idx)) if np.random.uniform() < eps else int(torch.argmax(q))
                    else:
                        eu, cu = draws[0][e, step, a], draws[1][e, step, a]
                        act = int(idx[min(int(cu * len(idx)), len(idx) - 1)]) if eu < eps else int(torch.argmax(q))
                    actions.append(act)
                    onehots.append(np.eye(A)[act])
                    last[a] = np.eye(A)[act]
                reward, terminated, _ = env.step(actions)
                o.append(obs); s.append(state); u.append(np.reshape(actions, [N, 1])); u_onehot.append(onehots)
                avail_u.append(avail); r.append([reward]); terminate.append([terminated]); padded.append([0.0])
                ep_reward += reward
                step += 1
                if anneal_scale == "step":
                    eps = eps - anneal_epsilon if eps > min_epsilon else eps
            o.append(env.get_obs()); s.append(env.get_state())
            o_next, s_next, o, s = o[1:], s[1:], o[:-1], s[:-1]
            avail_u.append([env.get_avail_agent_actions(a) for a in range(N)])
            avail_u_next, avail_u = avail_u[1:], avail_u[:-1]
            for _ in range(step, T):
                o.append(np.zeros((N, O))); u.append(np.zeros([N, 1])); s.append(np.zeros(S)); r.append([0.0])
                o_next.append(np.zeros((N, O))); s_next.append(np.zeros(S)); u_onehot.append(np.zeros((N, A)))
                avail_u.append(np.zeros((N, A))); avail_u_next.append(np.zeros((N, A))); padded.append([1.0]); terminate.append([1.0])
            ep = dict(o=o, s=s, u=u, r=r, avail_u=avail_u, o_next=o_next, s_next=s_next, avail_u_next=avail_u_next,
                      u_onehot=u_onehot, padded=padded, terminated=terminate)
            for k in keys:
                out[k].append(np.array(ep[k], dtype=np.float64))
            rewards.append(ep_reward)
            steps_tot += step
            if not evaluate and draws is None:
                cur = eps
    return {k: np.stack(v) for k, v in out.items()}, rewards, steps_tot
