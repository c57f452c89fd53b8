"""Batched data collection, the many-environments counterpart of ``rollout.py:3-173``.

The reference's ``RolloutWorker.generate_episodes`` plays ONE environment, asks ``mac.choose_action`` for one
agent at a time (a batch-1 network forward each, ``rollout.py:60-76``) and concatenates episodes with
``np.concatenate``.  ``BatchedRolloutWorker`` plays every instance of a batched environment
(``BatchedMatrixGame``) at once: one act launch (agent network and epsilon-greedy selection) for all (env, agent)
rows, one environment step launch; the episode batch comes out on the device in the ReplayBuffer layout
(``rollout.py:135-149``) and can go straight into ``marl_b200.common.replaybuffer.ReplayBuffer``.  The act launch is
``mac.act``: ``marl_agent_act`` for a ``SharedMAC``, ``marl_agent_act_separated`` (each agent on its own network) for the
``SeparatedMAC`` that ``runner.py:24-26`` builds when ``reuse_network`` is False.

RNG contract.  ``rng="numpy"`` draws, on the host, exactly what the reference would draw and in its order --
per episode, per agent: one ``np.random.uniform()``, then ``np.random.choice(available)`` only when exploring
(``share_params.py:67-68``) -- so a seeded run takes bit-identical actions; none of these draws depends on the
Q-values, which is what makes hoisting them out of the per-agent loop exact.  ``rng="device"`` draws with
``torch`` on the GPU for throughput (same distribution, different stream).  ``rng="philox"`` has the act launch draw
them itself from Philox4x64-10 under key ``args.seed`` (``controller.share_params.PhiloxDraws``): the draws of episode
k depend only on (seed, k, step, agent), where k counts the episodes the worker has started (``episode_base``), so a
seeded run takes the same actions however its episodes are split between calls or devices, and nothing is drawn on
the host or held in memory.  Epsilon follows the reference's schedule (``rollout.py:47-49, 103-104, 166-167``):
annealed per step or per episode, carried across calls.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch as th

from . import _lib as L
from .controller.share_params import PhiloxDraws

RNG_FORMS = ("numpy", "device", "philox")


def epsilon_schedule(cur, anneal, min_eps, k):
    """v_0 .. v_k of the reference's schedule v_0 = cur, v_i = v_{i-1} - anneal if v_{i-1} > min_eps else v_{i-1}
    (rollout.py:47-49, 103-104), as its shortest prefix p: v_i = p[min(i, len(p) - 1)] for every i <= k.

    Until the first value <= min_eps the schedule is the running difference cur - anneal - anneal - ..., which
    np.subtract.accumulate computes as the same sequential float64 left fold as the loop, so the values are bit-identical;
    from that value on it is constant."""
    k = int(k)
    if k <= 0 or not cur > min_eps or anneal == 0:
        return np.array([cur], dtype=np.float64)
    m = k                                                  # evaluate only as far as the cut can be
    if anneal > 0:
        m = min(k, int((cur - min_eps) / anneal) + 2)
    while True:
        v = np.full(m + 1, anneal, dtype=np.float64)
        v[0] = cur
        np.subtract.accumulate(v, out=v)
        cut = np.flatnonzero(~(v > min_eps))
        if cut.size:
            return v[:cut[0] + 1]
        if m == k:
            changed = np.flatnonzero(v != v[-1])           # no cut within k: keep up to the last value that changes
            return v[:changed[-1] + 2] if changed.size else v[:1]
        m = min(k, 2 * m)


class BatchedRolloutWorker:
    def __init__(self, env, mac, args):
        self.env = env
        self.mac = mac
        self.episode_limit = args.episode_limit
        self.n_actions = args.n_actions
        self.n_agents = args.n_agents
        self.state_shape = args.state_shape
        self.obs_shape = args.obs_shape
        self.args = args
        self.epsilon = args.epsilon
        self.anneal_epsilon = args.anneal_epsilon
        self.min_epsilon = args.min_epsilon
        # one-step matrix game: the fused record-writing env kernel; anything else that speaks the batched protocol
        # (reset / get_obs / get_state / get_avail_actions / step(actions, active)) goes through the generic multi-step loop
        self._generic = not (hasattr(env, "payoff_table") and self.episode_limit == 1)
        self._active_host = None             # page-locked word: instances still active, stored by marl_rollout_record
        # episodes started so far: rng="philox" draws episode episode_base + e for instance e, and every call advances
        # it by env.n_envs.  A data-parallel caller sets it before each call (rank g: the global count + g * n_local).
        self.episode_base = 0

    def _record(self, dims, t, ep_s, obs, state, avail, actions, onehot, reward, term, active, last, rewards, counters):
        L.call("marl_rollout_record", C.byref(dims), t, C.byref(ep_s), obs.data_ptr(), state.data_ptr(), avail.data_ptr(),
               actions.data_ptr(), onehot.data_ptr(), L.ptr(reward), L.ptr(term), active.data_ptr(), last.data_ptr(),
               rewards.data_ptr(), counters.data_ptr(), self._active_host.data_ptr(), L.stream_ptr())

    def _eps_table(self, n, evaluate):
        """Epsilon of each of n one-step episodes played in sequence, as a table t (episode e acts with
        t[min(e, len(t) - 1)]: the schedule's distinct values), and the worker's epsilon after them."""
        scale = self.args.epsilon_anneal_scale
        if evaluate:                                           # acts with 0 (annealed once per episode), epsilon stays
            eps = 0.0 - self.anneal_epsilon if scale == 'episode' and 0 > self.min_epsilon else 0.0
            return np.array([eps], dtype=np.float64), self.epsilon
        if scale not in ('step', 'episode'):
            return np.array([self.epsilon], dtype=np.float64), self.epsilon
        v = epsilon_schedule(self.epsilon, self.anneal_epsilon, self.min_epsilon, n)
        after = float(v[min(n, len(v) - 1)])
        if scale == 'episode':                                 # annealed before the episode's step: e acts with v[e + 1]
            return (v[1:] if len(v) > 1 else v), after
        return v[:max(n, 1)], after                            # annealed after the step: e acts with v[e]

    def _epsilons(self, n, evaluate):
        """Per-episode epsilon, advanced exactly like n sequential episodes of the reference would."""
        table, cur = self._eps_table(n, evaluate)
        return table[np.minimum(np.arange(n), len(table) - 1)], cur

    def generate_episodes(self, n_episodes=None, evaluate=False, random_select=False, rng="numpy", draws=None):
        """Plays env.n_envs one-step episodes.  Returns (episodes, episode_rewards, win_tags, steps) like
        rollout.py:173; `episodes` is a dict of CUDA tensors [n_envs, 1, ...] owned by the environment."""
        n, N, A = self.env.n_envs, self.n_agents, self.n_actions
        if n_episodes not in (None, n):
            raise ValueError("a batched worker plays exactly env.n_envs episodes per call")
        if rng not in RNG_FORMS:
            raise ValueError(f"rng={rng!r}: expected one of {RNG_FORMS}")
        if rng == "philox" and draws is not None:
            raise ValueError("rng='philox' draws inside the act launch: draws= cannot be given with it")
        base = self.episode_base
        self.episode_base = base + n
        if self._generic:
            return self._generate_multistep(evaluate, random_select, draws,
                                            PhiloxDraws(self.args.seed, base) if rng == "philox" else None)
        if random_select:
            raise NotImplementedError("random_select is not used by the in-scope drivers")
        dev = self.mac.device
        if rng == "philox":                                    # one act launch draws everything: no host draws
            table, eps_after = self._eps_table(n, evaluate)
            return self._finish_matrix(n, evaluate, eps_after, philox=PhiloxDraws(self.args.seed, base),
                                       eps_table=th.from_numpy(table).to(dev))
        eps, eps_after = self._epsilons(n, evaluate)
        avail_idx = np.arange(A)                               # every action of the matrix game is available
        if rng == "numpy":
            explore = np.zeros((n, N), dtype=np.uint8)
            rand_a = np.zeros((n, N), dtype=np.int64)
            for e in range(n):                                 # the reference's draw order: episode-major, agent-minor
                for a in range(N):
                    if np.random.uniform() < eps[e]:
                        explore[e, a] = 1
                        rand_a[e, a] = np.random.choice(avail_idx)
            explore_d = th.from_numpy(explore).to(dev, non_blocking=True)
            rand_d = th.from_numpy(rand_a).to(dev, non_blocking=True)
        else:
            eps_d = th.from_numpy(eps).to(dev).to(th.float32).unsqueeze(1)
            explore_d = (th.rand(n, N, device=dev) < eps_d).to(th.uint8).contiguous()
            rand_d = th.randint(0, A, (n, N), device=dev, dtype=th.int64)
        return self._finish_matrix(n, evaluate, eps_after, explore=explore_d, random_action=rand_d)

    def _finish_matrix(self, n, evaluate, eps_after, **explore):
        """The matrix game's only step: one act launch with the given exploration arguments, one env launch."""
        N, A, dev = self.n_agents, self.n_actions, self.mac.device
        # the worker's view of the game at the only step: obs = get_obs() (zeros), no last action, fresh hidden state
        obs = th.zeros(n, N, self.obs_shape, device=dev)
        last = th.zeros(n, N, A, device=dev) if self.args.last_action else None
        hidden = th.zeros(n * N, self.args.rnn_hidden_dim, device=dev)
        actions = self.mac.act(n, obs, last, None, hidden, **explore)
        self.mac.hidden_states = hidden                                                 # [n*N, H], as an unroll leaves it
        episodes = self.env.step(actions)
        self._keep = tuple(explore.values())
        if not evaluate:
            self.epsilon = eps_after
        rewards = episodes["r"].reshape(n)
        return episodes, rewards, [False] * n, n

    def _epsilon_after_multistep(self, steps_tot, n):
        """The worker's epsilon moved as steps_tot environment steps (at most 2^20; 'step' scale) or n episodes (any
        other scale) in sequence would move it."""
        k = min(steps_tot, 1 << 20) if self.args.epsilon_anneal_scale == 'step' else n
        v = epsilon_schedule(float(self.epsilon), self.anneal_epsilon, self.min_epsilon, k)
        return float(v[min(k, len(v) - 1)])

    # ---- multi-step episodes (rollout.py:52-149 for every instance at once) ------------------------------------------
    def _generate_multistep(self, evaluate, random_select, draws, philox=None):
        """All env.n_envs instances step together until each has terminated or hit ``episode_limit``.

        Per step: ONE act launch (``mac.act``) over the (instance, agent) rows -- agent forward with the carried hidden
        state and the last actions (share_params.py:37-60), availability mask (``-inf``, first maximum) and exploration
        (share_params.py:62-72) -- then ``env.step``, then ONE ``marl_rollout_record`` launch that writes what the step
        produced into the episode buffers.  Nothing in the step loop waits for the GPU: the record kernel stores the
        number of instances still active into a page-locked host word that the loop polls, a step issued after
        every instance has finished does nothing on the device, and the one synchronisation of the call reads the
        device step counter at the end.  Every hidden-state row advances on every step in which some instance is
        active (finished instances feed their frozen observation and last action).  Finished instances are frozen and their remaining steps are
        the reference's padding (rollout.py:122-133): zeros everywhere, ``padded = 1``, ``terminated = 1``; the trailing
        observation / state / availability read after an instance's last step fill ``o_next`` / ``s_next`` /
        ``avail_u_next`` (rollout.py:106-120).

        RNG contract: ``draws=(explore_u, choice_u)``, two [n, episode_limit, N] arrays of uniforms in [0, 1) (host
        numpy or device tensors); agent a of instance e explores at step t iff explore_u[e, t, a] < epsilon_t and then
        takes the floor(choice_u * n_available)-th available action -- the same rule as oracle.rollout_oracle, so a
        seeded run is bit-identical to the sequential restatement.  ``philox`` (a ``PhiloxDraws`` of the call's seed and
        episode_base, rng="philox") has every act launch draw the same rule's uniforms itself, step t from counter word
        t; no [n, episode_limit, N] array exists.  Anything else draws the uniforms on the device.  Every instance
        starts the call from the worker's current epsilon (they run side by side) and anneals it per step; afterwards
        the worker's epsilon has moved by the total number of environment steps, as n sequential episodes would have
        moved it."""
        if random_select:
            raise NotImplementedError("random_select is not used by the in-scope drivers")
        env, mac, dev = self.env, self.mac, self.mac.device
        n, N, A, O, S, T = env.n_envs, self.n_agents, self.n_actions, self.obs_shape, self.state_shape, self.episode_limit
        f = lambda *shape: th.zeros(*shape, dtype=th.float32, device=dev)
        ep = dict(o=f(n, T, N, O), s=f(n, T, S), u=th.zeros(n, T, N, 1, dtype=th.int64, device=dev), r=f(n, T, 1),
                  o_next=f(n, T, N, O), s_next=f(n, T, S), avail_u=f(n, T, N, A), avail_u_next=f(n, T, N, A),
                  u_onehot=f(n, T, N, A), padded=th.ones(n, T, 1, device=dev), terminated=th.ones(n, T, 1, device=dev))
        if philox is None:
            if isinstance(draws, (tuple, list)):
                explore_u, choice_u = (th.as_tensor(d, dtype=th.float64, device=dev) for d in draws)
            else:
                explore_u = th.rand(n, T, N, dtype=th.float64, device=dev)
                choice_u = th.rand(n, T, N, dtype=th.float64, device=dev)
        eps = 0.0 if evaluate else float(self.epsilon)
        if self.args.epsilon_anneal_scale == 'episode':
            eps = eps - self.anneal_epsilon if eps > self.min_epsilon else eps
        if philox is None:
            explore_u, choice_u = explore_u.transpose(0, 1).contiguous(), choice_u.transpose(0, 1).contiguous()   # [T, n, N]
        env.reset()
        hidden = th.zeros(n * N, self.args.rnn_hidden_dim, device=dev)
        last = f(n, N, A)
        active = th.ones(n, dtype=th.bool, device=dev)
        rewards = th.zeros(n, dtype=th.float64, device=dev)
        actions = th.empty(n, N, dtype=th.int64, device=dev)
        onehot = th.empty(n, N, A, dtype=th.float32, device=dev)
        counters = th.zeros(T + 2, dtype=th.int32, device=dev)      # [t]: active at the start of step t, [T]: their sum
        counters[0:1].fill_(n)              # fills, not scalar copies: no host synchronisation
        counters[T:T + 1].fill_(n)
        if self._active_host is None:
            self._active_host = th.zeros(1, dtype=th.int32).pin_memory()
        host = self._active_host.numpy()
        host[0] = n                          # the previous call ended with a synchronisation: no launch still writes it
        dims = L.Dims(n, T, N, A, O, S)
        ep_s = L.EpisodeF32(*(ep[k].data_ptr() for k in L.EPISODE_KEYS))
        grab = lambda: tuple(x.to(dev, th.float32).contiguous() for x in (env.get_obs(), env.get_state(), env.get_avail_actions()))
        reward = term = None
        t = 0
        with th.no_grad():
            for t in range(T):
                if host[0] == 0:             # every instance has finished (a stale read only adds steps that do nothing)
                    break
                obs, state, avail = grab()
                if t == 0:                   # every instance is active: step 0 opens with the first observation
                    ep["o"][:, 0] = obs
                    ep["s"][:, 0] = state
                    ep["avail_u"][:, 0] = avail
                else:                        # close step t-1, open step t (the getters are consumed before env.step)
                    self._record(dims, t, ep_s, obs, state, avail, actions, onehot, reward, term, active, last, rewards, counters)
                explore = (dict(explore_u=explore_u[t], choice_u=choice_u[t]) if philox is None else
                           dict(philox=philox._replace(step=t)))
                mac.act(n, obs, last, avail, hidden, eps=eps, gate=counters[t:], actions=actions, onehot=onehot, **explore)
                reward, term = env.step(actions, active)
                reward = reward.to(dev, th.float64).contiguous()
                term = term.to(dev, th.bool).contiguous()
                if self.args.epsilon_anneal_scale == 'step':
                    eps = eps - self.anneal_epsilon if eps > self.min_epsilon else eps
            else:
                t = T
            obs, state, avail = grab()       # what the instances that acted last see afterwards
            self._record(dims, t, ep_s, obs, state, avail, actions, onehot, reward, term, active, last, rewards, counters)
            steps_tot = int(counters[T].item())          # the call's one synchronisation
        if not evaluate:
            self.epsilon = self._epsilon_after_multistep(steps_tot, n)
        mac.hidden_states = hidden
        return ep, rewards, [False] * n, steps_tot
