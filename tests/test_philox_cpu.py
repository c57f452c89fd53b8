"""Host side of the Philox exploration form (rng="philox"): the loop-free epsilon schedule against the loops it
replaced, bit for bit; the known-answer block that pins numpy's Philox as the tests' reference generator; the ctypes
mirror of marl_act_philox; and the argument checks of BatchedRolloutWorker.generate_episodes."""
import ctypes
import os
import shutil
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest

from marl_b200 import _lib as L
from marl_b200.rollout import BatchedRolloutWorker, epsilon_schedule

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
# Random123's known answer for Philox4x64-10, counter 0 and key 0
KAT_ZERO = (0x16554d9eca36314c, 0xdb20fe9d672d0fdc, 0xd7e772cee186176b, 0x7e68b68aec7ba23b)
DEFAULTS = (1.0, (1.0 - 0.05) / 50000, 0.05)          # the reference's epsilon, anneal_epsilon, min_epsilon


def _loop_schedule(cur, anneal, min_eps, k):
    out = [cur]
    for _ in range(k):
        cur = cur - anneal if cur > min_eps else cur
        out.append(cur)
    return out


def _expand(p, k):
    return [p[min(i, len(p) - 1)] for i in range(k + 1)]


SCHEDULES = [DEFAULTS + (200000,),                     # the reference's defaults over 200000 episodes
             (0.5, 0.01, 0.02, 1000), (0.5, 0.01, 0.02, 48),   # crosses the minimum / stops short of it
             (0.05, 0.01, 0.05, 100), (0.01, 0.01, 0.05, 100),   # starts at / below the minimum
             (0.9, 0.0, 0.05, 500), (0.7, 0.003, 0.05, 1), (0.7, 0.003, 0.05, 0), (1.0, 1e-18, 0.5, 300),
             (0.3, 0.3, 0.0, 5), (0.25, 0.07, 0.0, 10), (1.0, 2.0 ** -40, 0.05, 5000)]


@pytest.mark.parametrize("cur,anneal,min_eps,k", SCHEDULES)
def test_schedule_equals_the_sequential_loop(cur, anneal, min_eps, k):
    p = epsilon_schedule(cur, anneal, min_eps, k)
    want = _loop_schedule(cur, anneal, min_eps, k)
    assert p.dtype == np.float64 and 1 <= len(p) <= k + 1
    assert np.array_equal(np.array(_expand(p, k)), np.array(want))        # bit for bit (no tolerance)
    assert len(p) == 1 or p[-2] != p[-1]                                   # the prefix ends where the values stop changing


def test_schedule_table_stays_short_with_the_reference_defaults():
    """(1 - 0.05) / anneal = 50000 subtractions in exact arithmetic; float64 rounding leaves v_50000 a hair above 0.05, so
    the schedule takes one more: the table is v_0 .. v_50001, not 2^22 values."""
    p = epsilon_schedule(*DEFAULTS, 1 << 22)
    assert len(p) == 50002 and p[-1] <= DEFAULTS[2] < p[-2]


def _worker(scale, epsilon, anneal, min_eps):
    args = SimpleNamespace(episode_limit=1, n_actions=3, n_agents=2, state_shape=1, obs_shape=1, epsilon=epsilon,
                           anneal_epsilon=anneal, min_epsilon=min_eps, epsilon_anneal_scale=scale, seed=0)
    return BatchedRolloutWorker(SimpleNamespace(n_envs=4), None, args)


def _loop_epsilons(w, n, evaluate):
    """BatchedRolloutWorker._epsilons as a loop over the episodes (the sequential reference, rollout.py:47-49, 103-104)."""
    eps = np.empty(n, dtype=np.float64)
    cur = w.epsilon
    for e in range(n):
        epsilon = 0 if evaluate else cur
        if w.args.epsilon_anneal_scale == 'episode':
            epsilon = epsilon - w.anneal_epsilon if epsilon > w.min_epsilon else epsilon
        eps[e] = epsilon
        if w.args.epsilon_anneal_scale == 'step':
            epsilon = epsilon - w.anneal_epsilon if epsilon > w.min_epsilon else epsilon
        if not evaluate:
            cur = epsilon
    return eps, cur


def _loop_after_multistep(w, steps_tot, n):
    cur = float(w.epsilon)
    if w.args.epsilon_anneal_scale == 'step':
        for _ in range(min(steps_tot, 1 << 20)):
            if not cur > w.min_epsilon:
                break
            cur -= w.anneal_epsilon
    else:
        for _ in range(n):
            cur = cur - w.anneal_epsilon if cur > w.min_epsilon else cur
    return cur


CASES = [("step",) + DEFAULTS, ("episode",) + DEFAULTS, ("step", 0.5, 0.01, 0.02), ("episode", 0.5, 0.01, 0.02),
         ("step", 0.05, 0.01, 0.05), ("episode", 0.01, 0.01, 0.05), ("step", 0.3, 0.0, 0.05), ("episode", 0.3, 0.0, 0.05),
         ("step", 0.2, 0.001, -0.5), ("episode", 0.2, 0.001, -0.5), ("constant", 0.4, 0.01, 0.05)]


@pytest.mark.parametrize("scale,epsilon,anneal,min_eps", CASES)
@pytest.mark.parametrize("n", [1, 7, 60, 3000])
@pytest.mark.parametrize("evaluate", [False, True])
def test_epsilons_and_table_equal_the_loop(scale, epsilon, anneal, min_eps, n, evaluate):
    w = _worker(scale, epsilon, anneal, min_eps)
    want, want_after = _loop_epsilons(w, n, evaluate)
    got, after = w._epsilons(n, evaluate)
    assert np.array_equal(got, want) and after == want_after
    table, after = w._eps_table(n, evaluate)
    assert 1 <= len(table) <= n and after == want_after
    assert np.array_equal(table[np.minimum(np.arange(n), len(table) - 1)], want)


def test_epsilons_carry_across_calls_like_one_call():
    """Two calls of n / 2 episodes leave the epsilon one call of n leaves (the schedule crosses the minimum in call 2)."""
    for scale in ("step", "episode"):
        one, two = _worker(scale, 0.5, 0.01, 0.02), _worker(scale, 0.5, 0.01, 0.02)
        want, one.epsilon = one._epsilons(80, False)
        a, two.epsilon = two._epsilons(40, False)
        b, two.epsilon = two._epsilons(40, False)
        assert np.array_equal(np.concatenate([a, b]), want) and two.epsilon == one.epsilon


@pytest.mark.parametrize("scale,epsilon,anneal,min_eps", CASES)
@pytest.mark.parametrize("steps_tot,n", [(0, 1), (1, 1), (57, 64), (6400, 64), ((1 << 20) + 5, 4096)])
def test_multistep_epsilon_update_equals_the_loop(scale, epsilon, anneal, min_eps, steps_tot, n):
    w = _worker(scale, epsilon, anneal, min_eps)
    assert w._epsilon_after_multistep(steps_tot, n) == _loop_after_multistep(w, steps_tot, n)


def test_multistep_epsilon_update_is_capped_at_2_pow_20_steps():
    w = _worker("step", 1.0, 1e-7, 0.0)                 # 10^7 steps to the minimum: the cap decides
    got = w._epsilon_after_multistep(1 << 22, 1)
    assert got == _loop_after_multistep(w, 1 << 22, 1) and got > 0.5


def test_numpy_philox_reproduces_the_known_answer_block():
    """The tests' reference: np.random.Philox(counter=c - 1, key=k).random_raw(4) is the block of counter c (numpy
    increments before it generates; the counter wraps modulo 2^256)."""
    assert tuple(int(x) for x in np.random.Philox(counter=(1 << 256) - 1, key=0).random_raw(4)) == KAT_ZERO
    g = np.random.Philox(counter=0, key=0)
    g.state = {"bit_generator": "Philox", "state": {"counter": np.array([2 ** 64 - 1] * 4, dtype=np.uint64),
                                                    "key": np.zeros(2, dtype=np.uint64)},
               "buffer": np.zeros(4, dtype=np.uint64), "buffer_pos": 4, "has_uint32": 0, "uinteger": 0}
    assert tuple(int(x) for x in g.random_raw(4)) == KAT_ZERO
    # Generator.random() is (word >> 11) * 2^-53 on the block's words in order
    c, k = (5 + (3 << 64) + (2 << 128)), 123
    words = np.random.Philox(counter=c - 1, key=k).random_raw(2)
    pair = np.random.Generator(np.random.Philox(counter=c - 1, key=k)).random(2)
    assert np.array_equal(pair, (words >> np.uint64(11)).astype(np.float64) * 2.0 ** -53)


def test_act_philox_mirror_has_the_headers_layout(tmp_path):
    if shutil.which("gcc") is None:
        pytest.skip("no C compiler")
    fields = [f for f, _ in L.ActPhilox._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "marl_b200.h"', 'int main(void) {',
             '  printf("size %zu\\n", sizeof(marl_act_philox));']
    lines += [f'  printf("{f} %zu\\n", offsetof(marl_act_philox, {f}));' for f in fields]
    lines += ['  return 0;', '}']
    (tmp_path / "probe.c").write_text("\n".join(lines))
    r = subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(tmp_path / "probe.c"), "-o", str(tmp_path / "probe")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    got = dict(line.split() for line in subprocess.run([str(tmp_path / "probe")], capture_output=True,
                                                       text=True).stdout.splitlines())
    assert int(got["size"]) == ctypes.sizeof(L.ActPhilox)
    for f in fields:
        assert int(got[f]) == getattr(L.ActPhilox, f).offset, f


def test_generate_episodes_rejects_bad_rng_arguments_before_any_work():
    w = _worker("step", 0.5, 0.01, 0.02)
    with pytest.raises(ValueError):
        w.generate_episodes(rng="cuda")
    with pytest.raises(ValueError):
        w.generate_episodes(rng="philox", draws=(np.zeros((4, 1, 2)), np.zeros((4, 1, 2))))
    assert w.episode_base == 0
