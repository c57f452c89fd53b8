"""Exploration drawn inside the act launch (rng="philox") against the host- and torch-drawn forms.

In one run it times:
  * matrix: BatchedRolloutWorker.generate_episodes on BatchedMatrixGame at 2^12 / 2^16 / 2^20 / 2^22 instances with
    rng="numpy" (host draws in the reference's order), "device" (torch's generator outside the kernel) and "philox",
    alternated in rounds; host clock around calls that end in a device synchronisation, us per call and env-steps/s.
    Every call starts from epsilon 1.0 with the reference's anneal (2^20 instances cross min_epsilon inside the call);
  * act: the act launch alone at the config-2/3/4 agent shapes (N/A/O = 5/11/80, 8/14/128, 27/36/285) and 256 / 4096 /
    65536 instances, uniform form (explore_u / choice_u arrays) against Philox form, CUDA events around loops of launches,
    alternated in rounds; the uniform form is fed the Philox pairs (marl_philox_uniforms), and the two forms' actions
    must agree or the run fails;
  * multistep: generate_episodes on the ragged test game of tests/envs.py at 4096 instances, torch-drawn [n, T, N] arrays
    ("device") against "philox": us per environment step (one batched env.step of every instance) and the call's peak
    device memory (torch.cuda.max_memory_allocated above what was allocated before the call).
Medians over the rounds, with [min, max].  The GPU name and power limit are read in the same run.
usage: python tools/philox_rollout_bench.py [--quick] [--out FILE]
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

import numpy as np
import torch

from marl_b200 import _lib as L
from marl_b200.common.arguments import default_args
from marl_b200.controller.share_params import PhiloxDraws, SharedMAC
from marl_b200.env.single_state_matrix_game import BatchedMatrixGame
from marl_b200.rollout import BatchedRolloutWorker
from tests.envs import CountdownGameBatched
from tools.rollout_bench import gpu_info

H = 64
SHAPES = {"cfg2": (5, 11, 80), "cfg3": (8, 14, 128), "cfg4": (27, 36, 285)}
PAYOFF = [[8, -12, -12], [-12, 0, 0], [-12, 0, 0]]


def summary(v):
    return round(statistics.median(v), 2), [round(min(v), 2), round(max(v), 2)]


def host_timed(fn, calls):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(calls):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / calls * 1e6


def event_timed(fn, calls):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / calls


def matrix_case(n, rounds, forms):
    args = default_args(alg="qmix", n_agents=2, n_actions=3, obs_shape=1, state_shape=1, episode_limit=1)
    torch.manual_seed(0)
    worker = BatchedRolloutWorker(BatchedMatrixGame(PAYOFF, n), SharedMAC(args), args)
    np.random.seed(0)

    def call(rng):
        worker.epsilon = 1.0
        worker.generate_episodes(rng=rng)

    calls = max(1, (1 << 16) // n)
    for rng in forms:
        call(rng)                                          # warm-up: allocations, module load
    times = {rng: [] for rng in forms}
    for _ in range(rounds):
        for rng in forms:
            times[rng].append(host_timed(lambda: call(rng), 1 if rng == "numpy" and n >= 1 << 18 else calls))
    res = {"n": n, "calls_per_round": calls}
    for rng, v in times.items():
        med, spread = summary(v)
        res[f"us_call_{rng}"], res[f"us_call_{rng}_spread"] = med, spread
        res[f"env_steps_per_s_{rng}"] = round(n / (med * 1e-6))
    return res


def act_case(name, n, rounds, calls):
    N, A, O = SHAPES[name]
    args = default_args(alg="qmix", n_agents=N, n_actions=A, obs_shape=O, state_shape=4, episode_limit=1)
    torch.manual_seed(0)
    mac = SharedMAC(args)
    g = torch.Generator(device="cuda").manual_seed(n + N)
    obs = torch.randn(n, N, O, device="cuda", generator=g)
    last = torch.nn.functional.one_hot(torch.randint(0, A, (n, N), device="cuda", generator=g), A).float()
    avail = (torch.rand(n, N, A, device="cuda", generator=g) < 0.7).float()
    h0 = torch.randn(n * N, H, device="cuda", generator=g) * 0.5
    draws = PhiloxDraws(seed=1, episode_base=0, step=3)
    pairs = torch.empty(n * N, 2, dtype=torch.float64, device="cuda")
    L.call("marl_philox_uniforms", *draws, n, N, pairs.data_ptr(), L.stream_ptr())
    eu, cu = pairs[:, 0].contiguous(), pairs[:, 1].contiguous()
    acts = {k: torch.empty(n, N, dtype=torch.int64, device="cuda") for k in ("uniform", "philox")}
    hs = {k: h0.clone() for k in acts}
    arms = {"uniform": lambda: mac.act(n, obs, last, avail, hs["uniform"], explore_u=eu, choice_u=cu, eps=0.25,
                                       actions=acts["uniform"]),
            "philox": lambda: mac.act(n, obs, last, avail, hs["philox"], eps=0.25, philox=draws, actions=acts["philox"])}
    with torch.no_grad():
        for f in arms.values():
            f()
        torch.cuda.synchronize()
        if not torch.equal(acts["uniform"], acts["philox"]):
            raise SystemExit(f"{name} n={n}: the two exploration forms disagree")
        times = {k: [] for k in arms}
        for _ in range(rounds):
            for k, f in arms.items():
                times[k].append(event_timed(f, calls))
    res = {"cfg": name, "n": n, "N": N, "A": A, "O": O, "rows": n * N, "calls_per_round": calls}
    for k, v in times.items():
        res[f"us_act_{k}"], res[f"us_act_{k}_spread"] = summary(v)
    res["philox_over_uniform"] = round(res["us_act_philox"] / res["us_act_uniform"], 4)
    return res


def multistep_case(n, rounds):
    N, A, O, S, T = 3, 5, 4, 3, 60
    args = default_args(alg="qmix", n_agents=N, n_actions=A, obs_shape=O, state_shape=S, episode_limit=T)
    torch.manual_seed(0)
    env = CountdownGameBatched(n, n_agents=N, n_actions=A, episode_limit=T)
    worker = BatchedRolloutWorker(env, SharedMAC(args), args)
    n_steps = []
    step = env.step
    env.step = lambda a, act: n_steps.append(1) or step(a, act)
    forms = ("device", "philox")
    per_step, peak = {k: [] for k in forms}, {}
    for _ in range(rounds + 1):                            # round 0 warms up
        for rng in forms:
            worker.epsilon = 0.5
            torch.cuda.synchronize()
            before = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            n_steps.clear()
            t0 = time.perf_counter()
            worker.generate_episodes(rng=rng)
            torch.cuda.synchronize()
            per_step[rng].append((time.perf_counter() - t0) * 1e6 / len(n_steps))
            peak[rng] = torch.cuda.max_memory_allocated() - before
    res = {"n": n, "N": N, "A": A, "T": T, "env_steps_per_call": len(n_steps)}
    for rng in forms:
        res[f"us_per_env_step_{rng}"], res[f"us_per_env_step_{rng}_spread"] = summary(per_step[rng][1:])
        res[f"peak_bytes_{rng}"] = peak[rng]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7_philox_rollout.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("philox_rollout_bench needs a CUDA device")
    rounds, act_calls = (2, 5) if a.quick else (5, 50)
    sizes = (1 << 12, 1 << 16) if a.quick else (1 << 12, 1 << 16, 1 << 20, 1 << 22)
    out = {"gpu": gpu_info(), "rounds": rounds,
           "matrix": [matrix_case(n, min(rounds, 3), ("numpy", "device", "philox")) for n in sizes],
           "act": [act_case(name, n, rounds, act_calls) for name in SHAPES for n in (256, 4096, 65536)],
           "multistep": multistep_case(4096, rounds)}
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
