"""The shared controller (SharedMAC) with and without the last-action input block (args.last_action).

In one run it times, with last_action on (the default [obs | last action | agent id] input) and off ([obs | agent id]):
  * step: QLearner.train, QMIX, on the fused device step at the config-2/3/4 shapes (synthetic.CONFIGS: 2s3z, 3s5z,
    27m_vs_30m; CUDA graph replay, device-resident batch, so no host->device copy is timed);
  * act: one SharedMAC.act call (one marl_agent_act_input launch) at 256 and 4096 instances, at the same agent shapes.
The two settings are timed alternately in rounds (host clock around `steps` calls that end in a device synchronisation) and
the median per-call time of the rounds is reported with the spread.  The GPU name and power limit are read in the same run.
usage: python tools/shared_input_bench.py [--quick] [--out FILE]
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

import torch

from marl_b200.common.arguments import default_args
from marl_b200.controller.share_params import SharedMAC
from marl_b200.synthetic import CONFIGS, synthetic_batch
from tools.rollout_bench import gpu_info

SHAPES = [("cfg2", "2s3z"), ("cfg3", "3s5z"), ("cfg4", "27m_vs_30m")]


def _args(c, last_action):
    args = default_args(alg="qmix", n_agents=c["N"], n_actions=c["A"], obs_shape=c["O"], state_shape=c["S"],
                        episode_limit=c["T"], map="bench", model_dir="/tmp/marl_b200_model", last_action=last_action)
    args.target_update_cycle = 10 ** 9
    return args


def _rounds(arms, rounds, steps):
    """arms: {key: callable doing one timed call}; alternated in rounds, median and spread of the per-call time in us."""
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, f in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                f()
            torch.cuda.synchronize()
            times[k].append((time.perf_counter() - t0) / steps * 1e6)
    return {k: (round(statistics.median(v), 1), [round(min(v), 1), round(max(v), 1)]) for k, v in times.items()}


def step_case(cfg, name, rounds, steps):
    from marl_b200.algorithm.q_learner import QLearner
    c = dict(CONFIGS[name])
    b = synthetic_batch(0, c["B"], c["T"], c["N"], c["A"], c["O"], c["S"])
    batch = {k: torch.as_tensor(v, device="cuda") for k, v in b.items()}
    batch = {k: (v.to(torch.int64) if k == "u" else v.to(torch.float32)) for k, v in batch.items()}
    learners, counter = {}, {}
    for la in (True, False):
        torch.manual_seed(0)
        args = _args(c, la)
        learners[la] = QLearner(SharedMAC(args), args)
        for i in range(4):                        # eager sightings, graph capture, a replay
            learners[la].train(batch, i)
        counter[la] = 4
    res = {"cfg": cfg, "map": name, "alg": "qmix", "B": c["B"], "T": c["T"], "N": c["N"], "A": c["A"], "O": c["O"]}

    def arm(la):
        def f():
            learners[la].train(batch, counter[la])
            counter[la] += 1
        return f
    t = _rounds({"on": arm(True), "off": arm(False)}, rounds, steps)
    for k, (med, spread) in t.items():
        res[f"us_step_last_action_{k}"], res[f"us_step_last_action_{k}_spread"] = med, spread
    res["off_over_on"] = round(t["off"][0] / t["on"][0], 3)
    del learners
    torch.cuda.empty_cache()
    return res


def act_case(cfg, name, n, rounds, steps):
    c = dict(CONFIGS[name])
    N, A, O = c["N"], c["A"], c["O"]
    g = torch.Generator(device="cuda").manual_seed(0)
    obs = torch.randn(n, N, O, device="cuda", generator=g)
    last = torch.zeros(n, N, A, device="cuda")
    avail = torch.ones(n, N, A, device="cuda")
    arms = {}
    for la in (True, False):
        torch.manual_seed(0)
        mac = SharedMAC(_args(c, la))
        hidden = torch.zeros(n * N, 64, device="cuda")
        actions = torch.empty(n, N, dtype=torch.int64, device="cuda")
        arms["on" if la else "off"] = (lambda mac=mac, h=hidden, a=actions, l=(last if la else None):
                                       mac.act(n, obs, l, avail, h, actions=a))
    for f in arms.values():
        f()
    t = _rounds(arms, rounds, steps)
    res = {"cfg": cfg, "map": name, "n": n, "N": N, "A": A, "O": O}
    for k, (med, spread) in t.items():
        res[f"us_act_last_action_{k}"], res[f"us_act_last_action_{k}_spread"] = med, spread
    res["off_over_on"] = round(t["off"][0] / t["on"][0], 3)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_shared_input.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("shared_input_bench needs a CUDA device")
    rounds, steps, act_steps = (2, 5, 20) if a.quick else (7, 20, 200)
    out = {"gpu": gpu_info(), "rounds": rounds, "steps_per_round": steps, "act_calls_per_round": act_steps,
           "step": [step_case(cfg, name, rounds, steps) for cfg, name in SHAPES],
           "act": [act_case(cfg, name, n, rounds, act_steps) for cfg, name in SHAPES for n in (256, 4096)]}
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
