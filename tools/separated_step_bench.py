"""Learner step time with one network per agent (SeparatedMAC, reuse_network=False).

At the config-2/3/4 shapes (synthetic.CONFIGS: 2s3z QMIX, 3s5z QPLEX, 27m_vs_30m QTRAN-base, plus 27m_vs_30m with QMIX,
whose module path exists: QTRAN-base has no module-path step) it times, in one run:
  * fused: QLearner.train on the fused device step, per-agent weights in the recurrence and the batched dense layers
    (CUDA graph replay);
  * modules: the same learner with train_through_modules=True, autograd over each agent's own unroll;
  * shared: the parameter-sharing learner (SharedMAC, reuse_network=True) on its fused step at the same shape.
The batch is device-resident (fp32 CUDA tensors), so no host->device copy is timed.  Each train() call ends in a
synchronisation; the arms are timed alternately in rounds (host clock around `steps` calls) and the median per-step
time of the rounds is reported.  Before timing, the first loss of the fused step is checked against the module path on
identical weights (relative 1e-4); a disagreement fails the run.  The GPU name and power limit are read in the same run.
usage: python tools/separated_step_bench.py [--quick] [--out FILE]
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
from marl_b200.controller.share_params import SeparatedMAC, SharedMAC
from marl_b200.synthetic import CONFIGS, synthetic_batch
from tools.rollout_bench import gpu_info

CASES = [("cfg2", "2s3z", "qmix"), ("cfg3", "3s5z", "qplex"), ("cfg4", "27m_vs_30m", "qtran_base"), ("cfg4", "27m_vs_30m", "qmix")]


def _learner(c, alg, separated, modules=False):
    from marl_b200.algorithm.q_learner import QLearner
    from marl_b200.algorithm.qtran_learner import QTRANLearner
    args = default_args(alg=alg, n_agents=c["N"], n_actions=c["A"], obs_shape=c["O"], state_shape=c["S"],
                        episode_limit=c["T"], map="bench", model_dir="/tmp/marl_b200_model")
    args.reuse_network = not separated
    args.train_through_modules = modules
    args.target_update_cycle = 10 ** 9
    torch.manual_seed(0)
    mac = SeparatedMAC(args) if separated else SharedMAC(args)
    return (QTRANLearner if alg == "qtran_base" else QLearner)(mac, args)


def _device_batch(c):
    b = synthetic_batch(0, c["B"], c["T"], c["N"], c["A"], c["O"], c["S"])
    out = {k: torch.as_tensor(v, device="cuda") for k, v in b.items()}
    out = {k: (v.to(torch.int64) if k == "u" else v.to(torch.float32)) for k, v in out.items()}
    return out


def _time(learner, batch, steps, step0):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(steps):
        learner.train(batch, step0 + i)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / steps * 1e6


def case(cfg, name, alg, rounds, steps, mod_steps):
    c = dict(CONFIGS[name])
    batch = _device_batch(c)
    arms = {"fused": _learner(c, alg, True), "shared": _learner(c, alg, False)}
    if alg != "qtran_base":
        arms["modules"] = _learner(c, alg, True, modules=True)
    res = {"cfg": cfg, "map": name, "alg": alg, "B": c["B"], "T": c["T"], "N": c["N"], "A": c["A"], "O": c["O"],
           "params_separated": arms["fused"]._flat.numel, "params_shared": arms["shared"]._flat.numel}
    first = {k: l.train(batch, 0) for k, l in arms.items()}
    if "modules" in first and abs(first["fused"] - first["modules"]) > 1e-4 * abs(first["modules"]):
        raise SystemExit(f"{cfg} {alg}: fused loss {first['fused']} != module path {first['modules']}")
    res["loss_fused"], res["loss_modules"] = first["fused"], first.get("modules")
    for k, l in arms.items():                  # warm-up: eager sightings, graph capture, replays
        for i in range(3):
            l.train(batch, 1 + i)
    times = {k: [] for k in arms}
    for r in range(rounds):
        for k, l in arms.items():
            times[k].append(_time(l, batch, mod_steps if k == "modules" else steps, 10 + r * steps))
    for k, v in times.items():
        res[f"us_{k}"] = round(statistics.median(v), 1)
        res[f"us_{k}_spread"] = [round(min(v), 1), round(max(v), 1)]
    if "modules" in arms:
        res["modules_over_fused"] = round(res["us_modules"] / res["us_fused"], 2)
    res["fused_over_shared"] = round(res["us_fused"] / res["us_shared"], 3)
    del arms
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--quick", action="store_true")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_separated_step.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("separated_step_bench needs a CUDA device")
    rounds, steps, mod_steps = (2, 5, 2) if a.quick else (5, 20, 4)
    out = {"gpu": gpu_info(), "rounds": rounds, "steps_per_round": steps, "module_steps_per_round": mod_steps,
           "cases": [case(cfg, name, alg, rounds, steps, mod_steps) for cfg, name, alg in CASES]}
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
