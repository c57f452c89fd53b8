"""Learner step, acting and rollout time against rnn_hidden_dim H.

Times, in one run, for H in {32, 64, 128}:
  * step: QLearner.train (QMIX) on the fused device step (CUDA graph replay, batch resident in HBM) at the config-2 shape
    (2s3z: B 32, T 120, N 5, S 120); each train() call ends in a synchronisation.  The widths are interleaved in rounds
    after a warm-up of every width; the median per-step time over all timed steps is reported;
  * act: SharedMAC.act and SeparatedMAC.act (one marl_agent_act_input / marl_agent_act_separated launch, greedy) over
    4096 instances at the config-2, 3 and 4 acting shapes, CUDA events around 200 launches, median of 5 rounds;
  * rollout: BatchedRolloutWorker.generate_episodes on 4096 matrix games (one env step per instance), env-steps per second
    over synchronised calls, median of rounds.
Writes the GPU name and power limit beside the times (default profiles/r9_rnn_hidden.json).  Needs a CUDA device.
usage: python tools/rnn_hidden_bench.py [--steps 200] [--out FILE]
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

WIDTHS = (32, 64, 128)
ACT_SHAPES = {"cfg2": (5, 11, 80), "cfg3": (8, 14, 128), "cfg4": (27, 36, 285)}      # N, A, O
INSTANCES = 4096


def _args(N, A, O, S, T, H, **kw):
    a = default_args(alg="qmix", n_agents=N, n_actions=A, obs_shape=O, state_shape=S, episode_limit=T, map="bench",
                     model_dir="/tmp/marl_b200_model", rnn_hidden_dim=H)
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def time_steps(steps, rounds=8):
    from marl_b200.algorithm.q_learner import QLearner
    c = CONFIGS["2s3z"]
    b = synthetic_batch(0, c["B"], c["T"], c["N"], c["A"], c["O"], c["S"])
    batch = {k: torch.as_tensor(v, device="cuda").to(torch.int64 if k == "u" else torch.float32) for k, v in b.items()}
    learners = {}
    for H in WIDTHS:
        args = _args(c["N"], c["A"], c["O"], c["S"], c["T"], H, target_update_cycle=10 ** 9)
        torch.manual_seed(0)
        learners[H] = QLearner(SharedMAC(args), args)
    for H, lr in learners.items():
        for i in range(10):
            lr.train(batch, i)
    per = {H: [] for H in WIDTHS}
    n = -(-steps // rounds)
    for r in range(rounds):
        for H, lr in learners.items():
            torch.cuda.synchronize()
            for i in range(n):
                t0 = time.perf_counter()
                lr.train(batch, 10 + r * n + i)          # (ends in a stream synchronisation)
                per[H].append(time.perf_counter() - t0)
    return {str(H): {"median_us": 1e6 * statistics.median(v), "steps": len(v)} for H, v in per.items()}


def time_act(launches=200, rounds=5):
    out = {}
    for name, (N, A, O) in ACT_SHAPES.items():
        for kind, cls in (("shared", SharedMAC), ("separated", SeparatedMAC)):
            for H in WIDTHS:
                torch.manual_seed(0)
                mac = cls(_args(N, A, O, 4, 10, H, reuse_network=kind == "shared"))
                n = INSTANCES
                g = torch.Generator(device="cuda").manual_seed(0)
                obs = torch.randn(n, N, O, device="cuda", generator=g)
                last = torch.zeros(n, N, A, device="cuda")
                avail = torch.ones(n, N, A, device="cuda")
                hidden = torch.zeros(n * N, H, device="cuda")
                actions = torch.empty(n, N, dtype=torch.int64, device="cuda")
                launch = lambda: mac.act(n, obs, last, avail, hidden, actions=actions)
                for _ in range(20):
                    launch()
                per = []
                for _ in range(rounds):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(launches):
                        launch()
                    e1.record()
                    e1.synchronize()
                    per.append(1e3 * e0.elapsed_time(e1) / launches)
                out[f"{name}_{kind}_H{H}"] = {"median_us": statistics.median(per), "instances": n, "N": N, "A": A, "O": O}
    return out


def time_rollout(rounds=20):
    from marl_b200.env.single_state_matrix_game import BatchedMatrixGame
    from marl_b200.rollout import BatchedRolloutWorker
    payoff = [[8, -12, -12], [-12, 0, 0], [-12, 0, 0]]
    out = {}
    for H in WIDTHS:
        args = _args(2, 3, 1, 1, 1, H)
        torch.manual_seed(0)
        worker = BatchedRolloutWorker(BatchedMatrixGame(payoff, INSTANCES), SharedMAC(args), args)
        for _ in range(5):
            worker.generate_episodes(rng="philox")
        per = []
        for _ in range(rounds):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            _, _, _, steps = worker.generate_episodes(rng="philox")
            torch.cuda.synchronize()
            per.append(steps / (time.perf_counter() - t0))
        out[str(H)] = {"median_env_steps_per_s": statistics.median(per), "envs": INSTANCES}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r9_rnn_hidden.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rnn_hidden_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "widths": list(WIDTHS), "step_qmix_cfg2": time_steps(a.steps), "act": time_act(),
           "rollout_matrix_game": time_rollout(),
           "notes": "step: QLearner.train (QMIX), graph replay, device-resident batch, host clock per synchronised step, "
                    "median; act: one greedy act launch over 4096 instances, CUDA events over 200 launches, median of 5; "
                    "rollout: 4096 matrix games, rng=philox, synchronised generate_episodes calls, median of 20"}
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
