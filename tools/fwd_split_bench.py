"""A/B of the split forward (marl_fwd_split_enable) in one process: two learners of the same seed, one captured with the
split forward and one without, timed in alternating windows of graph-replayed steps on one device batch.

usage: fwd_split_bench.py [--alg qmix,vdn] [--B 32,48,59] [--steps 200] [--rounds 3]
Prints one line per (alg, B): ms per step of each arm (median of the rounds), the difference, and the plan the call took."""
import argparse
import ctypes as C
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.join(os.path.dirname(__file__), ".."))
import torch
from bench import make_args, SHAPE, to_device_batch
from marl_b200 import _lib as L
from marl_b200.algorithm.q_learner import QLearner
from marl_b200.controller.share_params import SharedMAC
from marl_b200.synthetic import synthetic_batch


def learner_for(alg, shape, split):
    prev = L.load().marl_fwd_split_enable(split)
    try:
        args = make_args(alg)
        torch.manual_seed(0)
        lr = QLearner(SharedMAC(args), args)
        db = to_device_batch(torch, synthetic_batch(0, **shape), shape["T"])
        for i in range(5):                      # capture + warm-up under this setting
            lr.train(db, i)
        torch.cuda.synchronize()
        return lr, db
    finally:
        L.load().marl_fwd_split_enable(prev)


def window(lr, db, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(steps):
        lr.train(db, 100 + i)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--alg", default="qmix,vdn")
    ap.add_argument("--B", default=str(SHAPE["B"]))
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--rounds", type=int, default=3)
    opt = ap.parse_args()
    props = torch.cuda.get_device_properties(0)
    print(json.dumps({"device": props.name, "sms": props.multi_processor_count}))
    for alg in opt.alg.split(","):
        for B in (int(x) for x in opt.B.split(",")):
            shape = dict(SHAPE, B=B)
            arms = {s: learner_for(alg, shape, s) for s in (1, 0)}
            took = arms[1][0].launches_per_step - arms[0][0].launches_per_step == 3
            ms = {1: [], 0: []}
            for _ in range(opt.rounds):
                for s in (1, 0):
                    ms[s].append(window(*arms[s], opt.steps))
            on, off = statistics.median(ms[1]), statistics.median(ms[0])
            print(json.dumps({"alg": alg, "B": B, "rows": B * SHAPE["N"], "split_taken": took, "ms_split": round(on, 4),
                              "ms_one_launch": round(off, 4), "delta_pct": round(100 * (on / off - 1), 2),
                              "rounds_split": [round(x, 4) for x in ms[1]], "rounds_one_launch": [round(x, 4) for x in ms[0]]}))
            del arms
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
