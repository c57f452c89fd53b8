"""QMIX learner step and mixing kernel time against qmix_hidden_dim E.

Times, in one run, for E in {16, 32, 64, 128}:
  * step: QLearner.train on the fused device step (CUDA graph replay, batch resident in HBM as fp32 CUDA tensors) at the
    config-2 shape (2s3z: B 32, T 120, N 5, S 120) and at config 5's learner shape (4096 matrix-game episodes, T 1, N 2);
    each train() call ends in a synchronisation.  The widths are interleaved in rounds after a warm-up of every width, and
    the median per-step time over all timed steps (>= 200 per width and shape) is reported;
  * mix: marl_qmix_td_fwd_bwd with flags 3 (the mixing kernel alone: TD forward and backward of eval and target mixer, no
    hyper-network GEMMs, no fused selection) at the config-2 sample count, CUDA events around 200 launches, median of rounds.
Writes the GPU name and power limit beside the times (default profiles/r8_qmix_embed.json).  Needs a CUDA device.
usage: python tools/qmix_embed_bench.py [--steps 200] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

import torch

from marl_b200 import _lib as L
from marl_b200.common.arguments import default_args
from marl_b200.controller.share_params import SharedMAC
from marl_b200.network.mixer import hy_cols
from marl_b200.synthetic import CONFIGS, synthetic_batch
from tools.rollout_bench import gpu_info

EMBEDS = (16, 32, 64, 128)
SHAPES = {"cfg2_2s3z": CONFIGS["2s3z"], "cfg5_matrix_game_4096": CONFIGS["matrix_game_4096"]}


def _learner(c, E):
    from marl_b200.algorithm.q_learner import QLearner
    args = default_args(alg="qmix", n_agents=c["N"], n_actions=c["A"], obs_shape=c["O"], state_shape=c["S"],
                        episode_limit=c["T"], map="bench", model_dir="/tmp/marl_b200_model", qmix_hidden_dim=E)
    args.target_update_cycle = 10 ** 9
    torch.manual_seed(0)
    return QLearner(SharedMAC(args), args)


def _device_batch(c):
    b = synthetic_batch(0, c["B"], c["T"], c["N"], c["A"], c["O"], c["S"])
    return {k: torch.as_tensor(v, device="cuda").to(torch.int64 if k == "u" else torch.float32) for k, v in b.items()}


def time_steps(steps, rounds=8):
    out = {}
    for shape, c in SHAPES.items():
        batch = _device_batch(c)
        learners = {E: _learner(c, E) for E in EMBEDS}
        for E, lr in learners.items():                       # eager sightings, graph capture, replays
            for i in range(10):
                lr.train(batch, i)
        per = {E: [] for E in EMBEDS}
        n = -(-steps // rounds)
        for r in range(rounds):
            for E, lr in learners.items():
                torch.cuda.synchronize()
                for i in range(n):
                    t0 = time.perf_counter()
                    lr.train(batch, 10 + r * n + i)          # (ends in a stream synchronisation)
                    per[E].append(time.perf_counter() - t0)
        out[shape] = {str(E): {"median_us": 1e6 * statistics.median(v), "steps": len(v),
                               "loss": float(learners[E].train(batch, 10 ** 6))} for E, v in per.items()}
    return out


def time_mix(launches=200, rounds=5):
    c = CONFIGS["2s3z"]
    N, A, S, B, T = c["N"], c["A"], c["S"], c["B"], c["T"]
    M = B * T
    out = {}
    g = torch.Generator(device="cuda").manual_seed(0)
    rnd = lambda *s: torch.randn(*s, device="cuda", generator=g)
    for E in EMBEDS:
        Cc = hy_cols(N, E)
        hy, hy_t, dhy = rnd(M, Cc), rnd(M, Cc), torch.empty(M, Cc, device="cuda")
        wb2, bb2 = rnd(E), rnd(1)
        q, qt, r = rnd(M, N), rnd(M, N), rnd(M)
        term, pad = torch.zeros(M, device="cuda"), torch.zeros(M, device="cuda")
        u = torch.zeros(M, N, dtype=torch.int64, device="cuda")
        q_tot, q_tot_t, dq, sc = (torch.empty(M, device="cuda"), torch.empty(M, device="cuda"),
                                  torch.empty(M, N, A, device="cuda"), torch.zeros(2, device="cuda"))
        gw, gb = torch.zeros(E, device="cuda"), torch.zeros(1, device="cuda")
        p = L.QmixParams(None, None, wb2.data_ptr(), bb2.data_ptr(), E)
        gs = L.QmixGrads(None, None, gw.data_ptr(), gb.data_ptr(), E)
        d = L.Dims(B, T, N, A, 1, S)

        def launch():
            L.call("marl_qmix_td_fwd_bwd", C.byref(d), C.byref(p), C.byref(p), hy.data_ptr(), hy.data_ptr(), q.data_ptr(), qt.data_ptr(),
                   u.data_ptr(), r.data_ptr(), term.data_ptr(), pad.data_ptr(), 0.99, hy.data_ptr(), hy_t.data_ptr(),
                   dhy.data_ptr(), q_tot.data_ptr(), q_tot_t.data_ptr(), dq.data_ptr(), C.byref(gs), sc.data_ptr(), 3,
                   None, None, None, L.stream_ptr())
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
        out[str(E)] = {"median_us": statistics.median(per), "launches": launches * rounds, "samples": M, "hy_cols": Cc}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_qmix_embed.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("qmix_embed_bench.py needs a CUDA device")
    torch.cuda.set_device(0)
    res = {"gpu": gpu_info(), "embeds": list(EMBEDS),
           "step": time_steps(a.steps), "mix_kernel_cfg2": time_mix(),
           "notes": "step: QLearner.train, graph replay, device-resident batch, host clock per synchronised step, median; "
                    "mix: marl_qmix_td_fwd_bwd flags=3 (mixing kernel only), CUDA events over 200 launches, median of 5"}
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
