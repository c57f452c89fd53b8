#!/usr/bin/env python
"""bench.py -- QMIX learner episode-samples/s (2s3z shape) + matrix-game env-steps/s on B200.

    python bench.py --gpus N --steps K --warmup W          (N>1: launched under torch.distributed.run)
    python bench.py --impl reference ...                   (the CPU path of the reference algorithm)
    python bench.py ... --dump-outputs DIR                 (+ what the last timed step computed, as DIR/<name>.npy)

One JSON line on stdout (rank 0).  A "step" is one ``QLearner.train()`` on one synthetic 2s3z-shaped
episode batch (BASELINE.json configs[1]: 5 agents, 11 actions, T=120, batch 32 per GPU).
  value : whole-job episode-samples/s with the batches already resident in HBM (CUDA events, max over ranks)
  e2e   : the same through the reference-facing call with pinned float64 HOST batches in the ReplayBuffer
          layout -- H2D copy, f64->f32 ingest and the loss read-back inside the timed region
  env   : matrix-game env-steps/s of the batched environment kernel (4096 envs and 2^24 envs)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SHAPE = dict(B=32, T=120, N=5, A=11, O=80, S=120)        # BASELINE.json configs[1]
FLOP_PER_STEP = 6.98e9                                   # SURVEY.md section 8(d), cfg 2 QMIX, B=32
BYTES_PER_STEP = 18.71e6                                 # each batch element read once as fp32 (u int64)
GRU_FWD_FLOP = 3 * 32 * 120 * 5 * 2 * (3 * 64 * 64)      # 3 unrolls x rows x (W_hh h): the sequential kernel
GRU_FWD_BYTES = 32 * 120 * 5 * 4 * (3 * 192 + 3 * 64 + 256)   # gi in (3 unrolls), hidden out (3), saved gates out (eval unroll)
ENV_BYTES = 140                                          # 16 B actions in + 124 B episode record out
# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` captures (profiles/)
NCU_TRAFFIC = {"gru_unroll_fwd_kernel": 44405504 + 3192832, "gru_unroll_bwd_kernel": 29584128 + 183808,
               "linear_fwd_kernel": 7062784, "matrix_game_step_kernel": 268475136 + 2043086000}   # profiles/r1c_ncu_full_gru.txt, r1b_ncu_full_env.txt
PAYOFF1 = [[8, -12, -12], [-12, 0, 0], [-12, 0, 0]]


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """SM clock / throttle reasons sampled every 5 ms DURING the timed regions (NVML; the same counters the
    nvidia-smi line of B200_PROFILING.md prints)."""

    def __init__(self, index=0):
        self.index, self.rows, self._stop, self.t = index, [], False, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.t = threading.Thread(target=self._loop, daemon=True)
            self.t.start()
        except Exception as e:      # noqa: BLE001
            self.err = repr(e)

    def _loop(self):
        nv, h = self.nv, self.h
        while not self._stop:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:   # noqa: BLE001
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.rows.append((sm, reasons))
            except Exception:       # noqa: BLE001
                pass
            time.sleep(0.005)

    def stop(self):
        if self.t is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: " + getattr(self, "err", "?")]}
        self._stop = True
        self.t.join(timeout=1)
        nv = self.nv
        sm = [r[0] for r in self.rows]
        mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        bits = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        seen = 0
        for _, r in self.rows:
            seen |= r
        reasons = sorted(n for n, b in bits.items() if seen & b)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(mx), "reasons": reasons,
                "samples": len(sm)}


def make_args(alg="qmix"):
    from marl_b200.common.arguments import default_args
    return default_args(alg=alg, n_agents=SHAPE["N"], n_actions=SHAPE["A"], obs_shape=SHAPE["O"],
                        state_shape=SHAPE["S"], episode_limit=SHAPE["T"], map="synthetic_2s3z")


def oracle_state(args, seed=0):
    import torch
    from oracle import marl_oracle as MO
    torch.manual_seed(seed)
    cfg = MO.make_cfg(alg=args.alg, n_agents=args.n_agents, n_actions=args.n_actions, obs_shape=args.obs_shape,
                      state_shape=args.state_shape, episode_limit=args.episode_limit)
    return MO, MO.LearnerState(cfg)


WORKLOAD = ("QMIX learner step, synthetic 2s3z-shaped batch (5 agents, 11 actions, T=120, batch 32 per GPU, RMSprop, "
            "double-Q)")


def host_threads():
    """All the host cores this process may use, whatever OMP_NUM_THREADS torchrun exported."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def reference_learner(alg, shape, cuda=False, seed=0):
    """The UNMODIFIED reference (oracle/_ref, staged by oracle/fetch_ref.py) when it travelled with the snapshot,
    else the oracle port of its CPU path.  Returns (train_fn(batch, step) -> loss, kind)."""
    import torch
    from oracle import fetch_ref as FR
    if FR.available():
        ns = FR.load()
        a = FR.make_args(ns, alg, shape["N"], shape["A"], shape["O"], shape["S"], shape["T"], cuda=cuda)
        torch.manual_seed(seed)
        mac = ns.SharedMAC(a)
        learner = (ns.QTRANLearner if alg == "qtran_base" else ns.QLearner)(mac, a)
        return (lambda batch, step: learner.train({k: v.copy() for k, v in batch.items()}, step)), "reference"
    if cuda:
        return None, "port"
    from marl_b200.common.arguments import default_args
    args = default_args(alg=alg, n_agents=shape["N"], n_actions=shape["A"], obs_shape=shape["O"], state_shape=shape["S"],
                        episode_limit=shape["T"], map="synthetic")
    MO, st = oracle_state(args, seed)
    return (lambda batch, step: MO.train_step(st, batch, step)[0]), "port"


def time_reference(steps, warmup, alg="qmix", shape=None, cuda=False):
    """episode-samples/s of the reference's own train() on the host cores (or, cuda=True, on this GPU with stock ATen
    kernels: the same-box GPU baseline of SURVEY.md section 8(c))."""
    import torch
    from marl_b200.synthetic import synthetic_batch
    shape = shape or SHAPE
    torch.set_num_threads(host_threads())
    train, kind = reference_learner(alg, shape, cuda=cuda)
    if train is None:
        return None
    batch = synthetic_batch(0, **shape)
    for i in range(warmup):
        train(batch, i)
    if cuda:
        torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(steps):
        train(batch, warmup + i)          # returns loss.item(): synchronises every step, like the reference's caller
    if cuda:
        torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return {"value": shape["B"] * steps / dt, "unit": "episode-samples/s", "ms_per_step": dt / steps * 1e3, "kind": kind,
            "cores": torch.get_num_threads(), "steps": steps, "warmup": warmup}


def run_reference(opt):
    """--impl reference: the reference's own QLearner.train on this box's host cores (rank 0 only), plus the same
    code with args.cuda=True on GPU 0 as `gpu_baseline`."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    steps, warm = opt.steps, max(1, min(opt.warmup, 3))
    r = time_reference(steps, warm)
    sample = (f"{steps} train steps (after {warm} warm-up) of one B=32 synthetic 2s3z-shaped batch through "
              + ("the UNMODIFIED reference QLearner.train (oracle/_ref), args.cuda=False" if r["kind"] == "reference"
                 else "the oracle port of the reference's CPU path (oracle/_ref was not staged)")
              + f", torch.set_num_threads({r['cores']})")
    gpu = None
    if torch.cuda.is_available() and r["kind"] == "reference":
        try:
            g = time_reference(10, 3, cuda=True)
            gpu = {"value": g["value"], "unit": g["unit"], "ms_per_step": g["ms_per_step"],
                   "what": "UNMODIFIED reference QLearner.train with args.cuda=True on this GPU (stock ATen / cuBLAS kernels; "
                           "o / o_next / avail stay on the host as in controller/share_params.py:132-134)", "steps": 10}
        except Exception as e:      # noqa: BLE001
            gpu = {"unavailable": repr(e)[:200]}
    line = {"impl": "reference", "metric": "QMIX learner episode-samples/sec (2s3z shape)", "value": r["value"],
            "unit": "episode-samples/s", "n_gpus": opt.gpus, "steps": steps, "warmup": warm,
            "ms_per_step": r["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": {"workload": WORKLOAD},
            "cpu_baseline": {"value": r["value"], "unit": "episode-samples/s", "cores": r["cores"], "kind": r["kind"],
                             "sample": sample},
            "gpu_baseline": gpu,
            "e2e": {"value": r["value"], "unit": "episode-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def bench_env(torch, dist, world, n_envs, iters, hbm_peak):
    """n_envs independent matrix games PER GPU (env instances shard over ranks, no collective)."""
    from marl_b200.env.single_state_matrix_game import BatchedMatrixGame
    env = BatchedMatrixGame(PAYOFF1, n_envs)
    acts = torch.randint(0, 3, (n_envs, 2), device="cuda", dtype=torch.int64)
    for _ in range(5):
        env.step(acts)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        env.step(acts)
    b.record()
    torch.cuda.synchronize()
    ms = torch.tensor([a.elapsed_time(b) / iters], device="cuda")
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms)
    rate = n_envs * world / (ms * 1e-3)
    gbs = rate / world * ENV_BYTES / 1e9
    return {"n_envs_per_gpu": n_envs, "value": rate, "unit": "env-steps/s", "us_per_launch": ms * 1e3,
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                         "traffic": NCU_TRAFFIC["matrix_game_step_kernel"] if n_envs == (1 << 24) else None, "note": "per GPU"}}


def to_device_batch(torch, hb, T):
    db = {k: torch.as_tensor(v, device="cuda") for k, v in hb.items()}
    db = {k: (v.to(torch.int64) if k == "u" else v.to(torch.float32)).contiguous() for k, v in db.items()}
    db["max_episode_len"] = T
    return db


class Timer:
    """CUDA-event timing of K train steps on the current stream, max over ranks; also the per-step median."""

    def __init__(self, torch, dist, world):
        self.torch, self.dist, self.world = torch, dist, world

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def run(self, K, step_fn):
        torch = self.torch
        import gc
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
        gc.collect()
        gc.disable()                 # (as timeit does: a generation-2 collection in the middle of a 0.4 ms step is a multi-ms outlier)
        try:
            self.barrier()
            evs[0].record()
            for i in range(K):
                step_fn(i)
                evs[i + 1].record()
            self.barrier()
        finally:
            gc.enable()
        per = [evs[i].elapsed_time(evs[i + 1]) for i in range(K)]
        self.last_per_step = per
        t = torch.tensor([evs[0].elapsed_time(evs[K]) / K, float(np.median(per))], device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t[0]), float(t[1])


def dp_check(torch, dist, world, rank, make_learner):
    """Data-parallel correctness INSIDE the multi-GPU run: (a) replicas stay bit-identical, (b) loss and parameters after 3
    steps agree with a single-GPU learner trained on the concatenated global batch (fp32 summation order differs: 1e-5)."""
    from marl_b200.synthetic import synthetic_batch
    Bg = 8 * world
    shape = dict(SHAPE, B=Bg, T=40)
    hb = synthetic_batch(4242, **shape)
    dp = make_learner(shape, seed=11)
    dp.enable_data_parallel()
    single = make_learner(shape, seed=11)
    db = to_device_batch(torch, hb, shape["T"])
    losses_dp, losses_1 = [], []
    gerr = None
    for i in range(3):
        losses_dp.append(dp.train(dict(db), i))          # every rank passes the GLOBAL batch; the learner takes its shard
        losses_1.append(single.train(dict(db), i))
        if i == 0:      # same parameters on both sides: the exchanged, normalised, clipped gradient must be the single-GPU one
            g_dp, g_1 = dp._flat.grad, single._flat.grad
            gerr = float((g_dp - g_1).abs().max() / g_1.abs().max())
    p_dp, p_1 = dp._flat.data.clone(), single._flat.data
    gathered = [torch.empty_like(p_dp) for _ in range(world)]
    dist.all_gather(gathered, p_dp)
    identical = all(bool(torch.equal(gathered[0], g)) for g in gathered[1:])
    scale = float(p_1.abs().max())
    perr = float((p_dp - p_1).abs().max()) / scale
    lerr = max(abs(a - b) / max(abs(b), 1e-30) for a, b in zip(losses_dp, losses_1))
    # The well-conditioned statements are the gradient of the first step and the losses.  The parameters are reported, not gated:
    # RMSprop's first updates are lr * g / sqrt(0.01 g^2) = 10 lr sign(g), so a gradient element at the summation-order noise
    # floor can land 2 * 10 * lr apart per step whatever the exchange does (tests/parity_util.py documents the same floor)
    ok = identical and lerr <= 1e-5 and gerr is not None and gerr <= 1e-5
    return {"replicas_bit_identical": identical, "loss_rel_err_vs_1gpu": lerr, "grad_rel_err_vs_1gpu_step0": gerr,
            "param_rel_err_vs_1gpu": perr, "param_noise_floor": 2 * 10 * dp.lr * 3 / scale, "steps": 3,
            "global_batch": Bg, "exchange": "peer" if getattr(dp, "_peer", None) is not None else "nccl", "ok": bool(ok)}


def run_ours(opt):
    import torch
    import torch.distributed as dist
    from marl_b200 import _lib as L
    from marl_b200.algorithm.q_learner import QLearner
    from marl_b200.algorithm.qtran_learner import QTRANLearner
    from marl_b200.common.arguments import default_args
    from marl_b200.common.replaybuffer import ReplayBuffer
    from marl_b200.controller.share_params import SharedMAC
    from marl_b200.env.single_state_matrix_game import BatchedMatrixGame
    from marl_b200.synthetic import synthetic_batch, KEYS, CONFIGS

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if os.environ.get("MARL_BENCH_PIN", "1") != "0":
        pin_to_gpu_numa(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    hbm_peak, peak_src = peaks()
    K, W = opt.steps, max(opt.warmup, 3)
    B = SHAPE["B"]
    tm = Timer(torch, dist, world)

    def make_learner(shape, alg="qmix", seed=0, name="synthetic_2s3z"):
        a = default_args(alg=alg, n_agents=shape["N"], n_actions=shape["A"], obs_shape=shape["O"], state_shape=shape["S"],
                         episode_limit=shape["T"], map=name)
        torch.manual_seed(seed)
        return (QTRANLearner if alg == "qtran_base" else QLearner)(SharedMAC(a), a)

    args = make_args()
    learner = make_learner(SHAPE)
    seeded = [t.clone() for t in learner_state(learner)] if opt.dump_outputs else None
    if world > 1:
        learner.enable_data_parallel()

    # Each rank holds its own shard: weak scaling, B=32 episodes per GPU, global batch 32*world.
    NB = 8                                            # 8 x 18.7 MB = 150 MB of inputs > 126 MB L2
    dev_batches, host_batches = [], []
    for i in range(NB):
        hb = synthetic_batch(1000 * rank + i, **SHAPE)
        dev_batches.append(to_device_batch(torch, hb, SHAPE["T"]))
        if i < 2:                                     # pinned float64 host copies in the ReplayBuffer layout
            pinned = {k: torch.from_numpy(v).pin_memory() for k, v in hb.items()}
            host_batches.append({k: t.numpy() for k, t in pinned.items()})
            host_batches[-1]["_keep"] = pinned
    if world > 1:
        learner._shard = lambda B_glob: (0, B_glob)  # every rank already holds exactly its shard

    def host_view(i):
        return {k: host_batches[i % 2][k] for k in KEYS}

    state = {"step": 0}

    def train(b):
        loss = learner.train(b, state["step"])
        state["step"] += 1
        return loss

    # resident batches are read in place, each through its own captured graph: run every batch through the eager
    # call and the capture call before anything is timed (W warm-up replays follow)
    for _ in range(4):               # eager sightings + the capture + one replay of every resident batch's graph
        for b in dev_batches:
            train(b)
    for i in range(W):
        train(dev_batches[i % NB])
    for i in range(max(W, 3)):
        train(host_view(i))

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # ---- value: device-resident batches ---------------------------------------------------------------------------------
    ms_dev, ms_dev_median = tm.run(K, lambda i: train(dev_batches[i % NB]))
    dev_max = float(max(tm.last_per_step))
    last = (dev_batches[(K - 1) % NB], state["step"] - 1)        # batch and train_step of the last timed step

    # ---- e2e (headline): the reference's own loop, runner.py:92-97 -- one freshly generated HOST episode is stored
    # (pinned float64 -> read over PCIe by the cast kernel -> fp32 ring row), a batch of 32 is sampled, train() returns the loss ----
    rb_args = make_args()
    rb_args.buffer_size = 512
    buf = ReplayBuffer(rb_args)
    for i in range(0, 512, B):                       # untimed: fill the ring
        buf.store_episode({k: dev_batches[(i // B) % NB][k] for k in KEYS})
    new_eps = []
    for i in range(8):
        hb = synthetic_batch(5000 + 1000 * rank + i, **dict(SHAPE, B=1))
        pinned = {k: torch.from_numpy(np.ascontiguousarray(v, dtype=np.float64)).pin_memory() for k, v in hb.items()}
        new_eps.append(({k: t.numpy() for k, t in pinned.items()}, pinned))
    ep_bytes = sum(v.nbytes for v in new_eps[0][0].values())
    np.random.seed(1234 + rank)

    def replay_step(i):
        buf.store_episode(new_eps[i % 8][0])
        train(buf.sample(B))

    # sampled batches come with whatever max_episode_len their episodes have; a (B, L) graph is captured at its third sighting
    # (~ms each), so the frequent lengths are let through before anything is timed, as in a long training run
    for i in range(max(W, 96)):
        replay_step(i)
    ms_replay, ms_replay_median = tm.run(K, replay_step)
    replay_max = float(max(tm.last_per_step))

    # ---- e2e, host-dict variant: a caller that keeps whole float64 batches in host memory (the reference's ReplayBuffer
    # layout) and hands one to train() every step: 35.6 MB over PCIe per step ---------------------------------------------
    ms_e2e_sync, _ = tm.run(K, lambda i: train(host_view(i)))
    h2d = learner.h2d_bytes_last
    hv = [host_view(0), host_view(1)]
    learner.prefetch(hv[0])                           # untimed: first use allocates the two prefetch staging slots
    for i in range(4):
        learner.prefetch(hv[(i + 1) & 1])
        train(hv[i & 1])
    train(hv[0])
    learner.prefetch(hv[0])

    def prefetched_step(i):
        if i + 1 < K:
            learner.prefetch(hv[(i + 1) & 1])
        train(hv[i & 1])

    ms_e2e_host, _ = tm.run(K, prefetched_step)
    clocks = sampler.stop() if rank == 0 else None
    launches = learner.launches_per_step + 1          # + the ingest launch (host-batch path; device batches in the
                                                      # working-set layout are read in place: no ingest launch)

    # ---- multi-GPU only: correctness of the exchange, strong scaling, config 5 sharded ------------------------------------
    dp, strong = None, None
    if world > 1:
        dp = dp_check(torch, dist, world, rank, lambda shape, seed: make_learner(shape, seed=seed))
        # strong scaling: the GLOBAL batch stays at 32 episodes (B/world per GPU); latency-bound by design (SURVEY 8(e))
        if B % world == 0:
            ls = make_learner(SHAPE)
            ls.enable_data_parallel()
            gb = [to_device_batch(torch, synthetic_batch(77 + i, **SHAPE), SHAPE["T"]) for i in range(2)]
            for i in range(6):
                ls.train(dict(gb[i % 2]), i)
            ms_s, ms_s_med = tm.run(K, lambda i: ls.train(dict(gb[i % 2]), 6 + i))
            strong = {"global_batch": B, "episodes_per_gpu": B // world, "ms_per_step": ms_s, "ms_per_step_median": ms_s_med,
                      "value": B / (ms_s * 1e-3), "unit": "episode-samples/s",
                      "limiter": "the 2L = 240 dependent GRU steps do not shrink with the shard, the exchange (flag barrier "
                                 "inside the optimiser launch) is added: latency-bound, as SURVEY.md 8(e) expects"}
            del ls, gb

    # ---- BASELINE config 5: 4096 matrix-game envs (sharded over the ranks) feeding the data-parallel QMIX learner ----------
    n5 = 4096 // world
    a5 = default_args(alg="qmix", n_agents=2, n_actions=3, obs_shape=1, state_shape=1, episode_limit=1, map="matrix")
    torch.manual_seed(0)
    l5 = QLearner(SharedMAC(a5), a5)
    if world > 1:
        l5.enable_data_parallel()
        l5._shard = lambda B_glob: (0, B_glob)
    env5 = BatchedMatrixGame(PAYOFF1, n5)
    acts5 = torch.randint(0, 3, (n5, 2), device="cuda")

    def cfg5_step(i):
        ep = dict(env5.step(acts5))
        ep["max_episode_len"] = 1
        l5.train(ep, i)

    for i in range(6):
        cfg5_step(i)
    ms5, ms5_med = tm.run(K, lambda i: cfg5_step(6 + i))
    cfg5 = {"workload": "4096 matrix-game envs sharded over the ranks (one env launch per rank) -> QMIX train step on the "
                        "emitted device batch, gradients exchanged like config 2",
            "envs_per_gpu": n5, "ms_per_iteration": ms5, "ms_per_iteration_median": ms5_med,
            "env_steps_per_s": 4096 / (ms5 * 1e-3), "episode_samples_per_s": 4096 / (ms5 * 1e-3), "scaling": "strong",
            "limiter": "launch latency: 4096 one-step episodes are ~0.25 ms of fixed-size kernels on ONE GPU already"}
    del l5, env5

    # ---- per-kernel device time (eager pass, CUDA events around every launch of the library) ---------
    learner._use_graph = False
    L.profile(rank == 0)
    P = 10
    for i in range(P):
        L.call("marl_spin_us", 4000, L.stream_ptr())      # let the host run ahead: events then bracket device time only
        train(dev_batches[i % NB])
    prof = L.profile_collect() if rank == 0 else {}
    L.profile(False)
    learner._use_graph = True
    env_small = bench_env(torch, dist, world, 4096, 200, hbm_peak)
    env_big = bench_env(torch, dist, world, 1 << 24, 20, hbm_peak)
    outputs = None
    if opt.dump_outputs:
        # The last timed step once more, through the same captured graph of the default path, from the learner's seeded state.
        # The timed loop's own state differs from run to run: its weight gradients meet in fp32 atomics, and the training steps
        # grow those last-bit differences.  From the seeded state the step's inputs are identical every run.  (Untimed, after
        # every measurement: the numbers above are those of a run without --dump-outputs.)
        for t, s0 in zip(learner_state(learner), seeded):
            t.copy_(s0)
        loss = learner.train(last[0], last[1])
        outputs = snapshot_outputs(torch, learner, loss) if rank == 0 else None
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    tot_ms = sum(ms for _, ms in prof.values()) or 1.0
    kernels = {k: {"launches_per_step": c / P, "us_per_step": ms * 1e3 / P, "share": ms / tot_ms}
               for k, (c, ms) in sorted(prof.items(), key=lambda kv: -kv[1][1])}
    # FP32 FMA peak of this GPU (probe kernel), the compute-roofline denominator
    scratch = torch.zeros(4, device="cuda")
    import ctypes as C
    flops = C.c_double()
    for _ in range(2):
        L.call("marl_fma_probe", scratch.data_ptr(), 1 << 14, 148 * 8, C.byref(flops), L.stream_ptr())
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    L.call("marl_fma_probe", scratch.data_ptr(), 1 << 14, 148 * 8, C.byref(flops), L.stream_ptr())
    b.record()
    torch.cuda.synchronize()
    fp32_peak = flops.value / (a.elapsed_time(b) * 1e-3) / 1e12

    peaks_json = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else {}
    bf16_peak = peaks_json.get("bf16_tflops_sustained", 1400.0)      # kernels timed inside a long step: the sustained figure
    # ---- larger batches of the same shape (device-resident): where the step leaves the latency-bound regime ----
    sweep = None
    if world == 1 and not opt.no_sweep:
        sweep = []
        for Bs in (256, 1024):
            db = to_device_batch(torch, synthetic_batch(7, **dict(SHAPE, B=Bs)), SHAPE["T"])
            for i in range(4):
                train(db)
            torch.cuda.synchronize()
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_.record()
            for i in range(10):
                train(db)
            b_.record(); torch.cuda.synchronize()
            msb = a_.elapsed_time(b_) / 10
            tf = FLOP_PER_STEP * Bs / SHAPE["B"] / (msb * 1e-3) / 1e12
            sweep.append({"batch": Bs, "ms_per_step": msb, "episode_samples_per_s": Bs / (msb * 1e-3), "fp32_tflops": tf,
                          "frac_of_fp32_peak": tf / fp32_peak,
                          "hbm_frac": BYTES_PER_STEP * Bs / SHAPE["B"] / (msb * 1e-3) / 1e9 / hbm_peak})
            del db
        learner._ws = {k: v for k, v in learner._ws.items() if k[0] == "stage" or k == (B, SHAPE["T"])}
        torch.cuda.empty_cache()

    # ---- the other BASELINE configs (device batch, graph replay) with the reference's CPU path beside them ----------------
    configs = None
    if world == 1 and not opt.no_sweep:
        configs = {}
        for name, flop in (("2s3z:vdn", 6.03e9), ("3s5z", 157.9e9), ("27m_vs_30m", 107.7e9)):
            cname, _, alg_o = name.partition(":")
            c = dict(CONFIGS[cname])
            alg = alg_o or c["alg"]
            shape = {k: c[k] for k in ("B", "T", "N", "A", "O", "S")}
            lc = make_learner(shape, alg=alg, name=cname)
            db = to_device_batch(torch, synthetic_batch(0, **shape), shape["T"])
            for i in range(4):
                lc.train(db, i)
            torch.cuda.synchronize()
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_.record()
            for i in range(10):
                lc.train(db, 4 + i)
            b_.record(); torch.cuda.synchronize()
            msc = a_.elapsed_time(b_) / 10
            tf = flop / (msc * 1e-3) / 1e12
            entry = {"alg": alg, "shape": shape, "ms_per_step": msc, "episode_samples_per_s": shape["B"] / (msc * 1e-3),
                     "algorithmic_gflop_per_step": flop / 1e9, "fp32_tflops": tf, "frac_of_fp32_peak": tf / fp32_peak,
                     "launches_per_step": lc.launches_per_step}
            del lc, db
            torch.cuda.empty_cache()
            try:
                r = time_reference(2, 1, alg=alg, shape=shape)
                entry["cpu_baseline"] = {"value": r["value"], "unit": r["unit"], "ms_per_step": r["ms_per_step"], "cores": r["cores"],
                                         "kind": r["kind"], "sample": "2 train steps after 1 warm-up, same batch"}
            except Exception as e:      # noqa: BLE001
                entry["cpu_baseline"] = {"unavailable": repr(e)[:200]}
            configs[cname + ("_" + alg if alg_o else "")] = entry

    roofline = None
    if kernels:
        # dominant kernel = the longest single launch of the step (it sits on the critical path): the recurrent part of
        # the three agent unrolls.  Neither HBM nor the tensor pipe binds it: it is a dependent chain of 2L small
        # (rows x 64 x 192) fp32 mat-vecs, so it is reported against the measured FP32-FMA peak, with the HBM and
        # tensor-pipe fractions beside it for context.
        dom = max(kernels, key=lambda k: kernels[k]["us_per_step"] / max(kernels[k]["launches_per_step"], 1))
        dom_us = kernels[dom]["us_per_step"] / max(kernels[dom]["launches_per_step"], 1)
        is_gru = dom == "gru_unroll_fwd_kernel"
        flop = GRU_FWD_FLOP if is_gru else FLOP_PER_STEP * kernels[dom]["share"]
        ach = flop / (dom_us * 1e-6) / 1e12
        gru_bytes = GRU_FWD_BYTES if is_gru else None
        roofline = {"kernel": dom, "bound": "fp32",
                    "bound_note": "dependent chain of 2L = 240 GRU steps on B*N = 160 rows (~1.1 rows per SM): latency-bound at "
                                  "B=32; FP32 FMA is the nearest roof (HBM and tensor-pipe fractions given for context; see "
                                  "batch_sweep for the fraction at larger batches)",
                    "achieved": ach, "peak": fp32_peak, "unit": "TFLOP/s", "frac": ach / fp32_peak,
                    "traffic": NCU_TRAFFIC.get(dom), "traffic_source": "profiles/r1c_ncu_full_gru.txt (dram_read + dram_write, one --set full capture)",
                    "us_per_launch": dom_us, "algorithmic_flop_per_launch": flop, "algorithmic_bytes_per_launch": gru_bytes,
                    "hbm_frac": (gru_bytes / (dom_us * 1e-6) / 1e9 / hbm_peak) if gru_bytes else None,
                    "peak_source": "fp32: marl_fma_probe on this GPU, the builder's own probe (MEASURED_PEAKS.json has no fp32 "
                                   "figure; nominal 148 SMs x 128 lanes x 2 x 1.965 GHz = 74.4); hbm: " + peak_src}
    gemm_us = sum(v["us_per_step"] for k, v in kernels.items() if k.startswith(("linear_", "tgemm_", "wgrad_reduce", "agent_front_")))
    gemm_flop = FLOP_PER_STEP - GRU_FWD_FLOP - GRU_FWD_FLOP / 3        # everything but the two recurrent kernels
    roofline_gemm = None
    if gemm_us:
        ach = gemm_flop / (gemm_us * 1e-6) / 1e12
        roofline_gemm = {"kernel": "agent_front_kernel + linear_{fwd,dgrad,wgrad}_kernel (tcgen05 kind::tf32, 3xTF32)", "bound": "tensor",
                         "achieved": ach, "peak": bf16_peak, "unit": "TFLOP/s", "frac": ach / bf16_peak,
                         "traffic": NCU_TRAFFIC.get("linear_fwd_kernel"), "us_per_step": gemm_us,
                         "note": "algorithmic fp32 FLOPs of all dense layers / summed launch time (launches on parallel streams "
                                 "overlap, so the sum overstates the wall time); peak = measured sustained bf16.  Measured "
                                 "(tools/micro/mma_rate2.cu): one tcgen05.mma kind::tf32 (K = 8, M = 128) takes max(44.5, N/2) "
                                 "cycles, i.e. 1.19 PFLOP/s at N >= 128 and 0.79 at the N = 64 of these layers, and 3xTF32 issues "
                                 "every product three times; the layers are bound by what surrounds the MMAs (operand staging, "
                                 "hand-overs, epilogues), not by the tensor pipe (DESIGN.md section 4)"}
    step_tflops = FLOP_PER_STEP / (ms_dev * 1e-3) / 1e12

    cpu, gpu_base = None, None
    if world == 1:
        r = time_reference(20, 3)
        cpu = {"value": r["value"], "unit": "episode-samples/s", "cores": r["cores"], "kind": r["kind"],
               "sample": "20 train steps (after 3 warm-up) of the same B=32 2s3z-shaped batch, "
                         + ("UNMODIFIED reference QLearner.train (oracle/_ref)" if r["kind"] == "reference" else
                            "oracle port of the reference CPU path (oracle/_ref not staged)") + ", all host threads",
               "ms_per_step": r["ms_per_step"]}
        try:
            g = time_reference(10, 3, cuda=True)
            if g is not None:
                gpu_base = {"value": g["value"], "unit": g["unit"], "ms_per_step": g["ms_per_step"], "steps": 10,
                            "what": "UNMODIFIED reference QLearner.train with args.cuda=True on this B200 (stock ATen / cuBLAS)"}
        except Exception as e:      # noqa: BLE001
            gpu_base = {"unavailable": repr(e)[:200]}

    line = {
        "metric": "QMIX learner episode-samples/sec (2s3z shape)", "value": B * world / (ms_dev * 1e-3),
        "unit": "episode-samples/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_dev,
        "ms_per_step_median": ms_dev_median, "ms_per_step_max": dev_max,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "global_batch": B * world, "parallelism": f"dp{world}",
                   "gradient_exchange": (None if world == 1 else
                                         "fused into the optimiser launch over NVLink peer memory (marl_clip_step_peer)"
                                         if getattr(learner, "_peer", None) is not None else "ncclAllReduce between two graphs"),
                   "l2": f"inputs rotate over {NB} resident batches (150 MB > 126 MB L2)"},
        "e2e": {"value": B * world / (ms_replay * 1e-3), "unit": "episode-samples/s", "ms_per_step": ms_replay,
                "ms_per_step_median": ms_replay_median, "ms_per_step_max": replay_max,
                "h2d_bytes_per_step": int(ep_bytes), "d2h_bytes_per_step": 8,
                "how": "the reference's training loop (runner.py:92-97, n_episodes = 1, train_steps = 1) through the drop-in "
                       "classes: buffer.store_episode(one new float64 HOST episode, pinned) -> buffer.sample(32) -> "
                       "learner.train(batch) -> loss as a Python float; the episode crosses PCIe inside the timed region (its "
                       "arrays are page-locked, so the float64 -> fp32 cast kernel reads them in place and store_episode returns "
                       "when it has; pageable arrays take a packed staging copy instead), and so do the gather of the sampled "
                       "rows and the loss read-back",
                "host_dict_variant": {"value": B * world / (ms_e2e_host * 1e-3), "ms_per_step": ms_e2e_host,
                                      "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 8,
                                      "how": "QLearner.train(whole float64 host batch) every step, next batch prefetched: "
                                             "PCIe-bound (35.6 MB per step)",
                                      "without_prefetch": {"value": B * world / (ms_e2e_sync * 1e-3), "ms_per_step": ms_e2e_sync}}},
        "gpu_launches": int((launches - 1) * K + (launches + 1) * K + 2 * launches * K),   # value (in place) + replay (ingest + gather) + 2 host-dict legs
        "launches_per_step": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "roofline_gemm": roofline_gemm,
        "step_fp32": {"tflops": step_tflops, "frac_of_fp32_peak": step_tflops / fp32_peak, "fp32_peak_tflops": fp32_peak,
                      "hbm_frac": BYTES_PER_STEP / (ms_dev * 1e-3) / 1e9 / hbm_peak, "hbm_peak_gbs": hbm_peak,
                      "peak_source": peak_src},
        "kernels": kernels,
        "batch_sweep": sweep,
        "configs": configs,
        "dp_check": dp,
        "strong_scaling": strong,
        "env": {"metric": "matrix-game env-steps/sec", "value": env_big["value"], "unit": "env-steps/s",
                "bytes_per_env_step": ENV_BYTES, "cfg5_4096_envs": env_small, "bandwidth_regime_2^24_envs": env_big},
        "cfg5_env_plus_learner": cfg5,
        "cpu_baseline": cpu,
        "gpu_baseline": gpu_base,
    }
    if outputs is not None:
        write_outputs(opt.dump_outputs, outputs)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def learner_state(learner):
    """What a train() step reads besides its batch and then updates: parameters, target parameters, optimiser state."""
    return [learner._flat.data, learner._tflat.data] + list(learner.optimizer.state_dict().values())


def snapshot_outputs(torch, learner, loss):
    """Device copies of what a caller of QLearner.train holds after a step: the returned loss, the clipped gradients left
    in p.grad, the state_dicts of the trained and target networks, and the hidden states left in the two controllers."""
    out = {"loss": torch.tensor([loss], dtype=torch.float64)}
    for prefix, module in (("agent", learner.eval_net.agent), ("mixer", learner.mixer)):
        for k, p in module.named_parameters():
            out[f"grad.{prefix}.{k}"] = p.grad.detach().clone()
    for prefix, module in (("agent", learner.eval_net.agent), ("mixer", learner.mixer),
                           ("target_agent", learner.target_net.agent), ("target_mixer", learner.target_mixer)):
        for k, v in module.state_dict().items():
            out[f"{prefix}.{k}"] = v.detach().clone()
    out["hidden_states"] = learner.eval_net.hidden_states.detach().clone()
    out["target_hidden_states"] = learner.target_net.hidden_states.detach().clone()
    return out


def write_outputs(path, outputs):
    """One DIR/<name>.npy per array: float64 stays float64, everything else is written as float32 (~0.6 MB in all)."""
    os.makedirs(path, exist_ok=True)
    for name, t in outputs.items():
        a = t.cpu().numpy()
        np.save(os.path.join(path, name + ".npy"), a if a.dtype == np.float64 else a.astype(np.float32))


def pin_to_gpu_numa(local):
    """Binds this rank's host threads to the cores of its GPU's NUMA node (NVML affinity) so that the pinned staging
    buffers and the copy-issuing thread sit next to the PCIe root of the GPU; a no-op when NVML cannot tell."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        n = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, n)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        world = int(os.environ.get("WORLD_SIZE", "1"))
        if cpus and world > 1:
            # spread the ranks that share a node over disjoint slices of its cores
            cpus = sorted(cpus)
            per = max(1, len(cpus) // world)
            mine = cpus[(local * per) % len(cpus):][:per] or cpus
            os.sched_setaffinity(0, set(mine))
    except Exception:       # noqa: BLE001
        pass


def positive(v):
    n = int(v)
    if n < 1:
        raise argparse.ArgumentTypeError(f"must be >= 1, got {n}")
    return n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive, default=50,
                    help="timed train() steps of the headline, end-to-end and env+learner loops (the batch sweep, the other "
                         "configs, the per-kernel profile and the baselines time fixed counts)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-sweep", dest="no_sweep", action="store_true", help="skip the B=256/1024 legs")
    ap.add_argument("--dump-outputs", dest="dump_outputs", metavar="DIR",
                    help="after the measurements, restore the learner's seeded state, run the last timed step of the "
                         "headline (device-resident batch) loop once more through the same captured graph, and write what "
                         "it leaves a caller (loss, clipped gradients, networks, hidden states) to DIR/<name>.npy: the "
                         "step's inputs are identical every run, so two runs or two builds can be compared output for "
                         "output; the timings are those of a run without this option")
    opt = ap.parse_args()
    if opt.impl == "reference":
        run_reference(opt)
    else:
        run_ours(opt)


if __name__ == "__main__":
    main()
