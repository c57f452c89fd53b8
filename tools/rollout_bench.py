"""Data-collection throughput: batched acting, the one-step matrix-game rollout and the multi-step rollout.

Prints one JSON line:
  * act: at the config-2/3/4 agent shapes (N/A/O = 5/11/80, 8/14/128, 27/36/285) and n instances, the single
    marl_agent_act launch against the sequence it replaces (mac.agent.unroll with T = 1, then marl_epsgreedy_select),
    timed alternately in the same run with CUDA events; agent-rows/s, achieved FP32 FLOP/s and its share of the FMA
    rate marl_fma_probe measures in the same run; the two sequences' outputs are compared (q and h' within 1e-5,
    actions equal except where the top-2 gap is below 1e-5) and a disagreement fails the run;
  * matrix: BatchedRolloutWorker.generate_episodes on BatchedMatrixGame (device RNG), env-steps/s including acting;
  * multistep: generate_episodes on the ragged test game of tests/envs.py, us per environment step (wall clock
    around whole calls that end in a synchronisation) and library launches per step (L.profile, separate run);
  * separated: one network per agent (SeparatedMAC, reuse_network=False) at the same agent shapes:
    - act: SeparatedMAC.act (one marl_agent_act_separated launch) against SharedMAC.act (one marl_agent_act launch) at
      the same shape and n (same FLOPs: the agent-id block is one gathered column).  us_act_*: CUDA events around a loop
      of calls, timed alternately, which includes the host's enqueue cost when that is longer than the kernel (the
      separated call rebuilds its table of N parameter sets each time); us_kernel_*: the launches alone (L.profile,
      separate pass), where the difference is the per-agent weight restaging; FLOP/s from the kernel time.  Its q, h'
      and actions are checked against each agent's own unroll;
    - choose_action: one environment step of ONE instance acted as the reference does, SeparatedMAC.choose_action
      looped over the agents (N batch-1 forwards and an int() each), wall clock, against one act launch for that instance;
    - matrix: generate_episodes on BatchedMatrixGame with a SeparatedMAC, env-steps/s including acting.
The GPU name and power limit are read through NVML (queries only) in the same run.
usage: python tools/rollout_bench.py [--quick] [--out FILE]
"""
import ctypes as C
import json
import os
import sys
import time

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

import numpy as np
import torch

from marl_b200 import _lib as L
from marl_b200.common.arguments import default_args
from marl_b200.controller.share_params import SeparatedMAC, SharedMAC
from marl_b200.env.single_state_matrix_game import BatchedMatrixGame
from marl_b200.rollout import BatchedRolloutWorker
from tests.envs import CountdownGameBatched

H = 64
SHAPES = {"cfg2": (5, 11, 80), "cfg3": (8, 14, 128), "cfg4": (27, 36, 285)}


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())
        info["power_limit_w"] = pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
        info["sm_max_mhz"] = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
    except Exception as e:                                  # report, do not guess
        info["nvml_error"] = repr(e)
    return info


def fma_peak():
    """FP32 FLOP/s of marl_fma_probe (8 independent FMA chains per thread, 8 blocks of 256 per SM)."""
    scratch = torch.zeros(1, device="cuda")
    blocks = torch.cuda.get_device_properties(0).multi_processor_count * 8
    flops = C.c_double()
    L.call("marl_fma_probe", scratch.data_ptr(), 1 << 14, blocks, C.byref(flops), L.stream_ptr())
    torch.cuda.synchronize()
    best = 0.0
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        L.call("marl_fma_probe", scratch.data_ptr(), 1 << 14, blocks, C.byref(flops), L.stream_ptr())
        e1.record()
        e1.synchronize()
        best = max(best, flops.value / (e0.elapsed_time(e1) * 1e-3))
    return best


def timed(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / iters               # us per call


def act_ab(name, n, peak, reps):
    N, A, O = SHAPES[name]
    args = default_args(alg="qmix", n_agents=N, n_actions=A, obs_shape=O, state_shape=4, episode_limit=1)
    torch.manual_seed(0)
    mac = SharedMAC(args)
    g = torch.Generator(device="cuda").manual_seed(n + N)
    obs = torch.randn(n, N, O, device="cuda", generator=g)
    last = torch.nn.functional.one_hot(torch.randint(0, A, (n, N), device="cuda", generator=g), A).float()
    avail = (torch.rand(n, N, A, device="cuda", generator=g) < 0.7).float()
    h0 = torch.randn(n * N, H, device="cuda", generator=g) * 0.5
    rows = n * N
    q_new = torch.empty(n, N, A, device="cuda")
    h_new = h0.clone()
    act_new = torch.empty(n, N, dtype=torch.int64, device="cuda")
    act_old = torch.empty(n * N, dtype=torch.int64, device="cuda")
    onehot_new = torch.empty(n, N, A, device="cuda")
    onehot_old = torch.empty(n * N, A, device="cuda")

    def new(h=h_new):
        mac.act(n, obs, last, avail, h, actions=act_new, onehot=onehot_new, q=q_new)

    def old(h=h0):
        q, _, h1 = mac.agent.unroll(obs.unsqueeze(1), last.unsqueeze(1), h, 0)
        L.call("marl_epsgreedy_select", rows, A, q.data_ptr(), avail.data_ptr(), None, None, act_old.data_ptr(),
               onehot_old.data_ptr(), L.stream_ptr())
        return q, h1

    with torch.no_grad():
        # outputs first, from the same hidden state
        q_old, h_old = old()
        new()
        torch.cuda.synchronize()
        q_err = float((q_new.view(rows, A) - q_old.view(rows, A)).abs().max() / q_old.abs().max())
        h_err = float((h_new - h_old).abs().max() / h_old.abs().max())
        qm = torch.where(avail.view(rows, A) == 0, torch.full_like(q_old.view(rows, A), -float("inf")), q_old.view(rows, A))
        diff = (act_new.view(-1) != act_old).nonzero().view(-1)
        hard = 0
        if diff.numel():
            top = qm[diff].gather(1, act_old[diff].view(-1, 1)).view(-1)
            mine = qm[diff].gather(1, act_new.view(-1)[diff].view(-1, 1)).view(-1)
            hard = int(((top - mine).abs() > 1e-5 * top.abs().clamp(min=1.0)).sum())
        ok = q_err < 1e-5 and h_err < 1e-5 and hard == 0
        iters = max(3, min(200, int(2e6 // rows)))
        for _ in range(3):
            new(); old()
        t_new, t_old = [], []
        for _ in range(reps):                              # alternate the two in the same run
            t_new.append(timed(new, iters))
            t_old.append(timed(old, iters))
    us_new, us_old = float(np.median(t_new)), float(np.median(t_old))
    flop_row = 2 * H * (O + A + 1) + 2 * 2 * 3 * H * H + 2 * A * H
    return {"cfg": name, "n": n, "rows": rows, "us_act": round(us_new, 2), "us_unroll_select": round(us_old, 2),
            "speedup": round(us_old / us_new, 3), "rows_per_s": rows / us_new * 1e6,
            "tflops": rows * flop_row / us_new * 1e-6, "share_of_fma_peak": rows * flop_row / (us_new * 1e-6) / peak,
            "q_rel_err": q_err, "h_rel_err": h_err, "action_mismatches": int(diff.numel()), "action_hard_mismatches": hard,
            "outputs_agree": ok}


def matrix(n, calls, separated=False):
    args = default_args(alg="qmix", n_agents=2, n_actions=3, obs_shape=1, state_shape=1, episode_limit=1)
    args.epsilon, args.anneal_epsilon = 0.5, 0.0
    args.reuse_network = not separated
    torch.manual_seed(0)
    mac = SeparatedMAC(args) if separated else SharedMAC(args)
    w = BatchedRolloutWorker(BatchedMatrixGame([[8, -12, -12], [-12, 0, 0], [-12, 0, 0]], n), mac, args)
    for _ in range(3):
        w.generate_episodes(rng="device")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(calls):
        w.generate_episodes(rng="device")
    torch.cuda.synchronize()
    us = (time.perf_counter() - t0) / calls * 1e6
    return {"n_envs": n, "us_per_call": round(us, 2), "env_steps_per_s": n / us * 1e6}


def multistep(n, calls):
    N, A, O, S, T = 3, 5, 4, 3, 6
    args = default_args(alg="qmix", n_agents=N, n_actions=A, obs_shape=O, state_shape=S, episode_limit=T)
    args.epsilon, args.anneal_epsilon, args.epsilon_anneal_scale = 0.5, 0.0, "step"
    torch.manual_seed(0)
    env = CountdownGameBatched(n, n_agents=N, n_actions=A, episode_limit=T)
    w = BatchedRolloutWorker(env, SharedMAC(args), args)
    n_steps = []
    step = env.step
    env.step = lambda a, act: n_steps.append(1) or step(a, act)
    for _ in range(3):
        w.generate_episodes()
    torch.cuda.synchronize()
    n_steps.clear()
    t0 = time.perf_counter()
    for _ in range(calls):
        w.generate_episodes()                              # ends in its own synchronisation (the step count)
    us = (time.perf_counter() - t0) * 1e6
    k = len(n_steps)
    torch.cuda.synchronize()
    L.profile(True)
    try:
        L.profile_collect()
        n_steps.clear()
        w.generate_episodes()
        launches = L.profile_collect()
    finally:
        L.profile(False)
    per_step = {name: c / len(n_steps) for name, (c, _) in launches.items()}
    return {"n_envs": n, "episode_limit": T, "env_steps_per_call": k / calls, "us_per_env_step": round(us / k, 2),
            "library_launches_per_env_step": round(sum(per_step.values()), 3),
            "launches_per_env_step": per_step}


def act_separated(name, n, peak, reps):
    N, A, O = SHAPES[name]
    args = default_args(alg="qmix", n_agents=N, n_actions=A, obs_shape=O, state_shape=4, episode_limit=1)
    torch.manual_seed(0)
    shared = SharedMAC(args)
    args_sep = default_args(alg="qmix", n_agents=N, n_actions=A, obs_shape=O, state_shape=4, episode_limit=1)
    args_sep.reuse_network = False
    sep = SeparatedMAC(args_sep)
    g = torch.Generator(device="cuda").manual_seed(n + N)
    obs = torch.randn(n, N, O, device="cuda", generator=g)
    last = torch.nn.functional.one_hot(torch.randint(0, A, (n, N), device="cuda", generator=g), A).float()
    avail = (torch.rand(n, N, A, device="cuda", generator=g) < 0.7).float()
    h0 = torch.randn(n * N, H, device="cuda", generator=g) * 0.5
    rows = n * N
    q_sep, q_sh = torch.empty(n, N, A, device="cuda"), torch.empty(n, N, A, device="cuda")
    h_sep, h_sh = h0.clone(), h0.clone()
    a_sep, a_sh = torch.empty(n, N, dtype=torch.int64, device="cuda"), torch.empty(n, N, dtype=torch.int64, device="cuda")
    oh_sep, oh_sh = torch.empty(n, N, A, device="cuda"), torch.empty(n, N, A, device="cuda")

    def run_sep():
        sep.act(n, obs, last, avail, h_sep, actions=a_sep, onehot=oh_sep, q=q_sep)

    def run_shared():
        shared.act(n, obs, last, avail, h_sh, actions=a_sh, onehot=oh_sh, q=q_sh)

    with torch.no_grad():
        run_sep()
        x = torch.cat([obs, last], -1)                     # agent i's own [obs | last action] input, its own unroll
        outs = [net.unroll_full(x[:, i].reshape(n, 1, 1, -1).contiguous(), h0.view(n, N, H)[:, i].contiguous())
                for i, net in enumerate(sep.agent)]
        q_ref = torch.stack([o[0].view(n, A) for o in outs], 1)
        h_ref = torch.stack([o[2].view(n, H) for o in outs], 1)
        torch.cuda.synchronize()
        q_err = float((q_sep - q_ref).abs().max() / q_ref.abs().max())
        h_err = float((h_sep.view(n, N, H) - h_ref).abs().max() / h_ref.abs().max())
        qm = torch.where(avail == 0, torch.full_like(q_ref, -float("inf")), q_ref).view(rows, A)
        mine = qm.gather(1, a_sep.view(rows, 1)).view(-1)
        top = qm.max(1).values
        hard = int(((top - mine).abs() > 1e-5 * top.abs().clamp(min=1.0)).sum())
        ok = q_err < 1e-5 and h_err < 1e-5 and hard == 0
        iters = max(3, min(200, int(2e6 // rows)))
        for _ in range(3):
            run_sep(); run_shared()
        t_sep, t_sh = [], []
        for _ in range(reps):                              # alternate the two in the same run
            t_sep.append(timed(run_sep, iters))
            t_sh.append(timed(run_shared, iters))
        torch.cuda.synchronize()
        L.profile(True)                                    # device time of each launch alone (events around it)
        try:
            L.profile_collect()
            for _ in range(iters):
                run_sep(); run_shared()
            torch.cuda.synchronize()
            prof = L.profile_collect()
        finally:
            L.profile(False)
    us_sep, us_sh = float(np.median(t_sep)), float(np.median(t_sh))
    k_sep, k_sh = (prof[k][1] * 1e3 / prof[k][0] for k in ("agent_act_separated_kernel", "agent_act_kernel"))
    flop_row = 2 * H * (O + A) + 2 * 2 * 3 * H * H + 2 * A * H
    return {"cfg": name, "n": n, "rows": rows, "us_act_separated": round(us_sep, 2), "us_act_shared": round(us_sh, 2),
            "separated_over_shared": round(us_sep / us_sh, 3), "us_kernel_separated": round(k_sep, 2),
            "us_kernel_shared": round(k_sh, 2), "kernel_separated_over_shared": round(k_sep / k_sh, 3),
            "rows_per_s": rows / us_sep * 1e6, "tflops": rows * flop_row / k_sep * 1e-6,
            "share_of_fma_peak": rows * flop_row / (k_sep * 1e-6) / peak,
            "q_rel_err": q_err, "h_rel_err": h_err, "action_hard_mismatches": hard, "outputs_agree": ok}


def choose_action_loop(name, steps):
    """One instance, one environment step: SeparatedMAC.choose_action per agent (the reference's acting) against one
    marl_agent_act_separated launch; wall clock per step, each ending in a synchronisation."""
    N, A, O = SHAPES[name]
    args = default_args(alg="qmix", n_agents=N, n_actions=A, obs_shape=O, state_shape=4, episode_limit=1)
    args.reuse_network = False
    torch.manual_seed(0)
    mac = SeparatedMAC(args)
    rng = np.random.RandomState(N)
    obs, avail = rng.randn(N, O), np.ones((N, A))
    last = np.zeros((N, A))
    obs_d, last_d, avail_d = (torch.as_tensor(x[None], dtype=torch.float32, device="cuda") for x in (obs, last, avail))
    res = {"cfg": name, "n": 1}
    with torch.no_grad():
        for key, step in (("us_per_step_choose_action_loop",
                           lambda: [int(mac.choose_action(obs[a], last[a], a, avail[a], 0.0)) for a in range(N)]),
                          ("us_per_step_act", lambda: mac.choose_actions(obs_d, last_d, avail_d, 0.0, evaluate=True).cpu())):
            mac.init_hidden(1)
            for _ in range(3):
                step()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                step()
            torch.cuda.synchronize()
            res[key] = round((time.perf_counter() - t0) / steps * 1e6, 2)
    res["speedup"] = round(res["us_per_step_choose_action_loop"] / res["us_per_step_act"], 2)
    return res


def main():
    quick = "--quick" in sys.argv
    out = sys.argv[sys.argv.index("--out") + 1] if "--out" in sys.argv else None
    torch.cuda.init()
    L.ensure_scratch()
    res = {"metric": "rollout_bench", "gpu": gpu_info()}
    peak = fma_peak()
    res["fma_peak_tflops"] = peak * 1e-12
    sizes = (256, 4096) if quick else (256, 4096, 65536)
    res["act"] = [act_ab(c, n, peak, 2 if quick else 7) for c in SHAPES for n in sizes]
    res["matrix"] = [matrix(n, 5 if quick else 30) for n in ((4096,) if quick else (4096, 1 << 20))]
    res["multistep"] = multistep(4096, 3 if quick else 20)
    res["separated"] = {
        "act": [act_separated(c, n, peak, 2 if quick else 7) for c in SHAPES for n in sizes],
        "choose_action": [choose_action_loop(c, 5 if quick else 30) for c in SHAPES],
        "matrix": [matrix(n, 5 if quick else 30, separated=True) for n in ((4096,) if quick else (4096, 1 << 20))]}
    res["outputs_agree"] = all(r["outputs_agree"] for r in res["act"] + res["separated"]["act"])
    line = json.dumps(res)
    print(line)
    if out:
        with open(out, "w") as f:
            f.write(line + "\n")
    if not res["outputs_agree"]:
        sys.exit("an act launch disagrees with the unroll it replaces")


if __name__ == "__main__":
    main()
