"""QMIX at qmix_hidden_dim != 32 on the device: every marl_qmix_* entry point against fp64 autograd of the oracle's mixer,
the embed field of the C ABI, the fused learner step against the fp64 oracle and on its other routes (modules, graphs,
replay batches, SeparatedMAC, last_action, the TMA GEMM back end, launch plan), checkpoints, the matrix-game tables and
data parallelism."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from marl_b200 import _lib as L
from marl_b200.network.mixer import hy_cols
from marl_b200.synthetic import synthetic_batch
from oracle import marl_oracle as MO
from tests import parity_util as PU

pytestmark = pytest.mark.gpu
TOL = 1e-5
HEADS = ("hyper_w1", "hyper_b1", "hyper_w2", "hyper_b2.0")
CFG2 = (5, 11, 80, 120, 120, 32)        # N, A, O, S, T, B (2s3z-like shape of bench.py's headline)
TINY = (3, 4, 5, 6, 8, 4)


def _rel(x, y):
    return PU.rel_err(x, y)


# ------------------------------------------------------------------------------------------ library calls
def _mixer_params(E, N, S, seed, dtype=torch.float64):
    cfg = MO.make_cfg(n_agents=N, n_actions=1, state_shape=S, qmix_hidden_dim=E)
    torch.manual_seed(seed)
    sd = MO.init_mixer(cfg, "qmix")
    return cfg, {k: v.to(dtype) for k, v in sd.items()}


def _device_flat(sd, N, E, S):
    """wcat / bcat laid out as the C ABI reads them, plus hyper_b2.2; fp32 on the device."""
    wcat = torch.cat([sd[h + ".weight"] for h in HEADS]).float().cuda().contiguous()
    bcat = torch.cat([sd[h + ".bias"] for h in HEADS]).float().cuda().contiguous()
    wb2 = sd["hyper_b2.2.weight"].reshape(-1).float().cuda().contiguous()
    bb2 = sd["hyper_b2.2.bias"].float().cuda().contiguous()
    assert wcat.shape == (hy_cols(N, E), S)
    return wcat, bcat, wb2, bb2


def _params(t, E):
    return L.QmixParams(t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(), t[3].data_ptr(), E)


def _grads(E, N, S, dev="cuda"):
    Cc = hy_cols(N, E)
    g = [torch.zeros(Cc, S, device=dev), torch.zeros(Cc, device=dev), torch.zeros(E, device=dev), torch.zeros(1, device=dev)]
    return g, L.QmixGrads(*(x.data_ptr() for x in g), E)


def _oracle_grads(sd, loss):
    keys = [h + ".weight" for h in HEADS]
    bkeys = [h + ".bias" for h in HEADS]
    gr = torch.autograd.grad(loss, [sd[k] for k in keys + bkeys + ["hyper_b2.2.weight", "hyper_b2.2.bias"]])
    n = len(keys)
    return torch.cat(gr[:n]), torch.cat(gr[n:2 * n]), gr[-2].reshape(-1), gr[-1]


EMBEDS = [1, 7, 16, 33, 64, 128]
AGENTS = [2, 5, 27]


@pytest.mark.parametrize("E", EMBEDS)
@pytest.mark.parametrize("N", AGENTS)
def test_qmix_fwd_bwd_and_hyper_calls(E, N):
    """marl_qmix_fwd / _bwd, and the split form marl_qmix_hyper_fwd + marl_qmix_mix_fwd / _mix_bwd +
    marl_qmix_hyper_wgrad, against fp64 autograd of the oracle's mixer."""
    S, M = 9, 300
    cfg, sd = _mixer_params(E, N, S, seed=E * 100 + N)
    sd = {k: v.requires_grad_(True) for k, v in sd.items()}
    torch.manual_seed(1)
    q64, s64, w64 = torch.randn(M, N, dtype=torch.float64), torch.randn(M, S, dtype=torch.float64), torch.randn(M, dtype=torch.float64)
    q64.requires_grad_(True)
    out64 = MO.qmix_mix(sd, q64.view(M, 1, N), s64.view(M, 1, S), cfg).reshape(-1)
    loss = (out64 * w64).sum()
    want_dq = torch.autograd.grad(loss, q64, retain_graph=True)[0]
    want_g = _oracle_grads(sd, loss)

    t = _device_flat(sd, N, E, S)
    p = _params(t, E)
    q, s, w = q64.detach().float().cuda(), s64.float().cuda(), w64.float().cuda()
    Cc = hy_cols(N, E)
    for split in (False, True):
        hy, dhy = torch.empty(M, Cc, device="cuda"), torch.empty(M, Cc, device="cuda")
        q_tot, dq = torch.empty(M, device="cuda"), torch.empty(M, N, device="cuda")
        g, gs = _grads(E, N, S)
        sp = L.stream_ptr()
        if split:
            L.call("marl_qmix_hyper_fwd", M, N, S, C.byref(p), s.data_ptr(), hy.data_ptr(), sp)
            L.call("marl_qmix_mix_fwd", M, N, C.byref(p), q.data_ptr(), hy.data_ptr(), q_tot.data_ptr(), sp)
            L.call("marl_qmix_mix_bwd", M, N, C.byref(p), q.data_ptr(), hy.data_ptr(), w.data_ptr(), dhy.data_ptr(),
                   dq.data_ptr(), C.byref(gs), sp)
            L.call("marl_qmix_hyper_wgrad", M, N, S, s.data_ptr(), dhy.data_ptr(), C.byref(gs), sp)
        else:
            L.call("marl_qmix_fwd", M, N, S, C.byref(p), q.data_ptr(), s.data_ptr(), hy.data_ptr(), q_tot.data_ptr(), sp)
            L.call("marl_qmix_bwd", M, N, S, C.byref(p), q.data_ptr(), s.data_ptr(), hy.data_ptr(), w.data_ptr(),
                   dhy.data_ptr(), dq.data_ptr(), C.byref(gs), sp)
        torch.cuda.synchronize()
        assert _rel(q_tot, out64.detach()) < TOL, split
        assert _rel(dq, want_dq) < TOL, split
        for name, mine, ref in zip(("wcat", "bcat", "wb2", "bb2"), g, want_g):
            assert _rel(mine, ref) < TOL, (split, name)


def _td_reference(sd, sd_t, q, qt, s, s2, r, term, pad, gamma, cfg):
    M, N = q.shape
    S = s.shape[1]
    q = q.clone().requires_grad_(True)
    tot = MO.qmix_mix(sd, q.view(M, 1, N), s.view(M, 1, S), cfg).reshape(-1)
    with torch.no_grad():
        tot_t = MO.qmix_mix(sd_t, qt.view(M, 1, N), s2.view(M, 1, S), cfg).reshape(-1)
    mask = 1 - pad
    d = mask * (r + gamma * tot_t * (1 - term) - tot)
    loss = (d ** 2).sum()
    dq = torch.autograd.grad(loss, q, retain_graph=True)[0]
    return tot.detach(), tot_t, loss.detach(), mask.sum(), dq, _oracle_grads(sd, loss)


@pytest.mark.parametrize("E", EMBEDS)
@pytest.mark.parametrize("N", AGENTS)
@pytest.mark.parametrize("flags", [0, 3])
def test_qmix_td_fwd_bwd(E, N, flags):
    """The learner's fused TD call (eval + target mixer, TD loss, gradients, dense dq), with its own hyper GEMMs (flags 0)
    or after marl_qmix_hyper_fwd and before marl_qmix_hyper_wgrad (flags 3)."""
    S, B, Lq, A = 9, 6, 25, 4
    M = B * Lq
    cfg, sd = _mixer_params(E, N, S, seed=E + N)
    _, sd_t = _mixer_params(E, N, S, seed=E + N + 7)
    sd = {k: v.requires_grad_(True) for k, v in sd.items()}
    g = torch.Generator().manual_seed(2)
    q64, qt64 = torch.randn(M, N, generator=g, dtype=torch.float64), torch.randn(M, N, generator=g, dtype=torch.float64)
    s64, s264 = torch.randn(M, S, generator=g, dtype=torch.float64), torch.randn(M, S, generator=g, dtype=torch.float64)
    r64 = torch.randn(M, generator=g, dtype=torch.float64)
    term64 = (torch.rand(M, generator=g) < 0.1).double()
    pad64 = (torch.rand(M, generator=g) < 0.2).double()
    u = torch.randint(0, A, (M, N), generator=g)
    tot, tot_t, loss, msum, dq_ref, want_g = _td_reference(sd, sd_t, q64, qt64, s64, s264, r64, term64, pad64, 0.99, cfg)

    te, tt = _device_flat(sd, N, E, S), _device_flat(sd_t, N, E, S)
    p, pt = _params(te, E), _params(tt, E)
    f = lambda x: x.float().cuda().contiguous()
    q, qt, s, s2, r, term, pad, ud = f(q64), f(qt64), f(s64), f(s264), f(r64), f(term64), f(pad64), u.cuda()
    Cc = hy_cols(N, E)
    hy, hy_t, dhy = (torch.empty(M, Cc, device="cuda") for _ in range(3))
    q_tot, q_tot_t, dq, scalars = torch.empty(M, device="cuda"), torch.empty(M, device="cuda"), \
        torch.empty(M, N, A, device="cuda"), torch.zeros(2, device="cuda")
    gt, gs = _grads(E, N, S)
    d = L.Dims(B, Lq, N, A, 1, S)
    sp = L.stream_ptr()
    if flags:
        L.call("marl_qmix_hyper_fwd", M, N, S, C.byref(p), s.data_ptr(), hy.data_ptr(), sp)
        L.call("marl_qmix_hyper_fwd", M, N, S, C.byref(pt), s2.data_ptr(), hy_t.data_ptr(), sp)
    L.call("marl_qmix_td_fwd_bwd", C.byref(d), C.byref(p), C.byref(pt), s.data_ptr(), s2.data_ptr(), q.data_ptr(),
           qt.data_ptr(), ud.data_ptr(), r.data_ptr(), term.data_ptr(), pad.data_ptr(), 0.99, hy.data_ptr(),
           hy_t.data_ptr(), dhy.data_ptr(), q_tot.data_ptr(), q_tot_t.data_ptr(), dq.data_ptr(), C.byref(gs),
           scalars.data_ptr(), flags, None, None, None, sp)
    if flags:
        L.call("marl_qmix_hyper_wgrad", M, N, S, s.data_ptr(), dhy.data_ptr(), C.byref(gs), sp)
    torch.cuda.synchronize()
    assert _rel(q_tot, tot) < TOL and _rel(q_tot_t, tot_t) < TOL
    assert abs(float(scalars[0]) - float(loss)) <= TOL * float(loss)
    assert float(scalars[1]) == float(msum)
    dense = torch.zeros(M, N, A, dtype=torch.float64).scatter_(2, u.unsqueeze(2), dq_ref.unsqueeze(2))
    assert _rel(dq, dense) < TOL
    for name, mine, ref in zip(("wcat", "bcat", "wb2", "bb2"), gt, want_g):
        assert _rel(mine, ref) < TOL, name


@pytest.mark.parametrize("E", EMBEDS)
@pytest.mark.parametrize("N", AGENTS)
def test_qmix_hyper2_calls(E, N):
    """two_hyper_layers: marl_qmix_hyper2_fwd / _bwd around marl_qmix_mix_fwd / _bwd through QMixMixer.forward."""
    from marl_b200.network.mixer import QMixMixer
    S, hh, M = 9, 16, 200
    args = PU.make_args("qmix", N, 3, 4, S, 10, qmix_hidden_dim=E, two_hyper_layers=True, hyper_hidden_dim=hh)
    torch.manual_seed(E * 3 + N)
    mixer = QMixMixer(args)
    sd = {k: v.detach().cpu().double().requires_grad_(True) for k, v in mixer.state_dict().items()}
    # (positive weights: hyper_b2.2.bias's gradient is their sum, which a signed draw would make a cancelling one)
    q, s, w = torch.randn(M, 1, N), torch.randn(M, 1, S), torch.rand(M, 1, 1) + 0.5
    qc = q.cuda().requires_grad_(True)
    out = mixer(qc, s.cuda())
    (out * w.cuda()).sum().backward()
    q64 = q.double().requires_grad_(True)
    oo = MO.qmix_mix(sd, q64, s.double(), PU.oracle_cfg(args))
    (oo * w.double()).sum().backward()
    assert _rel(out, oo) < TOL and _rel(qc.grad, q64.grad) < TOL
    for k, prm in mixer.named_parameters():
        assert _rel(prm.grad, sd[k].grad) < TOL, k


# ------------------------------------------------------------------------------------------ the embed field of the ABI
def _fwd(p, N, S, M=64):
    torch.manual_seed(0)
    q, s = torch.randn(M, N, device="cuda"), torch.randn(M, S, device="cuda")
    hy, q_tot = torch.empty(M, hy_cols(N, 32), device="cuda"), torch.empty(M, device="cuda")
    L.call("marl_qmix_fwd", M, N, S, C.byref(p), q.data_ptr(), s.data_ptr(), hy.data_ptr(), q_tot.data_ptr(),
           L.stream_ptr())
    torch.cuda.synchronize()
    return hy, q_tot


def test_embed_zero_means_32_bit_for_bit():
    N, S = 5, 9
    _, sd = _mixer_params(32, N, S, seed=3)
    t = _device_flat(sd, N, 32, S)
    h0, q0 = _fwd(_params(t, 0), N, S)
    h1, q1 = _fwd(_params(t, 32), N, S)
    assert torch.equal(h0, h1) and torch.equal(q0, q1)


def test_out_of_range_and_mismatched_embed_raise():
    N, S, M, E = 3, 5, 16, 16
    _, sd = _mixer_params(E, N, S, seed=4)
    t = _device_flat(sd, N, E, S)
    z = torch.zeros(M * hy_cols(N, 128), device="cuda")
    for bad in (129, -1, 1000):
        with pytest.raises(ValueError):
            L.call("marl_qmix_fwd", M, N, S, C.byref(_params(t, bad)), z.data_ptr(), z.data_ptr(), z.data_ptr(),
                   z.data_ptr(), L.stream_ptr())
        with pytest.raises(ValueError):
            L.call("marl_qmix_mix_fwd", M, N, C.byref(_params(t, bad)), z.data_ptr(), z.data_ptr(), z.data_ptr(),
                   L.stream_ptr())
    d = L.Dims(4, 4, N, 2, 1, S)
    _, gs = _grads(E, N, S)
    u = torch.zeros(M * N, dtype=torch.int64, device="cuda")
    for pe, pte, ge in ((E, 32, E), (E, 0, E), (E, E, 64)):          # eval / target / gradient widths disagree
        gs.embed = ge
        with pytest.raises(ValueError):
            L.call("marl_qmix_td_fwd_bwd", C.byref(d), C.byref(_params(t, pe)), C.byref(_params(t, pte)), z.data_ptr(),
                   z.data_ptr(), z.data_ptr(), z.data_ptr(), u.data_ptr(), z.data_ptr(), z.data_ptr(), z.data_ptr(), 0.99,
                   z.data_ptr(), z.data_ptr(), z.data_ptr(), z.data_ptr(), z.data_ptr(), z.data_ptr(), C.byref(gs),
                   z.data_ptr(), 0, None, None, None, L.stream_ptr())
    gs.embed = 33
    with pytest.raises(ValueError):
        L.call("marl_qmix_mix_bwd", M, N, C.byref(_params(t, E)), z.data_ptr(), z.data_ptr(), z.data_ptr(), z.data_ptr(),
               z.data_ptr(), C.byref(gs), L.stream_ptr())
    p2 = L.QmixHyper2(*([z.data_ptr()] * 10), 16, 200)
    with pytest.raises(ValueError):
        L.call("marl_qmix_hyper2_fwd", M, N, S, C.byref(p2), z.data_ptr(), z.data_ptr(), z.data_ptr(), L.stream_ptr())
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------ learner against the fp64 oracle
def _shape_args(shape, E, **kw):
    N, A, O, S, T, _ = shape
    return PU.make_args("qmix", N, A, O, S, T, qmix_hidden_dim=E, **kw)


def _batch(shape, seed=0):
    N, A, O, S, T, B = shape
    return synthetic_batch(seed, B, T, N, A, O, S)


def _train_vs_fp64(args, batch, steps=3):
    """Per step, on the same weights (both oracles are re-loaded with the learner's weights before each step; targets stay
    those of step 0, as target_update_cycle says): the fused step's loss against the fp64 oracle, its clipped gradients
    against the fp32 oracle with the fp64 oracle as the arbiter of abs / ReLU kinks (PU.compare_grads: a tensor off by more
    than 1e-5 passes when it is as close to fp64 as the fp32 oracle is).  The update itself is the width-independent optimiser
    kernel; a kink-flipped gradient entry moves its parameter by up to ~lr under RMSprop, so parameters are not compared here."""
    learner, _ = PU.build_pair(args)
    st32, st64 = (MO.LearnerState(PU.oracle_cfg(args), PU.export_params(learner), dtype=dt) for dt in (torch.float32, torch.float64))
    report = []
    for step in range(steps):
        for st in (st32, st64):
            for g, m in PU.module_groups(learner).items():
                for k, v in m.state_dict().items():
                    st.params[g][k] = v.detach().cpu().to(st.dtype).requires_grad_(True)
        loss = learner.train({k: v.copy() for k, v in batch.items()}, step)
        oloss, info = MO.train_step(st64, batch, step)
        info32 = MO.train_step(st32, batch, step)[1]
        if abs(loss - oloss) > TOL * abs(oloss):
            report.append(f"step {step}: loss {loss} vs {oloss}")
        mine = {f"{g}.{k}": p.grad for g, m in PU.module_groups(learner).items() for k, p in m.named_parameters()}
        before = len(report)
        # (whole gradient within 5e-5: the entries of a tolerated kink flip count there too)
        PU.compare_grads(mine, info32["clipped_grads"], TOL, report, info["clipped_grads"], whole_tol=5 * TOL)
        report[before:] = [f"step {step}: {r}" for r in report[before:]]
    assert not report, "\n".join(report)
    return learner


CASES = {"rms": {}, "adam": dict(optimizer="Adam"), "no_double_q": dict(double_q=False),
         "two_hyper_16": dict(two_hyper_layers=True, hyper_hidden_dim=16),
         "two_hyper_64": dict(two_hyper_layers=True, hyper_hidden_dim=64)}


@pytest.mark.parametrize("E", [16, 64, 128])
@pytest.mark.parametrize("case", list(CASES))
def test_learner_tiny_shape_vs_fp64_oracle(E, case):
    _train_vs_fp64(_shape_args(TINY, E, **CASES[case]), _batch(TINY))


# cfg-2 shape: every width with RMSprop, each other case at one width (the fp64 oracle at this shape is the slow part)
@pytest.mark.parametrize("E,case", [(16, "rms"), (64, "rms"), (128, "rms"), (16, "adam"), (64, "no_double_q"),
                                    (128, "two_hyper_16"), (64, "two_hyper_64")])
def test_learner_cfg2_shape_vs_fp64_oracle(E, case):
    _train_vs_fp64(_shape_args(CFG2, E, **CASES[case]), _batch(CFG2), steps=2)


# ------------------------------------------------------------------------------------------ learner, other routes (E = 64)
def _losses(args, batches, seed=0, make=None):
    learner = make(args) if make else PU.build_pair(args, seed=seed)[0]
    return [learner.train(b if not isinstance(b, dict) else {k: v.copy() for k, v in b.items()}, i)
            for i, b in enumerate(batches)], learner


def test_fused_step_matches_module_path():
    batch = _batch(TINY)
    out = {}
    for modules in (False, True):
        args = _shape_args(TINY, 64, train_through_modules=modules)
        out[modules] = _losses(args, [batch] * 3)
    (lf, f), (lm, m) = out[False], out[True]
    assert np.allclose(lf, lm, rtol=TOL, atol=0), (lf, lm)
    assert _rel(f._flat.grad, m._flat.grad) < 1e-4        # clipped gradients after three updates of each path


def test_two_graph_captured_batch_shapes():
    """Two (B, L) keys, each replayed from its own captured graph, against eager runs of the same steps."""
    N, A, O, S, T, _ = TINY
    b1, b2 = synthetic_batch(0, 4, T, N, A, O, S), synthetic_batch(1, 6, T, N, A, O, S, full_length_first=False, min_len=3)
    seq = [b1, b2, b1, b2, b1, b2, b1, b2]
    lg, learner = _losses(_shape_args(TINY, 64), seq)
    assert sum(1 for v in learner._graphs.values() if isinstance(v, tuple)) == 2
    le, _ = _losses(_shape_args(TINY, 64, cuda_graph=False), seq)
    assert np.allclose(lg, le, rtol=TOL, atol=0), (lg, le)


def test_replay_buffer_sample_into_train():
    from marl_b200.common.replaybuffer import ReplayBuffer
    from oracle.replay_oracle import OracleReplayBuffer
    N, A, O, S, T, _ = TINY
    args = _shape_args(TINY, 64, buffer_size=10)
    la, st = PU.build_pair(args)
    lb, _ = PU.build_pair(args)
    buf, orc = ReplayBuffer(args), OracleReplayBuffer(10, T, N, A, O, S)
    for seed in range(3):
        ep = synthetic_batch(seed, 4, T, N, A, O, S, full_length_first=False, min_len=2)
        buf.store_episode({k: v.copy() for k, v in ep.items()})
        orc.store(ep)
    for step in range(3):
        np.random.seed(10 + step)
        host_batch, _ = orc.sample(6)
        np.random.seed(10 + step)
        view = buf.sample(6)
        a = la.train({k: v.copy() for k, v in host_batch.items()}, step)
        b = lb.train(view, step)
        assert abs(a - b) <= 1e-6 * abs(a)
        oloss, _ = MO.train_step(st, host_batch, step)
        assert abs(b - oloss) <= TOL * abs(oloss)


def _separated_learner(args):
    from marl_b200.controller.share_params import SeparatedMAC
    from marl_b200.algorithm.q_learner import QLearner
    torch.manual_seed(0)
    learner = QLearner(SeparatedMAC(args), args)
    learner._update_targets()
    return learner


def test_separated_mac():
    batch = _batch(TINY)
    args = _shape_args(TINY, 64, reuse_network=False)
    lf, learner = _losses(args, [batch] * 3, make=_separated_learner)
    args_m = _shape_args(TINY, 64, reuse_network=False, train_through_modules=True)
    lm, _ = _losses(args_m, [batch] * 3, make=_separated_learner)
    assert np.allclose(lf, lm, rtol=TOL, atol=0), (lf, lm)
    cfg = PU.oracle_cfg(args)
    cfg.separated, cfg.reuse_network = True, False
    fresh = _separated_learner(args)
    params = {f"agent.{n}": {k: v.detach().cpu().clone() for k, v in net.state_dict().items()}
              for n, net in enumerate(fresh.eval_net.agent)}
    params["mixer"] = {k: v.detach().cpu().clone() for k, v in fresh.mixer.state_dict().items()}
    st = MO.LearnerState(cfg, params)
    oloss, _ = MO.train_step(st, batch, 0)
    assert abs(lf[0] - oloss) <= TOL * abs(oloss)


def _separated_oracle(learner, args):
    cfg = PU.oracle_cfg(args)
    cfg.separated, cfg.reuse_network = True, False
    params = {f"agent.{n}": {k: v.detach().cpu().clone() for k, v in net.state_dict().items()}
              for n, net in enumerate(learner.eval_net.agent)}
    params["mixer"] = {k: v.detach().cpu().clone() for k, v in learner.mixer.state_dict().items()}
    return MO.LearnerState(cfg, params)


# Shapes whose fused selection staging sits just under 40 KB of dynamic shared memory: with the wider instantiations' larger
# static shared memory the launch passes 48 KB in total and needs the opt-in.  Shared: selection + heads (N 5, A 8: 40896 B);
# separated: selection only (N 10, A 64: 40960 B).
@pytest.mark.parametrize("E", [64, 96, 128])         # J = 2, 3, 4
@pytest.mark.parametrize("separated", [False, True])
def test_fused_step_with_staging_near_48kb(E, separated):
    N, A = (10, 64) if separated else (5, 8)
    shape = (N, A, 6, 7, 6, 4)
    args = _shape_args(shape, E, reuse_network=not separated)
    learner, st = (_separated_learner(args), None) if separated else PU.build_pair(args)
    if separated:
        st = _separated_oracle(learner, args)
    fused = learner._fusion()
    assert fused.select and fused.heads == (not separated)
    batch = _batch(shape)
    for step in range(3):                          # eager, eager, graph capture + replay
        loss = learner.train({k: v.copy() for k, v in batch.items()}, step)
        oloss, _ = MO.train_step(st, batch, step)
        assert abs(loss - oloss) <= TOL * abs(oloss), step


def _narrow(sd, N, E_from, E_to):
    """A state_dict of width E_from cut to its first E_to embed slots."""
    S = sd["hyper_b1.weight"].shape[1]
    out = dict(sd)
    out["hyper_w1.weight"] = sd["hyper_w1.weight"].view(N, E_from, S)[:, :E_to].reshape(N * E_to, S)
    out["hyper_w1.bias"] = sd["hyper_w1.bias"].view(N, E_from)[:, :E_to].reshape(-1)
    for h in ("hyper_b1", "hyper_w2", "hyper_b2.0"):
        out[h + ".weight"], out[h + ".bias"] = sd[h + ".weight"][:E_to], sd[h + ".bias"][:E_to]
    out["hyper_b2.2.weight"] = sd["hyper_b2.2.weight"][:, :E_to]
    return {k: v.contiguous() for k, v in out.items()}


def _wide_grad_rows(g, N, E_from, E_to):
    """(rows of a width-E_from wcat / bcat gradient that a width-E_to problem has, the others)."""
    idx = torch.zeros(hy_cols(N, E_from), dtype=torch.bool)
    for n in range(N):
        idx[n * E_from:n * E_from + E_to] = True
    for h in range(3):
        idx[N * E_from + h * E_from:N * E_from + h * E_from + E_to] = True
    return g[idx.to(g.device)], g[~idx.to(g.device)]


@pytest.mark.parametrize("E_small,E_big", [(31, 32), (32, 33)])
@pytest.mark.parametrize("N", [2, 5])
def test_neighbouring_widths_agree_with_e32(E_small, E_big, N):
    """qmix_mix_kernel (E = 32) and qmix_mix_kernel_e<J> are the same algorithm in two sources: on a width-E_big mixer whose
    last embed slot is zero (every head row, bias and hyper_b2.2 entry), the width-E_small mixer of the other slots gives the
    same q_tot, dq and gradients, and the zero slot's gradient rows are zero."""
    S, M = 9, 500
    _, sd = _mixer_params(E_big, N, S, seed=N)
    sd = {k: v.clone() for k, v in sd.items()}
    sd["hyper_w1.weight"].view(N, E_big, S)[:, E_small:] = 0
    sd["hyper_w1.bias"].view(N, E_big)[:, E_small:] = 0
    for h in ("hyper_b1", "hyper_w2", "hyper_b2.0"):
        sd[h + ".weight"][E_small:], sd[h + ".bias"][E_small:] = 0, 0
    sd["hyper_b2.2.weight"][:, E_small:] = 0
    small = _narrow(sd, N, E_big, E_small)
    torch.manual_seed(5)
    q, s, w = torch.randn(M, N, device="cuda"), torch.randn(M, S, device="cuda"), torch.rand(M, device="cuda") + 0.5
    res = {}
    for E, p_sd in ((E_big, sd), (E_small, small)):
        t = _device_flat(p_sd, N, E, S)
        p = _params(t, E)
        hy, dhy = torch.empty(M, hy_cols(N, E), device="cuda"), torch.empty(M, hy_cols(N, E), device="cuda")
        q_tot, dq = torch.empty(M, device="cuda"), torch.empty(M, N, device="cuda")
        g, gs = _grads(E, N, S)
        L.call("marl_qmix_fwd", M, N, S, C.byref(p), q.data_ptr(), s.data_ptr(), hy.data_ptr(), q_tot.data_ptr(),
               L.stream_ptr())
        L.call("marl_qmix_bwd", M, N, S, C.byref(p), q.data_ptr(), s.data_ptr(), hy.data_ptr(), w.data_ptr(),
               dhy.data_ptr(), dq.data_ptr(), C.byref(gs), L.stream_ptr())
        torch.cuda.synchronize()
        res[E] = (q_tot, dq, g)
    (qb, dqb, gb), (qs, dqs, gs_) = res[E_big], res[E_small]
    assert _rel(qb, qs) < 1e-6 and _rel(dqb, dqs) < 1e-6
    for i in (0, 1):                                                   # wcat, bcat
        kept, dropped = _wide_grad_rows(gb[i], N, E_big, E_small)
        assert _rel(kept, gs_[i]) < 1e-6, i
        assert torch.count_nonzero(dropped) == 0, i
    assert _rel(gb[2][:E_small], gs_[2]) < 1e-6 and float(gb[2][E_small:].abs().max()) == 0.0
    assert _rel(gb[3], gs_[3]) < 1e-6


def test_last_action_off():
    args = _shape_args(TINY, 64, last_action=False)
    learner, st = PU.build_pair(args)
    st.cfg.last_action = False
    batch = _batch(TINY)
    for step in range(3):
        loss = learner.train({k: v.copy() for k, v in batch.items()}, step)
        oloss, _ = MO.train_step(st, batch, step)
        assert abs(loss - oloss) <= TOL * abs(oloss), step


@pytest.mark.parametrize("E,N", [(64, 5), (7, 2)])
def test_tma_gemm_back_end(E, N):
    """MARL_B200_TGEMM=1: an hy whose pitch is TMA-addressable (N E + 3 E a multiple of 4) goes through tgemm.cu, one that
    is not (E = 7, N = 2: pitch 35) stays on linear.cu; both train like the oracle."""
    shape = (N, 4, 8, 12, 8, 8)
    prev = L.load().marl_tgemm_enable(1)
    try:
        args = _shape_args(shape, E, cuda_graph=False)
        learner, st = PU.build_pair(args)
        batch = _batch(shape)
        for step in range(2):
            loss = learner.train({k: v.copy() for k, v in batch.items()}, step)
            oloss, _ = MO.train_step(st, batch, step)
            assert abs(loss - oloss) <= TOL * abs(oloss), step
        # the hyper-network GEMM of the mixer alone
        M, S = 512, shape[3]
        s = torch.randn(M, S, device="cuda")
        hy = torch.empty(M, hy_cols(N, E), device="cuda")
        p, _ = learner._qmix_structs(learner._flat)
        torch.cuda.synchronize()
        L.profile(True)
        L.call("marl_qmix_hyper_fwd", M, N, S, C.byref(p), s.data_ptr(), hy.data_ptr(), L.stream_ptr())
        launched = L.profile_collect()
        L.profile(False)
        want = "tgemm_kernel" if hy_cols(N, E) % 4 == 0 else "linear_fwd_kernel"
        assert set(launched) == {want}, launched
        w0 = learner._flat.offsets["mixer.hyper_w1.weight"]
        b0 = learner._flat.offsets["mixer.hyper_w1.bias"]
        Cc = hy_cols(N, E)
        wcat = learner._flat.data[w0:w0 + Cc * S].view(Cc, S).double()
        bcat = learner._flat.data[b0:b0 + Cc].double()
        assert _rel(hy, s.double() @ wcat.T + bcat) < TOL
    finally:
        L.load().marl_tgemm_enable(prev)


def test_launch_count_equals_the_e32_count():
    batch = _batch(TINY)
    counts = {}
    for E in (32, 64, 7):
        _, learner = _losses(_shape_args(TINY, E, cuda_graph=False), [batch])
        counts[E] = learner.launches_per_step
        L.profile(True)
        learner.train({k: v.copy() for k, v in batch.items()}, 1)
        launched = L.profile_collect()
        L.profile(False)
        counts[E] = (counts[E], sum(c for c, _ in launched.values()), launched.get("qmix_mix_kernel", (0,))[0])
    assert counts[64] == counts[32] and counts[7] == counts[32], counts


# ------------------------------------------------------------------------------------------ other surfaces
def test_checkpoint_round_trip(tmp_path):
    args = _shape_args(TINY, 64)
    args.model_dir = str(tmp_path)
    src, _ = PU.build_pair(args, seed=0)
    batch = _batch(TINY)
    src.train({k: v.copy() for k, v in batch.items()}, 0)
    src.save_models(0)
    for k in ("rnn_net_params", "mixer_net_params"):
        os.replace(os.path.join(src.model_dir, f"0_{k}.pkl"), os.path.join(src.model_dir, f"{k}.pkl"))
    dst, _ = PU.build_pair(args, seed=1)
    dst.load_models()
    for a, b in ((src.mixer, dst.mixer), (src.eval_net.agent, dst.eval_net.agent)):
        sa, sb = a.state_dict(), b.state_dict()
        assert sa.keys() == sb.keys() and all(torch.equal(sa[k], sb[k]) for k in sa)
    assert tuple(dst.mixer.state_dict()["hyper_w1.weight"].shape) == (TINY[0] * 64, TINY[3])
    src._update_targets()
    dst._update_targets()
    a = src.train({k: v.copy() for k, v in batch.items()}, 1)
    b = dst.train({k: v.copy() for k, v in batch.items()}, 1)
    assert abs(a - b) <= 1e-6 * abs(a)


def test_matrix_game_q_tables_at_embed_8():
    args = PU.make_args("qmix", 2, 3, 1, 1, 1, qmix_hidden_dim=8)
    learner, st = PU.build_pair(args)
    qt, qi, qj = learner.get_q_and_q_tot_table()
    P = {g: {k: v.detach().double() for k, v in sd.items()} for g, sd in st.params.items()}
    x = torch.cat([torch.ones(2, 1), torch.zeros(2, 3), torch.eye(2)], dim=1).double()    # [o | last action | agent id]
    q, _ = MO.agent_step(P["agent"], x, torch.zeros(2, 64, dtype=torch.float64))
    assert _rel(qi, q[0]) < TOL and _rel(qj, q[1]) < TOL
    want = np.zeros((3, 3))
    for i in range(3):
        for j in range(3):
            chosen = torch.stack([q[0, i], q[1, j]]).view(1, 1, 2)
            want[i, j] = float(MO.qmix_mix(P["mixer"], chosen, torch.ones(1, 1, 1, dtype=torch.float64), st.cfg))
    assert _rel(qt, want) < TOL


def _dp_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    learner, _ = PU.build_pair(_shape_args(TINY, 64))
    learner.enable_data_parallel()
    batch = _batch(TINY)
    ret[rank] = ([learner.train({k: v.copy() for k, v in batch.items()}, i) for i in range(4)],
                 learner._flat.data.cpu().numpy())
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpu_data_parallel():
    import socket
    import torch.multiprocessing as mp
    sock = socket.socket()
    sock.bind(("127.0.0.1", 0))
    port = sock.getsockname()[1]
    sock.close()
    ret = mp.Manager().dict()
    mp.spawn(_dp_worker, args=(2, port, ret), nprocs=2, join=True)
    (l0, p0), (l1, p1) = ret[0], ret[1]
    assert l0 == l1 and np.array_equal(p0, p1)
    single, _ = PU.build_pair(_shape_args(TINY, 64))
    batch = _batch(TINY)
    ls = [single.train({k: v.copy() for k, v in batch.items()}, i) for i in range(4)]
    assert np.allclose(l0, ls, rtol=TOL)
