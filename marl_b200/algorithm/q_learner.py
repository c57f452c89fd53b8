"""VDN / QMIX / QPLEX learner on sm_100a kernels, drop-in for ``algorithm/q_learner.py:10-262``.

``QLearner(mac, args).train(batch, train_step) -> float`` keeps the reference's contract (same
batch dict in the ReplayBuffer layout, same loss value, same parameter update, same target-sync
cadence, ``mac.hidden_states`` left as the reference leaves it) but executes as a short fixed
sequence of libmarl_b200 calls, captured in a CUDA graph per (B, L):

    ingest (f64 -> f32)                      marl_ingest_f64            q_learner.py:63-91
    3 agent unrolls (eval/o, eval/o_next     marl_agent_unroll_fwd      :96-97, :103-104, :110
      chained to it, target/o_next)
    gather / masked argmax / target gather   marl_q_select              :100, :105, :111-117
    mixer + TD loss + their gradient         marl_{vdn,qmix}_td_fwd_bwd :161-168, :171
    BPTT through the eval/o unroll           marl_agent_unroll_bwd      :171
    [data parallel: one NCCL all-reduce of the flat gradient + (loss_sum, mask_sum)]
    clip_grad_norm_ + RMSprop/Adam           marl_clip_{rmsprop,adam}_step   :172-173
    target sync = one D2D copy               :176-177, :181-184

No autograd, no PyTorch arithmetic and no CPU fallback on this path.
"""
from __future__ import annotations

import copy
import ctypes as C
import os
from collections import namedtuple

import numpy as np
import torch as th

from .. import _lib as L
from ..flat import FlatBuffer, prefixed
from ..parallel import shard_bounds, allreduce_flat, PeerGradients
from ..common.replaybuffer import DeviceEpisodeBatch
from ..network.mixer import VDNMixer, QMixMixer, qmix_struct, qmix2_struct, qmix_tail_struct
from ..network.q_network import agent_param_struct

H = 64
BATCH_KEYS = ("o", "u", "s", "r", "o_next", "s_next", "avail_u", "avail_u_next", "u_onehot", "padded", "terminated")


# One stream of marl_agent_unroll_fwd: batch key of the input; shift of the last-action one-hot (1: u_onehot one step back, for
# o; 0: for o_next); target net's weights (else the eval net's); stream whose final hidden state it starts from (-1: zeros); keep
# the gates and W_ih^T for the BPTT
_Unroll = namedtuple("_Unroll", "obs shift target h0_from keep")
_EVAL_O = _Unroll("o", 1, False, -1, True)                # eval net on o          (q_learner.py:96-97)
_TARGET_O_NEXT = _Unroll("o_next", 0, True, -1, False)    # target net on o_next   (:103-104)
_EVAL_O_NEXT = _Unroll("o_next", 0, False, 0, False)      # eval net on o_next, hidden carried (:110)
_Fusion = namedtuple("_Fusion", "select heads dhext")       # QLearner._fusion


def host_max_episode_len(terminated, episode_limit):
    """q_learner.py:49-61 vectorised: 1 + the largest first-terminated index, limit if none."""
    term = np.asarray(terminated)[:, :episode_limit, 0] == 1
    has = term.any(axis=1)
    if not has.any():
        return int(episode_limit)
    return int(term.argmax(axis=1)[has].max()) + 1


class _FlatOptimizer:
    """Facade with the torch.optim surface the reference touches (zero_grad / state)."""

    def __init__(self, kind, lr, flat, device):
        self.kind, self.lr = kind, lr
        self.defaults = dict(lr=lr, alpha=0.99, eps=1e-8, betas=(0.9, 0.999))
        n = flat.numel
        z = lambda: th.zeros(n, dtype=th.float32, device=device)
        if kind == "RMS":
            self.square_avg = z()
        else:
            self.exp_avg, self.exp_avg_sq = z(), z()
            self.step_counter = th.zeros(1, dtype=th.int32, device=device)
        self._flat = flat

    def zero_grad(self, set_to_none=False):
        self._flat.grad_full.zero_()

    def state_dict(self):
        if self.kind == "RMS":
            return {"square_avg": self.square_avg}
        return {"exp_avg": self.exp_avg, "exp_avg_sq": self.exp_avg_sq, "step": self.step_counter}


class QLearner:
    def __init__(self, mac, args):
        self.max_episode_len = args.episode_limit
        self.gamma = args.gamma
        self.lr = args.lr
        self.model_dir = args.model_dir + '/' + args.alg + '/' + args.map
        self.args = args

        self.eval_net = mac
        self.target_net = copy.deepcopy(mac)
        self.params = list(mac.parameters())
        self.mixer = self._make_mixer(args)
        self.target_mixer = copy.deepcopy(self.mixer)
        self.params += list(self.mixer.parameters())
        self._build_extra(args)
        if args.optimizer not in ("RMS", "Adam"):
            raise ValueError("optimizer {} not recognised.".format(args.optimizer))

        self._dev = th.device("cuda") if th.cuda.is_available() else th.device("cpu")
        self._pack()
        self._ws = {}
        self._graphs = {}
        self._use_graph = bool(getattr(args, "cuda_graph", True))
        self._dist = None
        self._peer = None
        self._side = []
        self._copy_stream, self._prefetched, self._slot_free, self._prefetch_seq = None, {}, {}, 0
        self.last = {}
        self.launches_per_step = 0
        self.ingest_launches = 1
        self._inplace_keep, self._max_inplace_graphs = {}, 32
        self._capture_after = int(getattr(args, "graph_capture_after", 2))      # eager sightings of a (B, L) before its graph is captured

    # ---- construction helpers ---------------------------------------------------------------------
    def _make_mixer(self, args):
        if args.alg == 'vdn':
            return VDNMixer(args)
        if args.alg == 'qmix':
            return QMixMixer(args)
        if args.alg == 'qplex':
            from ..network.qplex import DMAQer
            return DMAQer(args)
        raise ValueError("Mixer {} not recognised.".format(args.alg))

    def _pack(self):
        """All optimised tensors into one flat buffer (+grad +2 tail scalars); targets mirror it."""
        dev = self._dev
        separated = isinstance(self.eval_net.agent, (list, tuple))          # SeparatedMAC: one network per agent
        agents_of = lambda mac: list(mac.agent) if separated else [mac.agent]
        tag = (lambda i: f"agent.{i}.") if separated else (lambda i: "agent.")
        named = []
        for i, ag in enumerate(agents_of(self.eval_net)):
            named += prefixed(tag(i), ag.flat_named_parameters())
        named += prefixed("mixer.", self.mixer.flat_named_parameters())
        for prefix, module in self._extra_groups():
            named += prefixed(prefix, module.flat_named_parameters())
        self._flat = FlatBuffer(named, device=dev, with_grad=True, extra_tail=2)
        tnamed = []
        for i, ag in enumerate(agents_of(self.target_net)):
            tnamed += prefixed(tag(i), ag.flat_named_parameters())
        tnamed += prefixed("mixer.", self.target_mixer.flat_named_parameters())
        self._tflat = FlatBuffer(tnamed, device=dev, with_grad=False)
        for ag in agents_of(self.eval_net):
            ag.adopt(self._flat)
        for ag in agents_of(self.target_net):
            ag.adopt(self._tflat)
        self._separated = separated
        if hasattr(self.mixer, "adopt"):
            self.mixer.adopt(self._flat)
            self.target_mixer.adopt(self._tflat)
        for _, module in self._extra_groups():
            module.adopt(self._flat)
        self.optimizer = _FlatOptimizer(self.args.optimizer, self.lr, self._flat, dev)
        self._partials = th.zeros(L.load().marl_optim_partials() if os.path.exists(L.LIB_PATH) else 148,
                                  dtype=th.float32, device=dev)
        self._graph_key = None
        self._inplace_cache = {}
        self._ring_structs = {}
        self._agent_sets = {}        # id(flat) -> agent stride (separated_stride), for the two flat buffers packed here
        # (loss, gradient norm) of a step: the optimiser kernel stores them straight into the page-locked host buffer (the host
        # pointer is the device pointer), so the read-back the reference's loss.item() implies is two posted PCIe writes at the end
        # of the step's last kernel instead of a copy queued behind it (317 -> 308 us per step, profiles/r2c_ab_loss_zerocopy.txt)
        self._loss_host = th.zeros(2, dtype=th.float32).pin_memory() if dev.type == "cuda" else th.zeros(2)
        self._ws, self._graphs = {}, {}

    def _build_extra(self, args):
        """Hook: networks created after the mixer, in the reference's construction order."""

    def _extra_groups(self):
        """(prefix, module) pairs optimised besides the agent and the mixer (QTRAN: the V network)."""
        return []

    def cuda(self):
        self._dev = th.device("cuda")
        self._pack()

    def enable_data_parallel(self, group=None):
        """Shard every batch along the episode axis over the ranks of `group` and all-reduce the
        flat [grad | loss_sum | mask_sum] buffer once per step (SURVEY.md section 8(e))."""
        import torch.distributed as dist
        self._dist = (dist, group)
        self._graphs = {}
        if self._peer is not None:      # called again: release the previous IPC mappings first
            self._flat.adopt_grad_storage(th.zeros_like(self._flat.grad_full))
            self._peer.close()
        self._peer = None
        # same node, <= 8 ranks, <= 2^18 parameters: the gradient sum happens inside the optimiser launch over NVLink
        # peer memory (marl_clip_step_peer) instead of an NCCL call between two graphs
        if (self._dev.type == "cuda" and dist.get_backend(group) == "nccl" and dist.get_world_size(group) > 1
                and os.environ.get("MARL_B200_PEER_ALLREDUCE", "1") != "0"):
            peer = PeerGradients(self._flat.numel, dist, group, self._dev)
            if peer.ok:
                self._flat.adopt_grad_storage(peer.grad_full)
                self._peer = peer

    # ---- reference surface: episode-length cut ------------------------------------------------------
    def get_max_episode_len(self, batch):
        L_ = host_max_episode_len(_to_numpy(batch["terminated"]), self.args.episode_limit)
        for key in batch.keys():
            batch[key] = batch[key][:, :L_]
        return batch, L_

    # ---- staging -------------------------------------------------------------------------------------
    def _dims(self, B, Lq):
        a = self.args
        return L.Dims(B, Lq, a.n_agents, a.n_actions, a.obs_shape, a.state_shape)

    def _workspace(self, B, Lq):
        key = (B, Lq)
        ws = self._ws.get(key)
        if ws is not None:
            return ws
        a, dev = self.args, self._dev
        N, A, O, S = a.n_agents, a.n_actions, a.obs_shape, a.state_shape
        rows, M = B * Lq * N, B * Lq
        f = lambda *shape: th.empty(*shape, dtype=th.float32, device=dev)
        ws = dict(
            batch=dict(o=f(B, Lq, N, O), s=f(B, Lq, S), u=th.empty(B, Lq, N, dtype=th.int64, device=dev), r=f(B, Lq),
                       o_next=f(B, Lq, N, O), s_next=f(B, Lq, S), avail_u=f(B, Lq, N, A), avail_u_next=f(B, Lq, N, A),
                       u_onehot=f(B, Lq, N, A), padded=f(B, Lq), terminated=f(B, Lq)),
            x=[f(rows, H) for _ in range(3)], gi=[f(rows, 3 * H) for _ in range(3)],
            # (zero-initialised: with args.early_exit the steps behind an episode's end are never written, and the masked
            # consumers must still read finite numbers there)
            hidden=[th.zeros(B, Lq, N, H, dtype=th.float32, device=dev) for _ in range(3)],
            q=[th.zeros(B, Lq, N, A, dtype=th.float32, device=dev) for _ in range(3)],
            ep_len=th.ones(B, dtype=th.int32, device=dev),
            # length-sorted deal of the recurrence rows under args.early_exit: one array per stream + one for the BPTT plan
            row_order=th.zeros(4, B * N, dtype=th.int32, device=dev),
            h_last=[f(B * N, H) for _ in range(3)], gates=f(rows, 4 * H), w_ih_t=f(H, 3 * H),
            q_chosen=f(B, Lq, N), q_tc=f(B, Lq, N), a_star=th.empty(B, Lq, N, dtype=th.int64, device=dev),
            q_tot=f(B, Lq, 1), q_tot_t=f(B, Lq, 1), dq=f(B, Lq, N, A),
            dhext=f(rows, H), dgi=f(rows, 3 * H), dgh=f(rows, 3 * H), dx=f(rows, H),
        )
        ws["h_last_sep"] = [h.view(B, N, H) for h in ws["h_last"]]
        if a.alg == "qmix":
            Ccols = N * 32 + 96
            ws.update(hy=f(M, Ccols), hy_t=f(M, Ccols), dhy=f(M, Ccols))
            if getattr(a, "two_hyper_layers", False):
                hh2 = 2 * a.hyper_hidden_dim
                ws.update(hh=f(M, hh2), hh_t=f(M, hh2), dhh=f(M, hh2))
        if a.alg == "qplex":
            from ..network.qplex import qplex_workspace
            ws.update(qp=qplex_workspace(M, a, dev), qp_t=qplex_workspace(M, a, dev), dqp=qplex_workspace(M, a, dev),
                      max_q=f(B, Lq, N), qt_max=f(B, Lq, N), oh_star=f(B, Lq, N, A), dq_tot=f(M), dq_small=f(B, Lq, N))
        self._ws[key] = ws
        return ws

    def _upload(self, batch, slot):
        """Host dict (numpy float64, [B, T_src, ...]) -> device staging buffers `slot` (async when pinned)."""
        a, dev = self.args, self._dev
        Lq = host_max_episode_len(_to_numpy(batch["terminated"]), a.episode_limit)
        arrs = {k: _to_numpy(batch[k]) for k in BATCH_KEYS}
        B_glob, T_src = arrs["o"].shape[0], arrs["o"].shape[1]
        lo, hi = self._shard(B_glob)
        B = hi - lo
        key = ("stage", B, T_src, slot)
        st = self._ws.get(key)
        if st is None:
            st = {}
            for k in BATCH_KEYS:
                shape = (B,) + arrs[k].shape[1:]
                dt = th.int64 if (k == "u" and arrs[k].dtype.kind in "iu") else th.float64
                st[k] = th.empty(shape, dtype=dt, device=dev)
            self._ws[key] = st
        h2d = 0
        # VDN / QMIX never read avail_u (only avail_u_next, q_learner.py:105,112): do not ship it
        skip = ("avail_u",) if a.alg in ("vdn", "qmix") else ()
        for k in BATCH_KEYS:
            if k in skip:
                continue
            src = arrs[k][lo:hi]
            want = np.int64 if st[k].dtype == th.int64 else np.float64
            if src.dtype != want or not src.flags.c_contiguous:
                src = np.ascontiguousarray(src, dtype=want)
            st[k].copy_(th.from_numpy(src), non_blocking=True)
            h2d += src.nbytes
        return dict(st=st, B=B, L=Lq, T_src=T_src, skip=skip, h2d=h2d)

    def prefetch(self, batch):
        """Optional: start the host->device copy of the NEXT batch on a copy stream while the current step
        computes.  A later ``train(batch)`` with the same dict object picks the copy up instead of repeating it.
        (The reference's loop samples a fresh mini-batch before every ``train`` call, runner.py:96-97, so the
        next batch is known early.)"""
        if self._dev.type != "cuda" or (th.is_tensor(batch["o"]) and batch["o"].is_cuda):
            return
        if self._copy_stream is None:
            self._copy_stream = th.cuda.Stream()
        slot = 1 + (self._prefetch_seq & 1)
        self._prefetch_seq += 1
        # two staging slots = at most two outstanding prefetches: whatever still claims this slot (a batch that was
        # prefetched and never trained) is dropped, so a stale entry can never be handed to a later train() call
        for key in [k for k, e in self._prefetched.items() if e["slot"] == slot]:
            del self._prefetched[key]
        free_ev = self._slot_free.get(slot)
        with th.cuda.stream(self._copy_stream):
            if free_ev is not None:
                self._copy_stream.wait_event(free_ev)       # the ingest that last read this slot has run
            up = self._upload(batch, slot)
            up["ready"] = th.cuda.Event()
            up["ready"].record(self._copy_stream)
        up["slot"] = slot
        up["batch"] = batch          # keeps the dict alive: its id() cannot be recycled while the entry exists
        self._prefetched[id(batch)] = up

    def _stage_host_batch(self, batch):
        """numpy (float64, [B, T_src, ...]) -> H2D (or a prefetched copy) -> marl_ingest_f64 -> fp32 working set."""
        up = self._prefetched.pop(id(batch), None)
        if up is not None and up.get("batch") is not batch:
            up = None
        cur = th.cuda.current_stream()
        if up is not None:
            cur.wait_event(up["ready"])
        else:
            up = self._upload(batch, 0)
            up["slot"] = 0
        st, B, Lq, T_src, skip = up["st"], up["B"], up["L"], up["T_src"], up["skip"]
        self.h2d_bytes_last = up["h2d"]
        ws = self._workspace(B, Lq)
        e64 = L.EpisodeF64()
        for k in BATCH_KEYS:
            setattr(e64, k, st["avail_u_next" if k in skip else k].data_ptr())
        e64.u_is_int64 = int(st["u"].dtype == th.int64)
        d = self._dims(B, Lq)
        e32 = _episode_struct(ws["batch"])
        L.call("marl_ingest_f64", C.byref(e64), T_src, C.byref(d), C.byref(e32), L.stream_ptr())
        if up["slot"]:
            ev = th.cuda.Event()
            ev.record(cur)
            self._slot_free[up["slot"]] = ev
        return ws["batch"], B, Lq, 1

    def _stage_device_batch(self, batch):
        """Dict of CUDA tensors in the device layout (fp32, u int64, [B, T_src, ...]) -> working set.

        One marl_ingest_f32 launch gathers (and truncates to L) the 11 keys into the static working
        set, so the captured CUDA graph never depends on the caller's addresses."""
        a = self.args
        Lq = batch.get("max_episode_len")
        # the same dict of the same tensors at the same addresses as in an earlier call (a resident batch that is trained on again):
        # its in-place staging is reused -- the checks below are ~3 us, the full path ~8 us of a ~285 us step
        ent = self._inplace_cache.get(id(batch))
        if ent is not None and ent[0] is batch and Lq is not None and ent[2] == int(Lq):
            same = True
            for k, t, p in ent[1]:
                v = batch[k]
                if v is not t or v.data_ptr() != p:
                    same = False
                    break
            if same:
                self.h2d_bytes_last, self.ingest_launches, self._graph_key = 0, 0, ent[3]
                return ent[4]
        if Lq is None:
            term = batch["terminated"].reshape(batch["terminated"].shape[0], -1)[:, :a.episode_limit] == 1
            has = term.any(dim=1)
            first = term.to(th.int32).argmax(dim=1)
            Lq = int((first[has].max() + 1).item()) if bool(has.any()) else int(a.episode_limit)
        B_glob, T_src = batch["o"].shape[0], batch["o"].shape[1]
        lo, hi = self._shard(B_glob)
        B = hi - lo
        ws = self._workspace(B, int(Lq))
        src = L.EpisodeF32()
        keep, converted = [], 0
        whole = lo == 0 and hi == B_glob               # (a slice is a new tensor object: ~1.5 us each, eleven per step)
        for k in BATCH_KEYS:
            t = batch[k] if whole else batch[k][lo:hi]
            want = th.int64 if k == "u" else th.float32
            if t.dtype != want or not t.is_contiguous():
                t = t.to(want).contiguous()
                converted += 1
            keep.append(t)
            setattr(src, k, t.data_ptr())
        self.h2d_bytes_last = 0
        if converted == 0 and T_src == int(Lq):
            # already in the working-set layout (fp32 / int64, contiguous, no padding beyond L): the kernels read the
            # caller's tensors in place.  The captured graph is then specific to these addresses, so it is cached
            # per batch (the tensors are kept alive with it); past a few dozen distinct batches the copy path below
            # takes over so that the cache stays bounded.
            bt = dict(zip(BATCH_KEYS, keep))
            key = (B, int(Lq)) + tuple(getattr(src, k) for k in BATCH_KEYS)
            if not self._use_graph or key in self._graphs or len(self._graphs) < self._max_inplace_graphs:
                if self._use_graph:
                    self._inplace_keep[key] = bt
                self.ingest_launches = 0
                self._graph_key = key                  # (_run would rebuild the same tuple from eleven data_ptr() calls)
                if whole and batch.get("max_episode_len") is not None:
                    if len(self._inplace_cache) >= 64:
                        self._inplace_cache.clear()
                    self._inplace_cache[id(batch)] = (batch, [(k, bt[k], bt[k].data_ptr()) for k in BATCH_KEYS],
                                                      int(Lq), key, (bt, B, int(Lq), 1))
                return bt, B, int(Lq), 1
        d = self._dims(B, int(Lq))
        dst = _episode_struct(ws["batch"])
        L.call("marl_ingest_f32", C.byref(src), T_src, C.byref(d), C.byref(dst), L.stream_ptr())
        self.ingest_launches = 1
        return ws["batch"], B, int(Lq), 1

    def _stage_replay_batch(self, batch):
        """``ReplayBuffer.sample()`` of the device-resident buffer (common/replaybuffer.py) -> working set: the
        sampled ring rows are gathered and cut to the batch's max episode length in ONE launch."""
        batch.check_fresh()
        ring, Lq = batch.ring, batch.max_episode_len
        B_glob = int(batch.idx.shape[0])
        lo, hi = self._shard(B_glob)
        B = hi - lo
        ws = self._workspace(B, Lq)
        # the ring's and the working set's address structs do not change from call to call: built once (22 setattr + data_ptr calls)
        rs = self._ring_structs.get(id(ring))
        if rs is None or rs[0] is not ring:
            src = L.EpisodeF32()
            for k in BATCH_KEYS:
                setattr(src, k, ring[k].data_ptr())
            rs = (ring, src, ring["o"].shape[1], tuple(ring[k].data_ptr() for k in BATCH_KEYS))
            self._ring_structs = {id(ring): rs}
        src, T_ring = rs[1], rs[2]
        gs = ws.get("_gather_structs")
        if gs is None:
            gs = ws["_gather_structs"] = (self._dims(B, Lq), _episode_struct(ws["batch"]))
        d, dst = gs
        idx = batch.idx if (lo == 0 and hi == B_glob) else batch.idx[lo:hi]
        L.call("marl_replay_gather_f32", C.byref(src), T_ring, idx.data_ptr(), C.byref(d), C.byref(dst), L.stream_ptr())
        self._keep_alive = idx
        self.h2d_bytes_last = 0
        return ws["batch"], B, Lq, 1

    def _shard(self, B_glob):
        if self._dist is None:
            return 0, B_glob
        dist, group = self._dist
        return shard_bounds(B_glob, dist.get_world_size(group), dist.get_rank(group))

    # ---- the device step -----------------------------------------------------------------------------
    def _agent_plan(self, B, Lq):
        """The step's agent unrolls (stream i writes ws["q" / "hidden" / "h_last" / "x" / "gi"][i]), and whether the
        recurrences stop at each episode's end.

        SURVEY 8(f) N3: args.early_exit: True / False, or None (default) = on from 640 agent rows when there is a time axis to
        cut.  Measured on ragged batches (lengths U{T/2..T}, tools/early_exit_bench.py, profiles/r2c_early_exit.txt): the QMIX
        step is 7 % / 5.5 % / 6 % shorter at B = 128 / 256 / 1024 (640 / 1280 / 5120 rows); at config 2 (160 rows, one or two
        per CTA) the kernels still end with the CTA that holds the longest episode and the shorter chains of the others (-4 us
        forward, -4 us BPTT in isolation) do not show in the step: 317.6 us either way.

        With one network per agent (SeparatedMAC) the recurrences always run to L, whatever args.early_exit says: the rows of
        a pass must belong to one agent, whose W_hh the pass holds in registers, and the length-sorted deal mixes agents."""
        a = self.args
        ee = getattr(a, "early_exit", None)
        early = (B * a.n_agents >= 640 and Lq >= 16) if ee is None else bool(ee)
        plan = (_EVAL_O, _TARGET_O_NEXT, _EVAL_O_NEXT) if a.double_q else (_EVAL_O, _TARGET_O_NEXT)
        return plan, early and not self._separated

    def _agent_structs(self, flat, grad=False):
        """(parameter or gradient struct, agent stride) of the agent in `flat`: the shared network with stride 0, or -- one
        network per agent -- agent 0's set and the distance in floats from agent n's set to agent n+1's."""
        cls, src = (L.AgentGrads, flat.grad) if grad else (L.AgentParams, None)
        if not self._separated:
            return agent_param_struct(flat.addrs("agent.", src), cls), 0
        stride = self._agent_sets.get(id(flat))
        if stride is None:
            stride = self._agent_sets[id(flat)] = separated_stride(flat, self.args.n_agents)
        return agent_param_struct(flat.addrs("agent.0.", src), cls), stride

    def _side_streams(self, n):
        self._side += [th.cuda.Stream() for _ in range(n - len(self._side))]
        return self._side[:n]

    def _fusion(self):
        """What the VDN / QMIX mixing kernel takes over: the greedy selection (it gathers / arg-maxes its own sample, the [N, A]
        slabs of a warp's sample staged in shared memory), the agents' heads q = fc2(h) (no head GEMMs after the unroll) and,
        dq having one non-zero per agent row, dq . fc2_w (no dgrad launch in the BPTT).  With one network per agent only the
        selection: the kernel stages one fc2, not one per agent."""
        a = self.args
        fuse = a.alg in ("vdn", "qmix") and bool(getattr(a, "fused_mixer_kernel", True))   # False: one kernel per stage
        fits = lambda heads: bool(L.load().marl_select_fits(int(a.alg == "qmix"), a.n_agents, a.n_actions, heads))
        select = fuse and fits(0)
        if self._separated:
            return _Fusion(select, False, False)
        fc2_w, fc2_wt = self._flat.ptr("agent.fc2.weight"), self._tflat.ptr("agent.fc2.weight")
        return _Fusion(select, select and fits(1) and fc2_w % 16 == 0 and fc2_wt % 16 == 0, fuse and fc2_w % 8 == 0)

    def _launch_forward_backward(self, bt, ws, B, Lq):
        """Everything between the staged batch and the flat un-normalised gradient: zero it, the mixer's prologue, every agent
        unroll in one launch, the mixer stage, the BPTT.  Each stage returns the launches it issues; this returns their sum."""
        d = self._dims(B, Lq)
        plan, early = self._agent_plan(B, Lq)
        fused = self._fusion()
        self._flat.grad_full.zero_()
        n = 1 + self._mixer_prologue(bt, ws, d)
        n += self._agent_forward(bt, ws, d, plan, early, heads=not fused.heads)
        n_mix, bptt = self._mixer_stage(bt, ws, d, fused)
        return n + n_mix + self._agent_backward(bt, ws, d, early, dhext_ready=fused.dhext, **bptt)

    def _agent_forward(self, bt, ws, d, plan, early, heads):
        """Every unroll of `plan` in one launch; `heads`: they also evaluate q = fc2(h) into ws["q"]."""
        (pe, stride), (pt, t_stride) = self._agent_structs(self._flat), self._agent_structs(self._tflat)
        if t_stride != stride:          # one stride per call: _pack lays both buffers' agents out alike
            raise ValueError(f"target agent stride {t_stride} differs from the eval stride {stride}")
        sep, last_action, agent_id = self._separated, int(self.args.last_action), int(self.args.reuse_network)
        continued = {u.h0_from for u in plan}
        arr = (L.UnrollStream * len(plan))()
        for i, u in enumerate(plan):
            s = arr[i]
            # an unroll that another one continues from runs to L (the reference carries the hidden state through the padded
            # steps, q_learner.py:96,110); stream 1, the target unroll, computes the BPTT's row order
            cut = early and i not in continued
            s.ep_len = ws["ep_len"].data_ptr() if cut else None
            s.padded = bt["padded"].data_ptr() if cut else None
            s.row_order = ws["row_order"][i].data_ptr() if cut else None
            s.row_order_bwd = ws["row_order"][3].data_ptr() if (early and i == 1) else None
            s.obs, s.onehot, s.shift_onehot, s.full_input = bt[u.obs].data_ptr(), bt["u_onehot"].data_ptr(), u.shift, 0
            s.h0_from, s.h0, s.params = u.h0_from, None, pt if u.target else pe
            s.q = ws["q"][i].data_ptr() if heads else None
            s.hidden, s.h_last = ws["hidden"][i].data_ptr(), ws["h_last"][i].data_ptr()
            s.x, s.gi = ws["x"][i].data_ptr(), ws["gi"][i].data_ptr()
            s.gates = ws["gates"].data_ptr() if u.keep else None
            s.w_ih_t = ws["w_ih_t"].data_ptr() if u.keep and not sep else None    # W_ih^T for the backward's data gradient
            s.agent_stride, s.last_action, s.agent_id, s.input_flags = stride, last_action, agent_id, int(not sep)
        L.call("marl_agent_unroll_fwd", C.byref(d), arr, len(plan), L.stream_ptr())
        # + episode lengths and row orders, launched by marl_agent_unroll_fwd beside the input layers
        return (3 if heads else 2) * len(plan) + 1 + (2 if early else 0)

    def _agent_backward(self, bt, ws, d, early, dhidden=None, dhext_ready=False, join=None):
        """BPTT through stream 0 (which kept its gates) from ws["dq"] and `dhidden`.  `dhext_ready`: the mixing kernel wrote
        dq . fc2_w into ws["dhext"].  `join`: a side stream with work beside the BPTT, waited for after it."""
        bw = L.UnrollBwd()
        bw.obs, bw.onehot, bw.shift_onehot, bw.full_input = bt["o"].data_ptr(), bt["u_onehot"].data_ptr(), 1, 0
        bw.params, bw.agent_stride = self._agent_structs(self._flat)
        bw.last_action, bw.agent_id = int(self.args.last_action), int(self.args.reuse_network)
        bw.input_flags = int(not self._separated)          # the shared network's input follows the same two switches
        bw.hidden, bw.x, bw.gates = ws["hidden"][0].data_ptr(), ws["x"][0].data_ptr(), ws["gates"].data_ptr()
        bw.h0, bw.dq, bw.dhidden = None, ws["dq"].data_ptr(), dhidden
        bw.dhext, bw.dgi, bw.dgh, bw.dx = (ws[k].data_ptr() for k in ("dhext", "dgi", "dgh", "dx"))
        bw.dh0 = None
        bw.dhext_ready = int(dhext_ready)
        bw.w_ih_t = None if self._separated else ws["w_ih_t"].data_ptr()
        bw.ep_len = ws["ep_len"].data_ptr() if early else None
        bw.row_order = ws["row_order"][3].data_ptr() if early else None
        bw.grads = self._agent_structs(self._flat, grad=True)[0]
        L.call("marl_agent_unroll_bwd", C.byref(d), C.byref(bw), L.stream_ptr())
        if join is not None:
            th.cuda.current_stream().wait_stream(join)
        return 7 - int(dhext_ready)

    def _mixer_prologue(self, bt, ws, d):
        """Mixer work that does not wait for the agent unrolls, issued ahead of them; returns its launches."""
        if self.args.alg != "qmix":
            return 0
        # QMIX: the hyper-networks only read the states: run them beside the (latency-bound) agent unrolls
        a, M = self.args, d.B * d.L
        (p, p2), (pt, pt2) = self._qmix_structs(self._flat), self._qmix_structs(self._tflat)
        side = self._side_streams(1)[0]
        side.wait_stream(th.cuda.current_stream())
        with th.cuda.stream(side):
            sp = L.stream_ptr()
            if p2 is not None:
                L.call("marl_qmix_hyper2_fwd", M, a.n_agents, a.state_shape, C.byref(p2), bt["s"].data_ptr(),
                       ws["hh"].data_ptr(), ws["hy"].data_ptr(), sp)
                L.call("marl_qmix_hyper2_fwd", M, a.n_agents, a.state_shape, C.byref(pt2), bt["s_next"].data_ptr(),
                       ws["hh_t"].data_ptr(), ws["hy_t"].data_ptr(), sp)
                return 2 * 5
            L.call("marl_qmix_hyper_fwd", M, a.n_agents, a.state_shape, C.byref(p), bt["s"].data_ptr(), ws["hy"].data_ptr(), sp)
            L.call("marl_qmix_hyper_fwd", M, a.n_agents, a.state_shape, C.byref(pt), bt["s_next"].data_ptr(),
                   ws["hy_t"].data_ptr(), sp)
            return 2

    def _mixer_stage(self, bt, ws, d, fused):
        """Selection, mixers, TD loss and their gradient down to ws["dq"]; returns (launches, options of _agent_backward)."""
        stage = {"vdn": self._vdn_stage, "qmix": self._qmix_stage, "qplex": self._qplex_stage}[self.args.alg]
        return stage(bt, ws, d, fused)

    def _select(self, bt, ws, d, fused):
        """Chosen and target agent Q-values: in the VDN / QMIX mixing kernel, or one marl_q_select.  Returns (launches,
        the mixing kernel's trailing arguments)."""
        a, double_q = self.args, bool(self.args.double_q)
        qplex = a.alg == "qplex"
        n, sel = 0, None
        fc2_w = self._flat.ptr("agent.fc2.weight") if (fused.heads or fused.dhext) else None
        if fused.select:
            sel = L.SelectFused()
            sel.q_evals, sel.q_targets = ws["q"][0].data_ptr(), ws["q"][1].data_ptr()
            sel.q_evals_next = ws["q"][2].data_ptr() if double_q else None
            sel.avail_u_next, sel.a_star = bt["avail_u_next"].data_ptr(), ws["a_star"].data_ptr()
            if fused.heads:
                sel.hidden_evals, sel.hidden_targets = ws["hidden"][0].data_ptr(), ws["hidden"][1].data_ptr()
                sel.hidden_evals_next = ws["hidden"][2].data_ptr() if double_q else None
                sel.fc2_w, sel.fc2_b = fc2_w, self._flat.ptr("agent.fc2.bias")
                sel.fc2_w_target, sel.fc2_b_target = self._tflat.ptr("agent.fc2.weight"), self._tflat.ptr("agent.fc2.bias")
        else:
            L.call("marl_q_select", C.byref(d), ws["q"][0].data_ptr(), bt["u"].data_ptr(),
                   ws["q"][2].data_ptr() if double_q else None, ws["q"][1].data_ptr(), bt["avail_u_next"].data_ptr(),
                   bt["avail_u"].data_ptr() if qplex else None, ws["q_chosen"].data_ptr(), ws["a_star"].data_ptr(),
                   ws["q_tc"].data_ptr(), ws["max_q"].data_ptr() if qplex else None,
                   ws["qt_max"].data_ptr() if qplex else None, ws["oh_star"].data_ptr() if qplex else None, L.stream_ptr())
            n = 1
        return n, (fc2_w if fused.dhext else None, ws["dhext"].data_ptr() if fused.dhext else None,
                   C.byref(sel) if fused.select else None)

    def _vdn_stage(self, bt, ws, d, fused):
        n, fused_tail = self._select(bt, ws, d, fused)
        L.call("marl_vdn_td_fwd_bwd", C.byref(d), ws["q_chosen"].data_ptr(), ws["q_tc"].data_ptr(), bt["u"].data_ptr(),
               bt["r"].data_ptr(), bt["terminated"].data_ptr(), bt["padded"].data_ptr(), float(self.gamma),
               ws["q_tot"].data_ptr(), ws["q_tot_t"].data_ptr(), ws["dq"].data_ptr(), self._flat.tail.data_ptr(), *fused_tail,
               L.stream_ptr())
        return n + 1, {}

    def _qmix_structs(self, flat, grad=False):
        """(mixing kernel, two-layer hyper-networks or None) structs of the QMIX mixer in `flat` or its gradient."""
        addr = flat.addrs("mixer.", flat.grad if grad else None)
        if not getattr(self.args, "two_hyper_layers", False):
            return qmix_struct(addr, L.QmixGrads if grad else L.QmixParams), None
        if grad:
            return qmix_tail_struct(addr, L.QmixGrads), qmix2_struct(addr, None, L.QmixHyper2Grads)
        return qmix_tail_struct(addr), qmix2_struct(addr, self.args.hyper_hidden_dim)

    def _qmix_stage(self, bt, ws, d, fused):
        a, M, sp = self.args, d.B * d.L, L.stream_ptr()
        (p, p2), (pt, _), (g, g2) = (self._qmix_structs(self._flat), self._qmix_structs(self._tflat),
                                     self._qmix_structs(self._flat, grad=True))
        n, fused_tail = self._select(bt, ws, d, fused)
        cur, side = th.cuda.current_stream(), self._side_streams(1)[0]
        cur.wait_stream(side)
        L.call("marl_qmix_td_fwd_bwd", C.byref(d), C.byref(p), C.byref(pt), bt["s"].data_ptr(), bt["s_next"].data_ptr(),
               ws["q_chosen"].data_ptr(), ws["q_tc"].data_ptr(), bt["u"].data_ptr(), bt["r"].data_ptr(),
               bt["terminated"].data_ptr(), bt["padded"].data_ptr(), float(self.gamma), ws["hy"].data_ptr(),
               ws["hy_t"].data_ptr(), ws["dhy"].data_ptr(), ws["q_tot"].data_ptr(), ws["q_tot_t"].data_ptr(),
               ws["dq"].data_ptr(), C.byref(g), self._flat.tail.data_ptr(), 3, *fused_tail, sp)
        # the hyper-network weight gradient runs beside the BPTT (whose kernel is launched at a higher priority)
        side.wait_stream(cur)
        with th.cuda.stream(side):
            if p2 is not None:
                L.call("marl_qmix_hyper2_bwd", M, a.n_agents, a.state_shape, C.byref(p2), bt["s"].data_ptr(),
                       ws["hh"].data_ptr(), ws["dhy"].data_ptr(), ws["dhh"].data_ptr(), C.byref(g2), L.stream_ptr())
                n += 7
            else:
                L.call("marl_qmix_hyper_wgrad", M, a.n_agents, a.state_shape, bt["s"].data_ptr(), ws["dhy"].data_ptr(),
                       C.byref(g), L.stream_ptr())
                n += 1
        return n + 1, dict(join=side)

    def _qplex_stage(self, bt, ws, d, fused):
        from ..network.qplex import qplex_struct, qplex_dims, ws_struct
        a, M, sp = self.args, d.B * d.L, L.stream_ptr()
        n, _ = self._select(bt, ws, d, fused)
        qd, K, nl = qplex_dims(a), a.num_kernel, int(getattr(a, "adv_hypernet_layers", 1))
        p = qplex_struct(self._flat.addrs("mixer.").__getitem__, K, layers=nl)
        ptg = qplex_struct(self._tflat.addrs("mixer.").__getitem__, K, layers=nl)
        g = qplex_struct(self._flat.addrs("mixer.", self._flat.grad).__getitem__, K, L.QplexGrads, layers=nl)
        wse, wst, dws = ws_struct(ws["qp"]), ws_struct(ws["qp_t"]), ws_struct(ws["dqp"])
        # q_tot = v_tot + a_tot (q_learner.py:120-135); target likewise with the eval net's argmax (:138-158)
        # the target mixer only shares the selection's outputs with the eval mixer: its chain of products runs beside it
        cur, side = th.cuda.current_stream(), self._side_streams(1)[0]
        side.wait_stream(cur)
        with th.cuda.stream(side):
            if a.double_q:
                L.call("marl_qplex_fwd", M, C.byref(qd), C.byref(ptg), ws["q_tc"].data_ptr(), bt["s_next"].data_ptr(),
                       ws["oh_star"].data_ptr(), ws["qt_max"].data_ptr(), C.byref(wst), None, None,
                       ws["q_tot_t"].data_ptr(), L.stream_ptr())
                n += 7
            else:
                L.call("marl_qplex_fwd", M, C.byref(qd), C.byref(ptg), ws["q_tc"].data_ptr(), bt["s_next"].data_ptr(),
                       None, None, C.byref(wst), ws["q_tot_t"].data_ptr(), None, None, L.stream_ptr())
                n += 2
        L.call("marl_qplex_fwd", M, C.byref(qd), C.byref(p), ws["q_chosen"].data_ptr(), bt["s"].data_ptr(),
               bt["u_onehot"].data_ptr(), ws["max_q"].data_ptr(), C.byref(wse), None, None, ws["q_tot"].data_ptr(), sp)
        n += 7
        cur.wait_stream(side)
        L.call("marl_td_loss", M, ws["q_tot"].data_ptr(), ws["q_tot_t"].data_ptr(), bt["r"].data_ptr(),
               bt["terminated"].data_ptr(), bt["padded"].data_ptr(), float(self.gamma), ws["dq_tot"].data_ptr(),
               self._flat.tail.data_ptr(), sp)
        L.call("marl_qplex_bwd", M, C.byref(qd), C.byref(p), ws["q_chosen"].data_ptr(), bt["s"].data_ptr(),
               bt["u_onehot"].data_ptr(), ws["max_q"].data_ptr(), C.byref(wse), ws["dq_tot"].data_ptr(),
               ws["dq_tot"].data_ptr(), C.byref(dws), ws["dq_small"].data_ptr(), C.byref(g), sp)
        n += 1 + 12
        L.call("marl_scatter_dq", C.byref(d), ws["dq_small"].data_ptr(), bt["u"].data_ptr(), ws["dq"].data_ptr(), sp)
        return n + 1, {}

    def _launch_optimizer(self):
        a, fl, opt, sp = self.args, self._flat, self.optimizer, L.stream_ptr()
        if self._peer is not None:
            adam = opt.kind != "RMS"
            L.call("marl_clip_step_peer", int(adam), fl.data.data_ptr(), fl.grad.data_ptr(),
                   (opt.exp_avg if adam else opt.square_avg).data_ptr(), opt.exp_avg_sq.data_ptr() if adam else None,
                   fl.numel, float(a.grad_norm_clip), float(self.lr), 0.9 if adam else 0.99, 0.999 if adam else 0.0, 1e-8,
                   opt.step_counter.data_ptr() if adam else None, self._loss_host.data_ptr(), C.byref(self._peer.struct), sp)
            return 1
        if opt.kind == "RMS":
            L.call("marl_clip_rmsprop_step", fl.data.data_ptr(), fl.grad.data_ptr(), opt.square_avg.data_ptr(), fl.numel,
                   fl.tail.data_ptr(), float(a.grad_norm_clip), float(self.lr), 0.99, 1e-8, self._partials.data_ptr(),
                   self._loss_host.data_ptr(), sp)
        else:
            L.call("marl_clip_adam_step", fl.data.data_ptr(), fl.grad.data_ptr(), opt.exp_avg.data_ptr(),
                   opt.exp_avg_sq.data_ptr(), fl.numel, fl.tail.data_ptr(), float(a.grad_norm_clip), float(self.lr),
                   0.9, 0.999, 1e-8, 0, opt.step_counter.data_ptr(), self._partials.data_ptr(),
                   self._loss_host.data_ptr(), sp)
        return 1 if fl.numel <= (1 << 18) else 2      # one cluster launch up to 2^18 parameters (csrc/optim.cu)

    def _device_step(self, bt, ws, B, Lq):
        if self._dist is not None and self._peer is None:
            n = self._launch_forward_backward(bt, ws, B, Lq)
            dist, group = self._dist
            allreduce_flat(self._flat.grad_full, dist, group)
            return n + self._launch_optimizer()
        return self._launch_forward_backward(bt, ws, B, Lq) + self._launch_optimizer()

    def _run(self, bt, ws, B, Lq):
        if not self._use_graph:
            self.launches_per_step = self._device_step(bt, ws, B, Lq)
            return
        key, self._graph_key = self._graph_key, None
        if key is None:
            key = (B, Lq) + tuple(bt[k].data_ptr() for k in BATCH_KEYS)
        entry = self._graphs.get(key)
        if entry is None or isinstance(entry, int):
            # the first calls with a shape run eagerly (lazy CUDA/NCCL init must not happen in capture).  A graph is only
            # captured at the third sighting: replay batches come with many different max_episode_len values, most of
            # them rare, and a capture (~tens of ms) is only worth it for the lengths that keep coming back
            self.launches_per_step = self._device_step(bt, ws, B, Lq)
            seen = (entry or 0) + 1
            self._graphs[key] = "warm" if seen >= self._capture_after else seen
            return
        if entry == "warm":
            if self._dist is None or self._peer is not None:
                g = th.cuda.CUDAGraph()
                with th.cuda.graph(g):
                    self._device_step(bt, ws, B, Lq)
                entry = (g,)
            else:
                # two graphs around the NCCL call: capturing torch.distributed's all-reduce inside the step graph was
                # tried on 2 x B200 and hung (test and bench both ran into their time limits), so the
                # collective stays an ordinary stream-ordered launch between them
                g1, g2 = th.cuda.CUDAGraph(), th.cuda.CUDAGraph()
                with th.cuda.graph(g1):
                    self._launch_forward_backward(bt, ws, B, Lq)
                with th.cuda.graph(g2):
                    self._launch_optimizer()
                entry = (g1, g2)
            self._graphs[key] = entry
        if len(entry) == 1:
            entry[0].replay()
        else:
            dist, group = self._dist
            entry[0].replay()
            allreduce_flat(self._flat.grad_full, dist, group)
            entry[1].replay()

    # ---- reference surface: the train step -------------------------------------------------------------
    def train(self, batch, train_step, episode_num=None):
        """One learner step; returns the loss as a Python float (q_learner.py:68-179).

        `batch`: the ReplayBuffer dict (numpy float64, host) or a dict of CUDA tensors in the device
        layout.  pymarl-style ``train(batch, t_env, episode_num)`` is accepted; the second argument
        drives the target sync exactly like the reference's ``train_step``."""
        if self._dev.type != "cuda":
            raise L.MarlLibraryError("QLearner.train needs a CUDA device: marl_b200 has no CPU path")
        if getattr(self.args, "train_through_modules", False):
            return self._train_modules(batch, train_step)
        self._graph_key = None
        if isinstance(batch, DeviceEpisodeBatch):
            bt, B, Lq, _ = self._stage_replay_batch(batch)
            ws = self._workspace(B, Lq)
        elif th.is_tensor(batch["o"]) and batch["o"].is_cuda:
            bt, B, Lq, _ = self._stage_device_batch(batch)
            ws = self._workspace(B, Lq)
        else:
            bt, B, Lq, _ = self._stage_host_batch(batch)
            ws = self._workspace(B, Lq)
        self.max_episode_len = Lq
        self._run(bt, ws, B, Lq)
        if train_step > 0 and train_step % self.args.target_update_cycle == 0:
            self._update_targets()
        th.cuda.current_stream().synchronize()
        # hidden states as the reference leaves them ([B*N, H], q_learner.py:96-110; [B, N, H] for SeparatedMAC): those of each
        # net's last unroll  (an nn.Module attribute store costs ~1.5 us: skipped while the controller already holds this working
        # set's tensors)
        last = {u.target: h for u, h in zip(self._agent_plan(B, Lq)[0], ws["h_last_sep" if self._separated else "h_last"])}
        he, ht = last[False], last[True]
        if self.eval_net.hidden_states is not he:
            self.eval_net.hidden_states = he
        if self.target_net.hidden_states is not ht:
            self.target_net.hidden_states = ht
        if self._peer is not None and float(self._loss_host[0]) != float(self._loss_host[0]) and int(self._peer.state[1]):
            raise RuntimeError("marl_clip_step_peer: a data-parallel peer did not reach the gradient exchange in time")
        self.last = dict(B=B, L=Lq, ws=ws, batch=bt, grad_norm=float(self._loss_host[1]))
        return float(self._loss_host[0])

    # ---- the same step through the drop-in MODULE surface (autograd over the library's kernels) -------------------------
    def _train_modules(self, batch, train_step):
        """q_learner.py:68-179 written against the controller / mixer modules: every unroll and every mixer call is a
        libmarl_b200 kernel sequence behind a torch.autograd.Function, the gather / mask / TD arithmetic between them is
        torch on the GPU, clip + RMSprop/Adam is the flat optimiser kernel.  ``args.train_through_modules`` selects it: an
        independent second implementation of the fused step for the tests."""
        a, dev = self.args, self._dev
        if isinstance(batch, DeviceEpisodeBatch):
            Lq = batch.max_episode_len
        else:
            Lq = host_max_episode_len(_to_numpy(batch["terminated"]), a.episode_limit)
        b = {}
        for k in BATCH_KEYS:
            t = batch[k]
            t = th.as_tensor(_to_numpy(t)) if not th.is_tensor(t) else t
            b[k] = t[:, :Lq].to(device=dev, dtype=th.int64 if k == "u" else th.float32)
        B = b["o"].shape[0]
        s, u, r, s_next, avail_u, avail_u_next, terminated = (b[k] for k in ("s", "u", "r", "s_next", "avail_u", "avail_u_next",
                                                                               "terminated"))
        u = u.reshape(B, Lq, a.n_agents, 1)
        r, terminated = r.reshape(B, Lq, 1), terminated.reshape(B, Lq, 1)
        mask = 1 - b["padded"].reshape(B, Lq, 1)
        self.eval_net.init_hidden(B)
        q_evals, _ = self.eval_net.get_current_q_values(b, Lq)
        q_chosen = th.gather(q_evals, dim=3, index=u).squeeze(3)
        with th.no_grad():
            self.target_net.init_hidden(B)
            q_targets, _ = self.target_net.get_next_q_values(b, Lq)
            q_targets = q_targets.clone()
            q_targets[avail_u_next == 0.0] = -9999999
            if a.double_q:
                q_next = self.eval_net.get_next_q_values(b, Lq)[0].clone()        # hidden carried (q_learner.py:110)
                q_next[avail_u_next == 0] = -9999999
                a_star = th.argmax(q_next, dim=3, keepdim=True)
                q_tc = th.gather(q_targets, 3, a_star).squeeze(3)
            else:
                a_star = None
                q_tc = q_targets.max(dim=3)[0]
        if a.alg == "qplex":
            v_tot = self.mixer(q_chosen, s, is_v=True)
            qd = q_evals.detach().clone()
            qd[avail_u == 0] = -9999999
            a_tot = self.mixer(q_chosen, s, actions=b["u_onehot"], max_q_i=qd.max(dim=3)[0], is_v=False)
            q_tot = v_tot + a_tot
            with th.no_grad():
                if a.double_q:
                    oh = th.zeros_like(q_targets).scatter_(3, a_star, 1)
                    tv = self.target_mixer(q_tc, s_next, is_v=True)
                    ta = self.target_mixer(q_tc, s_next, actions=oh, max_q_i=q_targets.max(dim=3)[0], is_v=False)
                    q_tot_t = tv + ta
                else:
                    q_tot_t = self.target_mixer(q_tc, s_next, is_v=True)
        else:
            q_tot = self.mixer(q_chosen, s)
            with th.no_grad():
                q_tot_t = self.target_mixer(q_tc, s_next)
        targets = r + self.gamma * q_tot_t * (1 - terminated)
        masked = mask * (q_tot - targets.detach())
        loss = (masked ** 2).sum() / mask.sum()
        self._flat.grad_full.zero_()
        self._flat.rebind_grads()
        loss.backward()
        # the optimiser kernel expects the gradient of the UN-normalised sum and (loss_sum, mask_sum): hand it the
        # normalised gradient with mask_sum = 1
        self._flat.tail.copy_(th.stack([loss.detach(), th.ones((), device=dev)]))
        self._launch_optimizer()
        if train_step > 0 and train_step % a.target_update_cycle == 0:
            self._update_targets()
        th.cuda.current_stream().synchronize()
        self.max_episode_len = Lq
        self.last = dict(B=B, L=Lq, q_evals=q_evals.detach(), q_tot=q_tot.detach(), a_star=a_star,
                         grad_norm=float(self._loss_host[1]))
        return float(self._loss_host[0])

    def _update_targets(self):
        # targets mirror the leading [agent | mixer] region of the flat buffer: one D2D copy
        self._tflat.data.copy_(self._flat.data[:self._tflat.numel])

    # ---- checkpoints -------------------------------------------------------------------------------------
    def save_models(self, train_step):
        num = str(train_step // self.args.save_cycle)
        if not os.path.exists(self.model_dir):
            os.makedirs(self.model_dir)
        self.eval_net.save_models(self.model_dir + '/' + num + '_rnn_net_params.pkl')
        th.save(self.mixer.state_dict(), self.model_dir + '/' + num + '_mixer_net_params.pkl')

    def load_models(self):
        if os.path.exists(self.model_dir + '/rnn_net_params.pkl'):
            path_rnn = self.model_dir + '/rnn_net_params.pkl'
            path_mix = self.model_dir + '/mixer_net_params.pkl'
            self.eval_net.load_models(path_rnn)
            self.mixer.load_state_dict(th.load(path_mix, map_location=self._dev))
            print('Successfully load the model: {} and {}'.format(path_rnn, path_mix))
        else:
            raise Exception("No model!")

    # ---- matrix-game tables (q_learner.py:211-262) ----------------------------------------------------------
    def get_q_and_q_tot_table(self):
        """3x3 Q_tot table and the two per-agent Q rows at o = s = 1 (matrix game only)."""
        with th.no_grad():
            dev = self._dev
            one = {'o': th.ones(1, 1, 2, 1, device=dev), 's': th.ones(1, 1, 1, device=dev),
                   'o_next': th.ones(1, 1, 2, 1, device=dev), 'u_onehot': th.zeros(1, 1, 2, 3, device=dev),
                   'avail_u': th.ones(1, 1, 2, 3, device=dev)}
            self.eval_net.init_hidden(episode_num=1)
            q_values, _ = self.eval_net.get_current_q_values(one, max_episode_len=1)     # (1,1,2,3)
            q_table_i = q_values[0, 0, 0].cpu().numpy()
            q_table_j = q_values[0, 0, 1].cpu().numpy()
            q_tot_table = np.zeros((3, 3))
            for i in range(3):
                for j in range(3):
                    chosen = th.stack((q_values[:, :, 0, i], q_values[:, :, 1, j]), dim=2)   # (1,1,2)
                    if self.args.alg == 'qplex':
                        v_tot = self.mixer(chosen, one['s'], is_v=True)
                        max_q = q_values.max(dim=3)[0]
                        oh = th.zeros_like(q_values)
                        oh[0, 0, 0, i] = 1
                        oh[0, 0, 1, j] = 1
                        a_tot = self.mixer(chosen, one['s'], actions=oh, max_q_i=max_q, is_v=False)
                        q_tot_table[i, j] = (v_tot + a_tot).item()
                    else:
                        q_tot_table[i, j] = self.mixer(chosen, one['s']).item()
            return q_tot_table, q_table_i, q_table_j


def separated_stride(flat, n_agents):
    """Distance in floats from agent n's parameter set to agent n+1's in a flat buffer packed agent after agent as
    ``agent.{n}.*`` (QLearner._pack).  ValueError unless it is the same positive multiple of 4 for every agent and every
    parameter: the library addresses agent n's set as agent 0's plus n strides."""
    off = flat.offsets
    names = [n[len("agent.0."):] for n in flat.names if n.startswith("agent.0.")]
    if n_agents > 1:
        stride = off["agent.1." + names[0]] - off["agent.0." + names[0]]
    else:
        end = max(off["agent.0." + k] + flat.view("agent.0." + k).numel() for k in names)
        stride = (end - off["agent.0." + names[0]] + 3) // 4 * 4
    for i in range(n_agents):
        for k in names:
            if off.get(f"agent.{i}.{k}") != off["agent.0." + k] + i * stride:
                raise ValueError(f"agent parameter sets are not evenly spaced in the flat buffer (agent.{i}.{k})")
    if stride <= 0 or stride % 4:
        raise ValueError(f"agent parameter stride {stride} is not a positive multiple of 4 floats")
    return stride


def _to_numpy(x):
    if isinstance(x, np.ndarray):
        return x
    if th.is_tensor(x):
        return x.detach().cpu().numpy()
    return np.asarray(x)


def _episode_struct(bt):
    e = L.EpisodeF32()
    for k in L.EPISODE_KEYS:
        setattr(e, k, bt[k].data_ptr())
    return e
