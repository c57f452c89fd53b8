"""QTRAN-base learner on sm_100a kernels, drop-in for ``algorithm/qtran_learner.py:10-272``.

Same surface as the reference's ``QTRANLearner`` (``train(batch, train_step) -> float`` with
L_td + lambda_opt L_opt + lambda_nopt L_nopt, ``mixer`` / ``target_mixer`` / ``v`` / ``q_sum_mixer``,
checkpoints with ``_v_net_params.pkl``); the step is the fixed launch sequence

    2 agent unrolls (eval/o with saved gates, target/o_next)     qtran_learner.py:95-101
    greedy actions + one-hots                                    :103-114
    Q(s, h, u), Q_target(s', h', a*_target), Q(s, h, a*_eval), V(s, h)        :165-200
    three losses and their gradients                             :116-152
    backward through Q and V into d(hidden), BPTT with d(q) and d(hidden)     :155
    clip + optimiser over agent + mixer + V (q_sum_mixer never receives a gradient, :37-38,131-132)

``qtran_alt`` is constructible in the reference but its forward is broken there (SURVEY.md section 2); it
raises here.
"""
from __future__ import annotations

import ctypes as C
import os

import torch as th

from .. import _lib as L
from ..network.mixer import QMixMixer
from ..network.qtran import QtranQBase, QtranV, net_struct, net_workspace, net_ws_struct
from .q_learner import QLearner, _EVAL_O, _TARGET_O_NEXT



class QTRANLearner(QLearner):
    def _build_extra(self, args):
        self.v = QtranV(args)                       # qtran_learner.py:34-35
        self.params += list(self.v.parameters())
        self.q_sum_mixer = QMixMixer(args)          # :37-38 -- handed to the optimiser by the reference, never used
        self.params += list(self.q_sum_mixer.parameters())

    def _make_mixer(self, args):
        if args.alg == 'qtran_base':
            return QtranQBase(args)
        if args.alg == 'qtran_alt':
            raise NotImplementedError("qtran_alt: the reference's own forward is inconsistent (mixer.py:320,349)")
        raise ValueError("Mixer {} not recognised.".format(args.alg))

    def _extra_groups(self):
        return [("v.", self.v)]

    def _workspace(self, B, Lq):
        fresh = (B, Lq) not in self._ws
        ws = super()._workspace(B, Lq)
        if fresh:
            a, dev = self.args, self._dev
            N, A, M, H = a.n_agents, a.n_actions, B * Lq, a.rnn_hidden_dim
            f = lambda *shape: th.empty(*shape, dtype=th.float32, device=dev)
            D, qh = H + A, a.qtran_hidden_dim
            ws.update(oh_e=f(B, Lq, N, A), oh_t=f(B, Lq, N, A), opt_e=th.empty(B, Lq, N, dtype=th.int64, device=dev),
                      q_max=f(B, Lq, N), q_taken=f(B, Lq, N), jq=f(M), jq_t=f(M), jq_hat=f(M), vv=f(M), d_jq=f(M),
                      d_v=f(M), dhid=f(B * Lq * N, H), parts=th.zeros(3, dtype=th.float32, device=dev),
                      nq=net_workspace(M, N, D, qh, dev), nqt=net_workspace(M, N, D, qh, dev),
                      nqh=net_workspace(M, N, D, qh, dev), nv=net_workspace(M, N, H, qh, dev),
                      dnq=net_workspace(M, N, D, qh, dev), dnv=net_workspace(M, N, H, qh, dev))
        return ws

    def _agent_plan(self, B, Lq):
        return (_EVAL_O, _TARGET_O_NEXT), False            # no double-Q unroll (qtran_learner.py:95-101), no early exit

    def _mixer_prologue(self, bt, ws, d):
        ws["parts"].zero_()
        return 1

    def _mixer_stage(self, bt, ws, d, fused):
        a, sp = self.args, L.stream_ptr()
        fl, tfl = self._flat, self._tflat
        L.call("marl_qtran_select", C.byref(d), ws["q"][0].data_ptr(), ws["q"][1].data_ptr(), bt["avail_u"].data_ptr(),
               bt["avail_u_next"].data_ptr(), bt["u"].data_ptr(), ws["oh_e"].data_ptr(), ws["oh_t"].data_ptr(),
               ws["opt_e"].data_ptr(), ws["q_max"].data_ptr(), ws["q_taken"].data_ptr(), sp)
        n = 1
        M, N, S, A, qh = d.B * d.L, a.n_agents, a.state_shape, a.n_actions, a.qtran_hidden_dim
        # net_struct takes the addresses in parameter order, the order the flat buffers list them in
        H = a.rnn_hidden_dim
        pq = net_struct(fl.addrs("mixer.").values(), hidden=H)
        pqt = net_struct(tfl.addrs("mixer.").values(), hidden=H)
        pv = net_struct(fl.addrs("v.").values(), hidden=H)
        gq = net_struct(fl.addrs("mixer.", fl.grad).values(), L.QtranNetGrads)
        gv = net_struct(fl.addrs("v.", fl.grad).values(), L.QtranNetGrads)
        hid_e, hid_t = ws["hidden"][0].data_ptr(), ws["hidden"][1].data_ptr()
        wq, wqt, wqh, wv = (net_ws_struct(ws[k]) for k in ("nq", "nqt", "nqh", "nv"))
        dwq, dwv = net_ws_struct(ws["dnq"]), net_ws_struct(ws["dnv"])
        # get_qtran (qtran_learner.py:165-200): the four network evaluations (joint Q at the taken actions, target joint Q, joint Q at
        # the greedy actions, V) only share their inputs -- chains of small, latency-bound products: three of them run on side
        # streams beside the first
        cur, sides = th.cuda.current_stream(), self._side_streams(3)
        calls = (
            (pq, bt["s"].data_ptr(), hid_e, bt["u_onehot"].data_ptr(), wq, ws["jq"], A),
            (pqt, bt["s_next"].data_ptr(), hid_t, ws["oh_t"].data_ptr(), wqt, ws["jq_t"], A),
            (pq, bt["s"].data_ptr(), hid_e, ws["oh_e"].data_ptr(), wqh, ws["jq_hat"], A),
            (pv, bt["s"].data_ptr(), hid_e, None, wv, ws["vv"], 0),
        )
        for k, (pp, st_, hid, act, w_, out, a_enc) in enumerate(calls):
            if k == 0:
                L.call("marl_qtran_net_fwd", M, N, S, a_enc, qh, C.byref(pp), st_, hid, act, C.byref(w_), out.data_ptr(), sp)
                continue
            side = sides[k - 1]
            side.wait_stream(cur)
            with th.cuda.stream(side):
                L.call("marl_qtran_net_fwd", M, N, S, a_enc, qh, C.byref(pp), st_, hid, act, C.byref(w_), out.data_ptr(), L.stream_ptr())
        for side in sides:
            cur.wait_stream(side)
        n += 6 * len(calls)
        L.call("marl_qtran_losses_fwd_bwd", C.byref(d), ws["jq"].data_ptr(), ws["jq_t"].data_ptr(), ws["jq_hat"].data_ptr(),
               ws["vv"].data_ptr(), ws["q_max"].data_ptr(), ws["q_taken"].data_ptr(), ws["opt_e"].data_ptr(),
               bt["u"].data_ptr(), bt["avail_u"].data_ptr(), bt["r"].data_ptr(), bt["terminated"].data_ptr(),
               bt["padded"].data_ptr(), float(self.gamma), float(a.lambda_opt), float(a.lambda_nopt), ws["d_jq"].data_ptr(),
               ws["d_v"].data_ptr(), ws["dq"].data_ptr(), fl.tail.data_ptr(), ws["parts"].data_ptr(), sp)
        n += 1
        # (measured and dropped: V's backward on a side stream into its own dL/dhidden buffer, folded afterwards -- 2851 .. 2951 us
        # per step against 2883: the two chains' products already share the machine through the weight-gradient lane)
        L.call("marl_qtran_net_bwd", M, N, S, A, qh, C.byref(pq), bt["s"].data_ptr(), hid_e, bt["u_onehot"].data_ptr(),
               C.byref(wq), ws["d_jq"].data_ptr(), C.byref(dwq), ws["dhid"].data_ptr(), 0, C.byref(gq), sp)
        L.call("marl_qtran_net_bwd", M, N, S, 0, qh, C.byref(pv), bt["s"].data_ptr(), hid_e, None, C.byref(wv),
               ws["d_v"].data_ptr(), C.byref(dwv), ws["dhid"].data_ptr(), 1, C.byref(gv), sp)
        return n + 2 * 11, dict(dhidden=ws["dhid"].data_ptr())

    def save_models(self, train_step):
        num = str(train_step // self.args.save_cycle)
        if not os.path.exists(self.model_dir):
            os.makedirs(self.model_dir)
        self.eval_net.save_models(self.model_dir + '/' + num + '_rnn_net_params.pkl')
        th.save(self.mixer.state_dict(), self.model_dir + '/' + num + '_mixer_net_params.pkl')
        th.save(self.v.state_dict(), self.model_dir + '/' + num + '_v_net_params.pkl')

    def load_models(self):
        if os.path.exists(self.model_dir + '/rnn_net_params.pkl'):
            self.eval_net.load_models(self.model_dir + '/rnn_net_params.pkl')
            self.mixer.load_state_dict(th.load(self.model_dir + '/mixer_net_params.pkl', map_location=self._dev))
            self.v.load_state_dict(th.load(self.model_dir + '/v_net_params.pkl', map_location=self._dev))
        else:
            raise Exception("No model!")
