"""ctypes binding of libmarl_b200.so (the C ABI declared in include/marl_b200.h).

There is no CPU fallback: if the library is missing, or a kernel is called without a CUDA
device, the call raises.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MARL_B200_LIB") or os.path.join(_HERE, "lib", "libmarl_b200.so")   # override: kernel A/B builds

c_float_p = C.c_void_p   # device pointers travel as integers (tensor.data_ptr())
c_ptr = C.c_void_p


class Dims(C.Structure):
    _fields_ = [(k, C.c_int) for k in ("B", "L", "N", "A", "O", "S")]


EPISODE_KEYS = ("o", "s", "u", "r", "o_next", "s_next", "avail_u", "avail_u_next", "u_onehot", "padded", "terminated")


class EpisodeF32(C.Structure):
    _fields_ = [(k, c_ptr) for k in EPISODE_KEYS]


class EpisodeF64(C.Structure):
    _fields_ = [(k, c_ptr) for k in ("o", "u", "s", "r", "o_next", "s_next", "avail_u", "avail_u_next", "u_onehot",
                                     "padded", "terminated")] + [("u_is_int64", C.c_int)]


AGENT_KEYS = ("fc1_w", "fc1_b", "w_ih", "w_hh", "b_ih", "b_hh", "fc2_w", "fc2_b")


class AgentParams(C.Structure):
    _fields_ = [(k, c_ptr) for k in AGENT_KEYS]


class AgentGrads(C.Structure):
    _fields_ = [(k, c_ptr) for k in AGENT_KEYS]


class UnrollStream(C.Structure):
    _fields_ = [("obs", c_ptr), ("onehot", c_ptr), ("shift_onehot", C.c_int), ("full_input", C.c_int),
                ("h0_from", C.c_int), ("h0", c_ptr),
                ("params", AgentParams), ("q", c_ptr), ("hidden", c_ptr), ("h_last", c_ptr), ("x", c_ptr),
                ("gi", c_ptr), ("gates", c_ptr), ("w_ih_t", c_ptr), ("ep_len", c_ptr), ("padded", c_ptr),
                ("row_order", c_ptr), ("row_order_bwd", c_ptr), ("agent_stride", C.c_int), ("last_action", C.c_int),
                ("agent_id", C.c_int), ("input_flags", C.c_int)]


class UnrollBwd(C.Structure):
    _fields_ = [("obs", c_ptr), ("onehot", c_ptr), ("shift_onehot", C.c_int), ("full_input", C.c_int),
                ("params", AgentParams), ("hidden", c_ptr), ("x", c_ptr), ("gates", c_ptr), ("h0", c_ptr), ("dq", c_ptr),
                ("dhidden", c_ptr), ("dhext", c_ptr), ("dgi", c_ptr), ("dgh", c_ptr), ("dx", c_ptr), ("dh0", c_ptr),
                ("grads", AgentGrads), ("dhext_ready", C.c_int), ("w_ih_t", c_ptr), ("ep_len", c_ptr), ("row_order", c_ptr),
                ("agent_stride", C.c_int), ("last_action", C.c_int), ("agent_id", C.c_int), ("input_flags", C.c_int)]


class ActPhilox(C.Structure):      # include/marl_b200.h: marl_act_philox
    _fields_ = [("seed", C.c_ulonglong), ("episode_base", C.c_ulonglong), ("step", C.c_int), ("eps_table", c_ptr),
                ("eps_len", C.c_int)]


class PeerGroup(C.Structure):
    _fields_ = [("world", C.c_int), ("rank", C.c_int), ("grads", c_ptr * 8), ("flags", c_ptr * 8), ("epoch", c_ptr),
                ("error", c_ptr)]


class SelectFused(C.Structure):
    _fields_ = [(k, c_ptr) for k in ("q_evals", "q_evals_next", "q_targets", "avail_u_next", "a_star", "hidden_evals",
                                     "hidden_targets", "hidden_evals_next", "fc2_w", "fc2_b", "fc2_w_target",
                                     "fc2_b_target")]


class QmixParams(C.Structure):
    _fields_ = [(k, c_ptr) for k in ("wcat", "bcat", "wb2", "bb2")]


class QmixGrads(C.Structure):
    _fields_ = [(k, c_ptr) for k in ("wcat", "bcat", "wb2", "bb2")]


QMIX_HYPER2_FIELDS = ("w_in", "b_in", "w1_out", "b1_out", "w2_out", "b2_out", "w_b1", "b_b1", "w_b20", "b_b20")


class QmixHyper2(C.Structure):       # two_hyper_layers=True parameters (include/marl_b200.h: marl_qmix_hyper2)
    _fields_ = [(k, c_ptr) for k in QMIX_HYPER2_FIELDS] + [("hh", C.c_int)]


class QmixHyper2Grads(C.Structure):
    _fields_ = [(k, c_ptr) for k in QMIX_HYPER2_FIELDS]


class QplexDims(C.Structure):
    _fields_ = [(k, C.c_int) for k in ("N", "A", "S", "he", "ae", "K", "weighted_head", "is_minus_one", "layers")]


QPLEX_FIELDS = ("w1s", "b1s", "w1a", "b1a", "w2", "b2", "w3k", "b3k", "w3n", "b3n", "wfv", "bfv")


class QplexParams(C.Structure):
    _fields_ = [(k, c_ptr) for k in QPLEX_FIELDS]


class QplexGrads(C.Structure):
    _fields_ = [(k, c_ptr) for k in QPLEX_FIELDS]


class QplexWs(C.Structure):
    _fields_ = [(k, c_ptr) for k in ("h1", "h2", "o3", "wv")]


QTRAN_FIELDS = ("we1", "be1", "we2", "be2", "w0", "b0", "w2", "b2", "w4", "b4")


class QtranNetParams(C.Structure):
    _fields_ = [(k, c_ptr) for k in QTRAN_FIELDS]


class QtranNetGrads(C.Structure):
    _fields_ = [(k, c_ptr) for k in QTRAN_FIELDS]


class QtranNetWs(C.Structure):
    _fields_ = [(k, c_ptr) for k in ("e1", "es", "enc", "a1", "a2")]


_P = C.POINTER
_SIGNATURES = {
    "marl_version": ([], C.c_int),
    "marl_device_info": ([_P(C.c_int)] * 3, C.c_int),
    "marl_matrix_game_step": ([_P(C.c_double), c_ptr, C.c_int, C.c_longlong, C.c_float, _P(EpisodeF32), c_ptr, c_ptr], C.c_int),
    "marl_matrix_game_validate_actions": ([c_ptr, C.c_int, C.c_longlong, c_ptr, c_ptr], C.c_int),
    "marl_ingest_f64": ([_P(EpisodeF64), C.c_int, _P(Dims), _P(EpisodeF32), c_ptr], C.c_int),
    "marl_ingest_f32": ([_P(EpisodeF32), C.c_int, _P(Dims), _P(EpisodeF32), c_ptr], C.c_int),
    "marl_replay_gather_f32": ([_P(EpisodeF32), C.c_int, c_ptr, _P(Dims), _P(EpisodeF32), c_ptr], C.c_int),
    "marl_fma_probe": ([c_ptr, C.c_int, C.c_int, _P(C.c_double), c_ptr], C.c_int),
    "marl_agent_unroll_fwd": ([_P(Dims), _P(UnrollStream), C.c_int, c_ptr], C.c_int),
    "marl_agent_unroll_bwd": ([_P(Dims), _P(UnrollBwd), c_ptr], C.c_int),
    "marl_q_select": ([_P(Dims)] + [c_ptr] * 12 + [c_ptr], C.c_int),
    "marl_td_loss": ([C.c_int] + [c_ptr] * 5 + [C.c_float, c_ptr, c_ptr, c_ptr], C.c_int),
    "marl_vdn_td_fwd_bwd": ([_P(Dims)] + [c_ptr] * 6 + [C.c_float] + [c_ptr] * 4 + [c_ptr, c_ptr, _P(SelectFused), c_ptr],
                            C.c_int),
    "marl_qmix_fwd": ([C.c_int, C.c_int, C.c_int, _P(QmixParams), c_ptr, c_ptr, c_ptr, c_ptr, c_ptr], C.c_int),
    "marl_qmix_bwd": ([C.c_int, C.c_int, C.c_int, _P(QmixParams)] + [c_ptr] * 6 + [_P(QmixGrads), c_ptr], C.c_int),
    "marl_qmix_td_fwd_bwd": ([_P(Dims), _P(QmixParams), _P(QmixParams)] + [c_ptr] * 8 + [C.c_float] + [c_ptr] * 6
                             + [_P(QmixGrads), c_ptr, C.c_int, c_ptr, c_ptr, _P(SelectFused), c_ptr], C.c_int),
    "marl_peer_alloc": ([C.c_size_t, _P(c_ptr)], C.c_int),
    "marl_peer_free": ([c_ptr], C.c_int),
    "marl_peer_export": ([c_ptr, C.c_char_p], C.c_int),
    "marl_peer_open": ([C.c_char_p, _P(c_ptr)], C.c_int),
    "marl_peer_close": ([c_ptr], C.c_int),
    "marl_clip_step_peer": ([C.c_int, c_ptr, c_ptr, c_ptr, c_ptr, C.c_longlong] + [C.c_float] * 5
                            + [c_ptr, c_ptr, _P(PeerGroup), c_ptr], C.c_int),
    "marl_qmix_hyper_fwd": ([C.c_int, C.c_int, C.c_int, _P(QmixParams), c_ptr, c_ptr, c_ptr], C.c_int),
    "marl_qmix_hyper2_fwd": ([C.c_int, C.c_int, C.c_int, _P(QmixHyper2), c_ptr, c_ptr, c_ptr, c_ptr], C.c_int),
    "marl_qmix_hyper2_bwd": ([C.c_int, C.c_int, C.c_int, _P(QmixHyper2), c_ptr, c_ptr, c_ptr, c_ptr, _P(QmixHyper2Grads), c_ptr], C.c_int),
    "marl_qmix_mix_fwd": ([C.c_int, C.c_int, _P(QmixParams), c_ptr, c_ptr, c_ptr, c_ptr], C.c_int),
    "marl_qmix_mix_bwd": ([C.c_int, C.c_int, _P(QmixParams)] + [c_ptr] * 5 + [_P(QmixGrads), c_ptr], C.c_int),
    "marl_qmix_hyper_wgrad": ([C.c_int, C.c_int, C.c_int, c_ptr, c_ptr, _P(QmixGrads), c_ptr], C.c_int),
    "marl_qplex_fwd": ([C.c_int, _P(QplexDims), _P(QplexParams)] + [c_ptr] * 4 + [_P(QplexWs)] + [c_ptr] * 4, C.c_int),
    "marl_qplex_bwd": ([C.c_int, _P(QplexDims), _P(QplexParams)] + [c_ptr] * 4 + [_P(QplexWs), c_ptr, c_ptr, _P(QplexWs), c_ptr,
                       _P(QplexGrads), c_ptr], C.c_int),
    "marl_scatter_dq": ([_P(Dims), c_ptr, c_ptr, c_ptr, c_ptr], C.c_int),
    "marl_qtran_net_fwd": ([C.c_int] * 5 + [_P(QtranNetParams), c_ptr, c_ptr, c_ptr, _P(QtranNetWs), c_ptr, c_ptr], C.c_int),
    "marl_qtran_net_bwd": ([C.c_int] * 5 + [_P(QtranNetParams), c_ptr, c_ptr, c_ptr, _P(QtranNetWs), c_ptr, _P(QtranNetWs),
                           c_ptr, C.c_int, _P(QtranNetGrads), c_ptr], C.c_int),
    "marl_qtran_select": ([_P(Dims)] + [c_ptr] * 10 + [c_ptr], C.c_int),
    "marl_qtran_losses_fwd_bwd": ([_P(Dims)] + [c_ptr] * 12 + [C.c_float] * 3 + [c_ptr] * 5 + [c_ptr], C.c_int),
    "marl_epsgreedy_select": ([C.c_int, C.c_int] + [c_ptr] * 6 + [c_ptr], C.c_int),
    "marl_agent_act": ([C.c_int] * 4 + [_P(AgentParams)] + [c_ptr] * 9 + [C.c_double] + [c_ptr] * 5, C.c_int),
    "marl_agent_act_input": ([C.c_int] * 6 + [_P(AgentParams)] + [c_ptr] * 9 + [C.c_double] + [c_ptr] * 5, C.c_int),
    "marl_agent_act_separated": ([C.c_int] * 6 + [_P(AgentParams)] + [c_ptr] * 9 + [C.c_double] + [c_ptr] * 5, C.c_int),
    "marl_agent_act_philox": ([C.c_int] * 6 + [_P(AgentParams)] + [c_ptr] * 5 + [_P(ActPhilox), C.c_double] + [c_ptr] * 5,
                              C.c_int),
    "marl_agent_act_separated_philox": ([C.c_int] * 6 + [_P(AgentParams)] + [c_ptr] * 5 + [_P(ActPhilox), C.c_double]
                                        + [c_ptr] * 5, C.c_int),
    "marl_philox_uniforms": ([C.c_ulonglong, C.c_ulonglong, C.c_int, C.c_int, C.c_int, c_ptr, c_ptr], C.c_int),
    "marl_rollout_record": ([_P(Dims), C.c_int, _P(EpisodeF32)] + [c_ptr] * 12 + [c_ptr], C.c_int),
    "marl_select_fits": ([C.c_int] * 4, C.c_int),
    "marl_episode_lengths": ([c_ptr, C.c_int, C.c_int, c_ptr, c_ptr], C.c_int),
    "marl_set_scratch": ([c_ptr, C.c_size_t], C.c_int),
    "marl_tgemm_trace": ([C.c_int, c_ptr], C.c_int),
    "marl_tgemm_enable": ([C.c_int], C.c_int),
    "marl_set_deterministic": ([C.c_int], C.c_int),
    "marl_linear_fwd": ([c_ptr, C.c_int, c_ptr, C.c_int, c_ptr, c_ptr, C.c_int] + [C.c_int] * 4 + [c_ptr], C.c_int),
    "marl_linear_dgrad": ([c_ptr, C.c_int, c_ptr, C.c_int, c_ptr, C.c_int, c_ptr, C.c_int] + [C.c_int] * 3 + [c_ptr], C.c_int),
    "marl_linear_wgrad": ([c_ptr, C.c_int, c_ptr, C.c_int, c_ptr, C.c_int, c_ptr] + [C.c_int] * 3 + [c_ptr], C.c_int),
    "marl_optim_partials": ([], C.c_int),
    "marl_host_registered": ([c_ptr, C.c_size_t], C.c_int),
    "marl_host_registered_all": ([c_ptr, c_ptr, C.c_int], C.c_int),
    "marl_front_enable": ([C.c_int], C.c_int),
    "marl_spin_us": ([C.c_int, c_ptr], C.c_int),
    "marl_profile_enable": ([C.c_int], C.c_int),
    "marl_profile_collect": ([C.c_char_p, C.c_int], C.c_int),
    "marl_profile_timeline": ([C.c_char_p, C.c_int], C.c_int),
    "marl_clip_rmsprop_step": ([c_ptr, c_ptr, c_ptr, C.c_longlong, c_ptr] + [C.c_float] * 4 + [c_ptr, c_ptr, c_ptr], C.c_int),
    "marl_clip_adam_step": ([c_ptr] * 4 + [C.c_longlong, c_ptr] + [C.c_float] * 5 + [C.c_int, c_ptr, c_ptr, c_ptr, c_ptr], C.c_int),
}

_lib = None


class MarlLibraryError(RuntimeError):
    pass


def load():
    """Load (once) and return the ctypes handle; raises if the .so is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MarlLibraryError(
            f"{LIB_PATH} is missing: run `python -m marl_b200.build` (needs nvcc); marl_b200 has no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (argtypes, restype) in _SIGNATURES.items():
        fn = getattr(lib, name)     # AttributeError if the .so does not export a declared symbol
        fn.argtypes, fn.restype = argtypes, restype
    _lib = lib
    return lib


def exported_symbols():
    return sorted(_SIGNATURES)


def check(rc, what):
    if rc == 0:
        return
    if rc < 0:
        raise ValueError(f"{what}: invalid argument (MARL_EINVAL)")
    raise MarlLibraryError(f"{what}: CUDA error {rc}")


def require_cuda(t: torch.Tensor, name="tensor"):
    if not t.is_cuda:
        raise MarlLibraryError(f"{name} must live on a CUDA device: marl_b200 has no CPU path")
    return t


def ptr(t):
    """Device address of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr():
    return torch.cuda.current_stream().cuda_stream


_scratch = {}


def ensure_scratch(nbytes=None):
    """One process-wide device arena per GPU for the split weight-gradient partials (csrc/tgemm.cu); never freed, so
    captured CUDA graphs that baked its addresses stay valid for the life of the process."""
    dev = torch.cuda.current_device()
    if dev not in _scratch:
        nbytes = nbytes or int(os.environ.get("MARL_B200_SCRATCH_MB", "512")) << 20
        buf = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{dev}")
        check(load().marl_set_scratch(buf.data_ptr(), nbytes), "marl_set_scratch")
        _scratch[dev] = buf
    return _scratch[dev]


def profile(on):
    load().marl_profile_enable(1 if on else 0)


def profile_collect():
    """{kernel name: (launch count, total ms)} since the last collect."""
    buf = C.create_string_buffer(1 << 16)
    check(load().marl_profile_collect(buf, len(buf)), "marl_profile_collect")
    out = {}
    for line in buf.value.decode().splitlines():
        name, cnt, ms = line.rsplit(",", 2)
        out[name] = (int(cnt), float(ms))
    return out


def profile_timeline():
    """[(kernel name, start_us, end_us)] of the launches recorded since the last collect (records are kept)."""
    buf = C.create_string_buffer(1 << 20)
    check(load().marl_profile_timeline(buf, len(buf)), "marl_profile_timeline")
    rows = []
    for line in buf.value.decode().splitlines():
        name, s, e = line.rsplit(",", 2)
        rows.append((name, float(s), float(e)))
    return rows


def call(name, *args):
    if not _scratch and torch.cuda.is_available():
        ensure_scratch()
    check(getattr(load(), name)(*args), name)
