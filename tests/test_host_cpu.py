"""CPU-only checks: host logic, state_dict compatibility, C-ABI library loads and exports its symbols."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from marl_b200 import _lib as L
from marl_b200.algorithm.q_learner import QLearner, host_max_episode_len
from marl_b200.common.arguments import default_args
from marl_b200.controller.share_params import SharedMAC
from marl_b200.env.single_state_matrix_game import TwoAgentsMatrixGame
from marl_b200.synthetic import synthetic_batch, KEYS
from oracle import marl_oracle as MO
from tests import golden_util as GU

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "marl_b200.h")).read()
    declared = set(re.findall(r"^int\s+(marl_\w+)\s*\(", hdr, flags=re.M))
    assert declared, "no declarations parsed"
    lib = ctypes.CDLL(L.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert declared == set(L.exported_symbols())
    assert lib.marl_version() == 100


def test_no_cpu_fallback():
    if torch.cuda.is_available():
        pytest.skip("CPU-only check")
    a = default_args(alg="vdn", n_agents=2, n_actions=3, obs_shape=4, state_shape=5, episode_limit=3)
    learner = QLearner(SharedMAC(a), a)
    with pytest.raises(L.MarlLibraryError):
        learner.train(synthetic_batch(0, 2, 3, 2, 3, 4, 5), 0)


def test_product_never_imports_oracle():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "marl_b200")):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, flags=re.M), f


def test_state_dict_keys_and_seeded_init_match_reference_goldens():
    z = GU.load("tiny_qmix_rms")
    cfg = GU.cfg_from(z)
    a = default_args(alg="qmix", n_agents=cfg.n_agents, n_actions=cfg.n_actions, obs_shape=cfg.obs_shape,
                     state_shape=cfg.state_shape, episode_limit=cfg.episode_limit)
    torch.manual_seed(0)                       # the seed make_golden.py used for the reference modules
    mac = SharedMAC(a)
    learner = QLearner(mac, a)
    for k, v in GU.group(z, "init/agent").items():
        assert torch.equal(mac.agent.state_dict()[k].cpu(), v), k
    for k, v in GU.group(z, "init/mixer").items():
        assert torch.equal(learner.mixer.state_dict()[k].cpu(), v), k


def test_flat_layout_concatenates_qmix_heads():
    a = default_args(alg="qmix", n_agents=5, n_actions=11, obs_shape=80, state_shape=120, episode_limit=120)
    learner = QLearner(SharedMAC(a), a)
    fl = learner._flat
    S, E, N = 120, 32, 5
    o = fl.offsets
    assert o["mixer.hyper_b1.weight"] == o["mixer.hyper_w1.weight"] + N * E * S
    assert o["mixer.hyper_w2.weight"] == o["mixer.hyper_b1.weight"] + E * S
    assert o["mixer.hyper_b2.0.weight"] == o["mixer.hyper_w2.weight"] + E * S
    assert o["mixer.hyper_b1.bias"] == o["mixer.hyper_w1.bias"] + N * E
    for p in learner.params:                    # parameters are views of the flat buffer, grads attached
        assert p.data_ptr() >= fl.data.data_ptr() and p.grad is not None
    assert all(off % 4 == 0 for off in o.values())
    assert sum(p.numel() for p in learner.params) == 62892


def test_gradient_buffer_can_move_to_caller_memory():
    """Data parallel puts [grad | loss_sum | mask_sum] into cudaIpc-shared memory (parallel.PeerGradients): the
    parameters' .grad views and the tail must follow, and the fused exchange needs numel % 4 == 0 and <= 2^18."""
    a = default_args(alg="qmix", n_agents=5, n_actions=11, obs_shape=80, state_shape=120, episode_limit=120)
    learner = QLearner(SharedMAC(a), a)
    fl = learner._flat
    assert fl.numel % 4 == 0 and fl.numel <= (1 << 18) and fl.grad_full.numel() == fl.numel + 2
    new = torch.full((fl.numel + 2,), 7.0, device=fl.grad_full.device)      # the learner packs on CUDA when there is one
    fl.adopt_grad_storage(new)
    assert float(new.abs().max()) == 0.0                       # zeroed on adoption
    assert fl.grad.data_ptr() == new.data_ptr() and fl.tail.data_ptr() == new.data_ptr() + 4 * fl.numel
    for name, p in zip(fl.names, fl.params):
        assert p.grad.data_ptr() == new.data_ptr() + 4 * fl.offsets[name] and p.grad.shape == p.shape


def test_peer_exchange_rejects_bad_arguments_without_touching_the_gpu():
    lib = L.load()
    pg = L.PeerGroup()
    pg.world, pg.rank = 9, 0                                   # more ranks than MARL_PEER_MAX_WORLD
    assert lib.marl_clip_step_peer(0, 16, 16, 16, None, 4, 10.0, 5e-4, 0.99, 0.0, 1e-8, None, None,
                                   ctypes.byref(pg), None) < 0               # MARL_EINVAL
    assert lib.marl_clip_step_peer(0, None, 16, 16, None, 4, 10.0, 5e-4, 0.99, 0.0, 1e-8, None, None,
                                   ctypes.byref(pg), None) < 0
    assert lib.marl_peer_export(None, None) < 0 and lib.marl_peer_open(None, None) < 0


def test_reference_checkpoint_keys_load():
    a = default_args(alg="vdn", n_agents=5, n_actions=11, obs_shape=80, state_shape=120, episode_limit=120)
    mac = SharedMAC(a)
    sd = {k: torch.randn_like(v) for k, v in MO.init_agent(MO.make_cfg(n_agents=5, n_actions=11, obs_shape=80,
                                                                    state_shape=120, episode_limit=120)).items()}
    mac.agent.load_state_dict(sd)
    assert torch.equal(mac.agent.fc1.weight.detach().cpu(), sd["fc1.weight"])
    assert mac.agent.fc1.weight.data_ptr() == mac.agent._flat.data.data_ptr()   # still a view of the flat buffer


def test_host_max_episode_len_matches_oracle():
    rng = np.random.RandomState(0)
    for _ in range(20):
        B, T = rng.randint(1, 6), rng.randint(1, 9)
        term = (rng.rand(B, T, 1) < 0.3).astype(np.float64)
        assert host_max_episode_len(term, T) == MO.max_episode_len(term, T)
    assert host_max_episode_len(np.zeros((2, 4, 1)), 4) == 4


def test_synthetic_batch_follows_rollout_padding_convention():
    b = synthetic_batch(0, 8, 12, 3, 5, 4, 6)
    assert set(b) == set(KEYS) and all(v.dtype == np.float64 for v in b.values())
    pad = b["padded"][..., 0] == 1
    for k in ("o", "s", "r", "o_next", "s_next", "avail_u", "avail_u_next", "u_onehot", "u"):
        assert not b[k][pad].any(), k                       # rollout.py:122-132
    assert (b["terminated"][..., 0][pad] == 1).all()        # rollout.py:133
    live = ~pad
    assert (np.take_along_axis(b["avail_u"], b["u"].astype(np.int64), -1)[..., 0][live] == 1).all()
    assert np.array_equal(b["u_onehot"].argmax(-1)[live], b["u"][..., 0][live].astype(np.int64))
    assert np.array_equal(b["o_next"][:, :-1][live[:, 1:]], b["o"][:, 1:][live[:, 1:]])


def test_env_matches_reference_golden():
    z = np.load(GU.GOLDEN_DIR + "/matrix_game_env.npz")
    for t in range(3):
        env = TwoAgentsMatrixGame(z[f"t{t}/payoff"])
        ep = env.get_episodes()
        for k, v in ep.items():
            ref = z[f"t{t}/episodes/{k}"]
            assert v.dtype == ref.dtype and np.array_equal(v, ref), k
        for a0 in range(3):
            for a1 in range(3):
                env.reset()
                r, term, info = env.step([a0, a1])
                assert r == z[f"t{t}/step_reward"][a0, a1] and isinstance(r, np.float64) and term is True and info == {}
        assert len(env.replay) == int(z[f"t{t}/replay_len"])
        assert np.array_equal(np.array(env.get_obs()), z[f"t{t}/obs"])
        assert np.array_equal(np.array(env.get_avail_actions()), z[f"t{t}/avail"])
        info = env.get_env_info()
        assert [info[k] for k in ("n_actions", "n_agents", "state_shape", "obs_shape", "episode_limit")] == list(z[f"t{t}/env_info"])
        env.close()
        assert len(env.replay) == 1 and env.current_episode == 0


def test_ctypes_structs_have_the_headers_layout(tmp_path):
    """Every struct that crosses the C ABI is declared twice -- include/marl_b200.h and the ctypes mirror in marl_b200/_lib.py.
    A tiny C program compiled against the header prints sizeof and the offset of every field; the mirror must agree (a
    field added on one side only would shift every pointer behind it)."""
    import shutil, subprocess
    if shutil.which("gcc") is None:
        pytest.skip("no C compiler")
    pairs = {"marl_dims": L.Dims, "marl_episode_f32": L.EpisodeF32, "marl_episode_f64": L.EpisodeF64,
             "marl_agent_params": L.AgentParams, "marl_agent_grads": L.AgentGrads, "marl_unroll_stream": L.UnrollStream,
             "marl_unroll_bwd": L.UnrollBwd, "marl_peer_group": L.PeerGroup, "marl_select_fused": L.SelectFused,
             "marl_qmix_params": L.QmixParams, "marl_qmix_grads": L.QmixGrads, "marl_qmix_hyper2": L.QmixHyper2,
             "marl_qmix_hyper2_grads": L.QmixHyper2Grads, "marl_qplex_dims": L.QplexDims, "marl_qplex_params": L.QplexParams,
             "marl_qplex_grads": L.QplexGrads, "marl_qplex_ws": L.QplexWs, "marl_qtran_net_params": L.QtranNetParams,
             "marl_qtran_net_grads": L.QtranNetGrads, "marl_qtran_net_ws": L.QtranNetWs}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "marl_b200.h"', 'int main(void) {']
    for cname, cls in pairs.items():
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    inc = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include")
    r = subprocess.run(["gcc", "-I", inc, str(src), "-o", str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr          # (a field name that only exists in the mirror fails right here)
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True).stdout.splitlines())
    for cname, cls in pairs.items():
        assert int(got[cname]) == ctypes.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(got[f"{cname}.{fname}"]) == getattr(cls, fname).offset, (cname, fname)


def test_bench_dump_outputs_file_layout(tmp_path):
    """bench.py --dump-outputs, file layout only (on hand-made hidden states; which step is dumped is bench.py's business):
    one <name>.npy per array a caller of QLearner.train holds after a step -- loss, clipped gradients, trained and target
    networks, the two controllers' hidden states -- float64 for the loss and float32 otherwise, far below 64 MB."""
    import bench
    a = bench.make_args()
    learner = QLearner(SharedMAC(a), a)
    rows = bench.SHAPE["B"] * bench.SHAPE["N"]
    learner.eval_net.hidden_states = torch.randn(rows, 64)            # as train() leaves them: [B*N, H]
    learner.target_net.hidden_states = torch.randn(rows, 64)
    bench.write_outputs(str(tmp_path), bench.snapshot_outputs(torch, learner, 1.5))
    got = {p.name[:-4]: np.load(p) for p in tmp_path.iterdir()}
    want = {"loss", "hidden_states", "target_hidden_states"}
    for prefix, module in (("agent", learner.eval_net.agent), ("mixer", learner.mixer)):
        for k, p in module.named_parameters():
            want.add(f"grad.{prefix}.{k}")
            assert np.array_equal(got[f"grad.{prefix}.{k}"], p.grad.cpu().numpy()), (prefix, k)
    for prefix, module in (("agent", learner.eval_net.agent), ("mixer", learner.mixer),
                           ("target_agent", learner.target_net.agent), ("target_mixer", learner.target_mixer)):
        for k, v in module.state_dict().items():
            want.add(f"{prefix}.{k}")
            assert np.array_equal(got[f"{prefix}.{k}"], v.cpu().numpy()), (prefix, k)
    assert set(got) == want
    assert got["loss"].dtype == np.float64 and got["loss"].tolist() == [1.5]
    assert all(v.dtype == np.float32 for k, v in got.items() if k != "loss")
    assert np.array_equal(got["hidden_states"], learner.eval_net.hidden_states.numpy())
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) < 64 << 20
