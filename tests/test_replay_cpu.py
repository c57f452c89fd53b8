"""Host logic of the device replay buffer (run on CPU tensors) against the oracle restatement and, when the
reference is staged in oracle/_ref (oracle/fetch_ref.py), against the reference's own ReplayBuffer (common/replaybuffer.py)."""
import sys
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from marl_b200.common.replaybuffer import ReplayBuffer, DeviceEpisodeBatch, KEYS
from marl_b200.synthetic import synthetic_batch
from oracle import fetch_ref as FR
from oracle.replay_oracle import OracleReplayBuffer

DIMS = dict(T=6, N=2, A=3, O=4, S=5)


def _args(size):
    return SimpleNamespace(n_actions=DIMS["A"], n_agents=DIMS["N"], state_shape=DIMS["S"], obs_shape=DIMS["O"],
                           buffer_size=size, episode_limit=DIMS["T"])


def test_ring_cursor_matches_oracle_over_many_wraps():
    mine = ReplayBuffer(_args(7), device="cpu")
    orc = OracleReplayBuffer(7, **DIMS)
    rng = np.random.RandomState(0)
    for _ in range(500):
        n = int(rng.randint(1, 6))
        got = mine._get_storage_idx(n)
        want = orc.next_positions(n)
        assert list(np.atleast_1d(got)) == want
        assert np.isscalar(got) or got.ndim == 0 if n == 1 else got.shape == (n,)
        assert (mine.current_idx, mine.current_size) == (orc.cursor, orc.filled)


@pytest.mark.skipif(not FR.available(), reason="reference not staged in oracle/_ref")
def test_ring_cursor_matches_reference():
    sys.path.insert(0, FR.DST)
    try:
        from common.replaybuffer import ReplayBuffer as Ref
    finally:
        sys.path.remove(FR.DST)
    ref, mine = Ref(_args(5)), ReplayBuffer(_args(5), device="cpu")
    rng = np.random.RandomState(1)
    for _ in range(300):
        n = int(rng.randint(1, 5))
        assert list(np.atleast_1d(ref._get_storage_idx(n))) == list(np.atleast_1d(mine._get_storage_idx(n)))
        assert (ref.current_idx, ref.current_size) == (mine.current_idx, mine.current_size)


def test_store_and_sample_match_oracle_bitwise_in_fp32():
    mine = ReplayBuffer(_args(9), device="cpu")
    orc = OracleReplayBuffer(9, **DIMS)
    for seed in range(5):                                   # 5 x 4 episodes into 9 slots: wraps twice
        ep = synthetic_batch(seed, 4, DIMS["T"], DIMS["N"], DIMS["A"], DIMS["O"], DIMS["S"], full_length_first=False)
        mine.store_episode({k: v.copy() for k, v in ep.items()})
        orc.store(ep)
    np.random.seed(123)
    want, idx = orc.sample(16)
    np.random.seed(123)
    got = mine.sample(16)
    assert isinstance(got, DeviceEpisodeBatch) and list(got.idx_host) == list(idx)
    for k in KEYS:
        w = want[k].astype(np.int64) if k == "u" else want[k].astype(np.float32)
        assert np.array_equal(got[k].numpy(), w), k
    # episode-length cut of q_learner.py:49-61 from the host-side bookkeeping
    term = want["terminated"][:, :, 0] == 1
    has = term.any(axis=1)
    expect = int(term.argmax(axis=1)[has].max()) + 1 if has.any() else DIMS["T"]
    assert got.max_episode_len == expect == got["max_episode_len"]
    # dict protocol the reference's get_max_episode_len relies on (q_learner.py:63-64)
    for key in got.keys():
        got[key] = got[key][:, :expect]
    assert got["o"].shape[1] == expect


def test_device_tensor_episodes_are_stored_like_host_ones():
    a, b = ReplayBuffer(_args(4), device="cpu"), ReplayBuffer(_args(4), device="cpu")
    ep = synthetic_batch(3, 3, DIMS["T"], DIMS["N"], DIMS["A"], DIMS["O"], DIMS["S"])
    a.store_episode(ep)
    b.store_episode({k: torch.from_numpy(v) for k, v in ep.items()})
    for k in KEYS:
        assert torch.equal(a.buffers[k], b.buffers[k]), k
    assert np.array_equal(a.first_terminated, b.first_terminated)
