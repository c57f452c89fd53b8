"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the reference's episode replay buffer.

Follows ``common/replaybuffer.py:5-80`` of the reference: eleven float64 numpy rings
``[buffer_size, episode_limit, ...]`` (``:19-30``), ``store_episode`` (``:35-51``), uniform sampling with
replacement through ``np.random.randint`` (``:54-60``) and the ring cursor of ``_get_storage_idx``
(``:63-80``).  Pinned against the reference itself by ``tests/test_replay_cpu.py`` when it is staged in
``oracle/_ref``.  Only tests may import this module; the product's buffer is ``marl_b200/common/replaybuffer.py``.
"""
import numpy as np

KEYS = ("o", "u", "s", "r", "o_next", "s_next", "avail_u", "avail_u_next", "u_onehot", "padded", "terminated")


def shapes(size, T, N, A, O, S):
    return {"o": (size, T, N, O), "u": (size, T, N, 1), "s": (size, T, S), "r": (size, T, 1), "o_next": (size, T, N, O),
            "s_next": (size, T, S), "avail_u": (size, T, N, A), "avail_u_next": (size, T, N, A),
            "u_onehot": (size, T, N, A), "padded": (size, T, 1), "terminated": (size, T, 1)}


class OracleReplayBuffer:
    def __init__(self, size, T, N, A, O, S):
        self.size, self.cursor, self.filled = size, 0, 0
        self.rings = {k: np.zeros(shp) for k, shp in shapes(size, T, N, A, O, S).items()}

    def next_positions(self, count):            # replaybuffer.py:63-80
        if self.cursor + count <= self.size:
            pos = list(range(self.cursor, self.cursor + count))
            self.cursor += count
        elif self.cursor < self.size:
            spill = count - (self.size - self.cursor)
            pos = list(range(self.cursor, self.size)) + list(range(spill))
            self.cursor = spill
        else:
            pos = list(range(count))
            self.cursor = count
        self.filled = min(self.size, self.filled + count)
        return pos

    def store(self, episodes):                  # replaybuffer.py:35-51
        pos = self.next_positions(episodes["o"].shape[0])
        for k in KEYS:
            self.rings[k][pos] = episodes[k]
        return pos

    def sample(self, batch_size):               # replaybuffer.py:54-60
        idx = np.random.randint(0, self.filled, batch_size)
        return {k: self.rings[k][idx] for k in KEYS}, idx
