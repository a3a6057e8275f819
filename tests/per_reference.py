"""TEST INFRASTRUCTURE ONLY -- float64 numpy restatement of tianshou 1.0 ``PrioritizedReplayBuffer`` over the device
replay ring, the reference that tests/test_prioritized_replay_{host,gpu}.py hold ``melissa_b200.replay.
DevicePrioritizedReplay`` and csrc/replay_per.cu to.  Not product code: melissa_b200 never imports this module."""
from __future__ import annotations

import numpy as np


class PrioritizedRingReference:
    """float64 numpy restatement of tianshou 1.0 ``PrioritizedReplayBuffer`` over the device replay ring, the reference
    of ``melissa_b200.replay.DevicePrioritizedReplay`` and ``csrc/replay_per.cu``.  PARITY UNPINNED, like the n-step
    recursion above: it restates the published algorithm (``init_weight``, ``sample_indices`` through
    ``SegmentTree.get_prefix_sum_idx``, ``get_weight``, ``update_weight``, ``set_beta``), not tianshou's code.

    * ``leaf[slot, cell]`` = p^alpha (cell = episode * N + agent); a stored round gives its acted cells max_prio^alpha
      and every other cell 0; ``max_prio = min_prio = 1`` at the start, eps = float32 machine epsilon;
    * sampling concatenates the leaves of the usable slots (oldest first), S = inclusive prefix sums, v = u * S[-1], and
      takes min{i : leaf_i > 0 and S_i >= v} -- tianshou's descent ``go right while the left sum < v`` -- or the last
      positive leaf when v passes it; a leaf of priority 0 is never taken (tianshou would return it for v = 0);
    * ``update`` sets leaf = (|td| + eps)^alpha with numpy fancy assignment (the last occurrence of a leaf wins) and
      tracks max_prio / min_prio on |td| + eps;
    * ``weights`` = (leaf / min_prio)^(-beta), divided by the batch maximum with ``weight_norm``."""

    def __init__(self, n_slots, n_cells, alpha, beta, weight_norm=True, eps=None):
        self.leaf = np.zeros((n_slots, n_cells), dtype=np.float64)
        self.alpha, self.beta, self.weight_norm = float(alpha), float(beta), bool(weight_norm)
        self.eps = float(np.finfo(np.float32).eps) if eps is None else float(eps)
        self.max_prio = self.min_prio = 1.0

    def store_round(self, slot, acted):
        self.leaf[slot] = np.where(np.asarray(acted, dtype=bool).reshape(-1), self.max_prio ** self.alpha, 0.0)

    def sample(self, u, slots):
        """u [M] in [0, 1), slots = usable ring slots oldest first -> (slot, cell, leaf value) arrays [M]."""
        flat = self.leaf[np.asarray(slots)].reshape(-1)
        S = np.cumsum(flat)
        v = np.asarray(u, dtype=np.float64) * S[-1]
        pos = np.flatnonzero(flat > 0)
        if len(pos) == 0:
            raise ValueError("no positive priority in the usable slots")
        k = np.minimum(np.searchsorted(S[pos], v, side="left"), len(pos) - 1)   # S is strictly rising on positive leaves
        i = pos[k]
        C = self.leaf.shape[1]
        return np.asarray(slots)[i // C], i % C, flat[i]

    def update(self, slot, cell, td):
        raw = np.abs(np.asarray(td, dtype=np.float64)) + self.eps
        if raw.size == 0:
            return
        key = np.asarray(slot, dtype=np.int64) * self.leaf.shape[1] + np.asarray(cell, dtype=np.int64)
        _, first_rev = np.unique(key[::-1], return_index=True)
        last = len(key) - 1 - first_rev                                  # the last occurrence of every leaf
        self.leaf.reshape(-1)[key[last]] = raw[last] ** self.alpha
        self.max_prio = max(self.max_prio, float(raw.max()))
        self.min_prio = min(self.min_prio, float(raw.min()))

    def weights(self, slot, cell):
        w = (self.leaf[np.asarray(slot), np.asarray(cell)] / self.min_prio) ** (-self.beta)
        return w / w.max() if self.weight_norm else w
