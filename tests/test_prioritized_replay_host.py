"""CPU: tests/per_reference.py PrioritizedRingReference (the reference of the prioritized replay kernels) against a
brute-force prefix-sum search and a binary segment tree restated from tianshou's SegmentTree, on random rings with
dyadic priorities (every summation order is exact)."""
import numpy as np
import pytest

from per_reference import PrioritizedRingReference


class BinarySegmentTree:
    """tianshou ``SegmentTree`` (power-of-two bound, node i = children 2i + 2i+1) and its ``get_prefix_sum_idx``:
    descend left while the left child's sum >= v, else subtract it and go right."""

    def __init__(self, values):
        self.bound = 1
        while self.bound < len(values):
            self.bound *= 2
        self.value = np.zeros(2 * self.bound)
        self.value[self.bound:self.bound + len(values)] = values
        for i in range(self.bound - 1, 0, -1):
            self.value[i] = self.value[2 * i] + self.value[2 * i + 1]

    def prefix_sum_idx(self, v):
        v = np.array(v, dtype=np.float64)
        index = np.ones(v.shape, dtype=np.int64)
        while index[0] < self.bound:
            index *= 2
            left = self.value[index]
            right = left < v
            v -= left * right
            index += right
        return index - self.bound


def brute_force(flat, v):
    """min{i : flat_i > 0 and S_i >= v}, else the last positive leaf, one v at a time."""
    S = np.cumsum(flat)
    out = []
    for x in np.atleast_1d(v):
        hits = [i for i in range(len(flat)) if flat[i] > 0 and S[i] >= x]
        out.append(hits[0] if hits else int(np.flatnonzero(flat > 0)[-1]))
    return np.array(out)


def random_ring(rng, R, C, p_acted=0.6, eps=0.0):
    """Reference with alpha = 1, eps = 0 and dyadic priorities in {1/4, 1/2, 1, 2, 4} on the acted cells."""
    ref = PrioritizedRingReference(R, C, alpha=1.0, beta=0.4, eps=eps)
    for s in range(R):
        acted = rng.random(C) < p_acted
        ref.store_round(s, acted)
        cells = np.flatnonzero(acted)
        ref.update(np.full(len(cells), s), cells, 2.0 ** rng.integers(-2, 3, size=len(cells)))
    return ref


@pytest.mark.parametrize("seed", range(6))
def test_reference_matches_brute_force_and_binary_segment_tree(seed):
    rng = np.random.default_rng(seed)
    R, C = int(rng.integers(2, 9)), int(rng.integers(1, 70))
    ref = random_ring(rng, R, C, p_acted=rng.uniform(0.05, 0.9))
    ref.leaf[rng.integers(R)] = 0.0                                     # a round of count 0
    first, n = int(rng.integers(R)), int(rng.integers(1, R + 1))
    slots = (first + np.arange(n)) % R
    flat = ref.leaf[slots].reshape(-1)
    if not (flat > 0).any():
        return
    u = rng.random(500)
    slot, cell, val = ref.sample(u, slots)
    i = np.searchsorted(slots, slot, sorter=np.argsort(slots))          # position of the slot in the order
    i = np.argsort(slots)[i] * C + cell
    np.testing.assert_array_equal(i, brute_force(flat, u * flat.sum()))
    np.testing.assert_array_equal(val, flat[i])
    assert (val > 0).all()
    v = u * flat.sum()
    inside = v > 0
    np.testing.assert_array_equal(i[inside], BinarySegmentTree(flat).prefix_sum_idx(v[inside]))


def test_boundaries_zero_cells_and_rounding_past_the_end():
    flat_leaves = np.array([[0.0, 0.5, 0.0, 0.25], [0.0, 0.0, 0.0, 0.0], [1.0, 0.0, 0.25, 0.0]])
    ref = PrioritizedRingReference(3, 4, alpha=1.0, beta=0.5, eps=0.0)
    ref.leaf[:] = flat_leaves
    slots = np.array([2, 0, 1])                                         # oldest first; slot 1 holds nothing
    flat = ref.leaf[slots].reshape(-1)                                  # [1, 0, .25, 0, 0, .5, 0, .25, 0, 0, 0, 0]
    T = flat.sum()
    assert T == 2.0
    S = np.cumsum(flat)
    # u exactly on every prefix sum: v = S_i picks the positive leaf that ends there
    for i in np.flatnonzero(flat > 0):
        s, c, _ = ref.sample([S[i] / T], slots)
        assert (s[0], c[0]) == (slots[i // 4], i % 4)
    # v = 0: the first positive leaf; v just above a prefix sum: the next positive leaf, skipping zero cells
    assert ref.sample([0.0], slots)[:2] == (2, 0)
    s, c, _ = ref.sample([S[0] / T + 1e-12], slots)
    assert (s[0], c[0]) == (2, 2)
    # v at or past the total: the last positive leaf
    for u in (1.0, 1.0 + 1e-9):
        s, c, val = ref.sample([u], slots)
        assert (s[0], c[0], val[0]) == (0, 3, 0.25)
    # zero cells and the empty round are never returned
    s, c, val = ref.sample(np.linspace(0.0, 1.0, 4097), slots)
    assert (val > 0).all() and (s != 1).all()
    with pytest.raises(ValueError):
        ref.sample([0.5], np.array([1]))


def test_duplicate_updates_last_wins_and_priority_tracking():
    ref = PrioritizedRingReference(2, 5, alpha=0.6, beta=0.4)
    ref.store_round(0, [1, 1, 0, 1, 1])
    ref.store_round(1, [1, 0, 1, 0, 0])
    np.testing.assert_array_equal(ref.leaf, [[1, 1, 0, 1, 1], [1, 0, 1, 0, 0]])
    slot = np.array([0, 1, 0, 0, 1, 0])
    cell = np.array([1, 2, 3, 1, 2, 1])
    td = np.array([3.0, -0.5, 2.0, 7.0, 0.25, -0.125], dtype=np.float32)
    ref.update(slot, cell, td)
    eps = float(np.finfo(np.float32).eps)
    assert ref.leaf[0, 1] == (0.125 + eps) ** 0.6                       # last of three writes to (0, 1)
    assert ref.leaf[1, 2] == (0.25 + eps) ** 0.6
    assert ref.leaf[0, 3] == (2.0 + eps) ** 0.6
    assert ref.max_prio == 7.0 + eps and ref.min_prio == 0.125 + eps
    ref.store_round(1, [0, 1, 1, 1, 1])                                 # a new round starts at max_prio^alpha
    np.testing.assert_array_equal(ref.leaf[1], [0.0] + [(7.0 + eps) ** 0.6] * 4)
    ref.update([0], [0], [0.0])
    assert ref.min_prio == eps and ref.max_prio == 7.0 + eps


@pytest.mark.parametrize("weight_norm", [True, False])
def test_weights(weight_norm):
    rng = np.random.default_rng(5)
    ref = PrioritizedRingReference(3, 40, alpha=0.7, beta=0.45, weight_norm=weight_norm)
    for s in range(3):
        ref.store_round(s, rng.random(40) < 0.5)
    cells = np.flatnonzero(ref.leaf.reshape(-1) > 0)
    ref.update(cells // 40, cells % 40, rng.normal(size=len(cells)))
    slot, cell, val = ref.sample(rng.random(300), np.array([1, 2, 0]))
    w = ref.weights(slot, cell)
    want = np.array([(v / ref.min_prio) ** -0.45 for v in val])
    if weight_norm:
        want = want / want.max()
        assert w.max() == 1.0
    np.testing.assert_allclose(w, want, rtol=1e-15)
    ref.beta = 0.0
    np.testing.assert_array_equal(ref.weights(slot, cell), np.ones(len(slot)))


@pytest.mark.parametrize("alpha,beta", [(0.0, 0.4), (-0.5, 0.4), (0.6, -0.1), (float("nan"), 0.4)])
def test_prioritized_replay_rejects_bad_alpha_and_beta_before_touching_the_device(alpha, beta):
    from melissa_b200.replay import DevicePrioritizedReplay
    with pytest.raises(ValueError):
        DevicePrioritizedReplay(4, 3, 8, alpha=alpha, beta=beta, device="cpu")
