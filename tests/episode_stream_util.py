"""Exact probabilities of the device episode sampler's draws (include/melissa_b200.h, MlsEpisodeSampler), for the
statistical tests of the episode stream."""
import math

import numpy as np

U_BITS = 53


def k_of_u(j: int, n_nodes: int) -> int:
    """Interested count of the 53-bit uniform u = j / 2^53, in the same fp64 operations as the sampler (and numpy's
    uniform(0.1, 1.0)): k = int((0.1 + (1.0 - 0.1) * u) * N)."""
    u = j * 2.0 ** -U_BITS
    return int((0.1 + (1.0 - 0.1) * u) * n_nodes)


def k_probabilities(n_nodes: int) -> np.ndarray:
    """P(k = m), m = 0..N: the share of the 2^53 grid points u whose k equals m.  k is non-decreasing in u, so each
    value owns an interval of grid points, found by bisection."""
    top = 1 << U_BITS

    def first_at_least(m):          # smallest j with k(j) >= m (top when none)
        lo, hi = 0, top
        while lo < hi:
            mid = (lo + hi) // 2
            if k_of_u(mid, n_nodes) >= m:
                hi = mid
            else:
                lo = mid + 1
        return lo

    edges = [first_at_least(m) for m in range(n_nodes + 2)]
    return np.array([(edges[m + 1] - edges[m]) / top for m in range(n_nodes + 1)], dtype=np.float64)


def node_inclusion(k, n_nodes: int):
    """P(node i is interested | k) and P(nodes i != j are both interested | k) of a uniform k-subset."""
    k = np.asarray(k, dtype=np.float64)
    return k / n_nodes, k * (k - 1) / (n_nodes * (n_nodes - 1))


def expected_duplicate_pairs(n_draws: int, n_nodes: int, pool_size: int) -> float:
    """Expected number of equal pairs among n_draws independent tuples without scripted agents:
    C(n, 2) * sum over tuples of p(tuple)^2, p = 1/G * 1/N * P(k) / C(N, k)."""
    pk = k_probabilities(n_nodes)
    s = sum(pk[m] ** 2 / math.comb(n_nodes, m) for m in range(n_nodes + 1))
    return n_draws * (n_draws - 1) / 2 * s / (pool_size * n_nodes)
