"""GPU: prioritized replay (csrc/replay_per.cu, melissa_b200.replay.DevicePrioritizedReplay) against
tests/per_reference.py PrioritizedRingReference -- the kernels through the C ABI on hand-built rings, sampling
statistics, the policy hook end to end with a collector driven in lockstep with oracle/env_oracle.py, and the absence of
host synchronisation.  Exact comparisons use alpha = 1, eps = 0 and dyadic priorities, so every summation order is
exact."""
import math

import numpy as np
import pytest
import torch

from melissa_b200 import _lib, reset_chain
from melissa_b200.topology import GraphPool
from oracle.env_oracle import BatchedEnvOracle
from per_reference import PrioritizedRingReference

pytestmark = pytest.mark.gpu
EPS32 = float(np.finfo(np.float32).eps)


class Trees:
    """The prioritized ring's trees driven straight through the C ABI."""

    def __init__(self, R, B, N):
        self.L = _lib.lib()
        self.R, self.B, self.N, self.C = R, B, N, B * N
        self.size = int(self.L.mls_per_tree_size(self.C))
        self.t = torch.zeros(R, self.size, dtype=torch.float64, device="cuda")
        self.prio = torch.ones(2, dtype=torch.float64, device="cuda")
        sizes = [self.C]
        while sizes[-1] > 1:
            sizes.append((sizes[-1] + 31) // 32)
        self.sizes, self.offs = sizes, np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
        assert sum(sizes) == self.size

    def build(self, slot, acted, alpha):
        flags = torch.as_tensor(np.asarray(acted, dtype=np.uint8).reshape(-1), device="cuda")
        _lib.check(self.L.mls_per_build(flags.data_ptr(), self.B, self.N, self.prio.data_ptr(), alpha,
                                        self.t[slot].data_ptr(), _lib.current_stream_ptr()))

    def sample(self, u, first, n):
        u = torch.as_tensor(u, dtype=torch.float64, device="cuda")
        M = int(u.shape[0])
        rho, ep, ag = (torch.empty(M, dtype=torch.int32, device="cuda") for _ in range(3))
        leaf = torch.empty(M, dtype=torch.float64, device="cuda")
        _lib.check(self.L.mls_per_sample(self.t.data_ptr(), self.R, self.B, self.N, first, n, u.data_ptr(), M, rho.data_ptr(),
                                         ep.data_ptr(), ag.data_ptr(), leaf.data_ptr(), _lib.current_stream_ptr()))
        return (rho.cpu().numpy().astype(np.int64), (ep.long() * self.N + ag.long()).cpu().numpy(), leaf.cpu().numpy())

    def update(self, slot, cell, td, alpha, eps):
        slot, cell = np.asarray(slot), np.asarray(cell)
        r = torch.as_tensor(slot.astype(np.int32), device="cuda")
        e = torch.as_tensor((cell // self.N).astype(np.int32), device="cuda")
        a = torch.as_tensor((cell % self.N).astype(np.int32), device="cuda")
        d = torch.as_tensor(np.asarray(td, dtype=np.float32), device="cuda")
        _lib.check(self.L.mls_per_update(self.t.data_ptr(), self.R, self.B, self.N, r.data_ptr(), e.data_ptr(), a.data_ptr(),
                                         d.data_ptr(), len(slot), alpha, eps, self.prio.data_ptr(), self.prio[1:].data_ptr(),
                                         _lib.current_stream_ptr()))

    def leaves(self):
        return self.t[:, :self.C].cpu().numpy()

    def check_internal_nodes(self, exact=True):
        t = self.t.cpu().numpy()
        for k in range(1, len(self.sizes)):
            child = np.zeros((self.R, self.sizes[k] * 32))
            child[:, :self.sizes[k - 1]] = t[:, self.offs[k - 1]:self.offs[k - 1] + self.sizes[k - 1]]
            got = t[:, self.offs[k]:self.offs[k] + self.sizes[k]]
            want = child.reshape(self.R, -1, 32).sum(axis=2)
            if exact:
                np.testing.assert_array_equal(got, want, err_msg=f"level {k}")
            else:
                np.testing.assert_allclose(got, want, rtol=1e-13, err_msg=f"level {k}")


def _usable(head, R, n_step):
    """DeviceReplay's usable-round rule -> (first slot, count) or None."""
    filled = min(head, R)
    n = filled - n_step
    return None if n <= 0 else ((head - filled) % R, n)


def _dyadic_ring(rng, R, B, N, p_acted=0.5, empty_slots=()):
    """Every slot built from random flags (at max_prio 1), then every acted cell set to a dyadic priority by an update
    (alpha 1, eps 0) -- the same on the device and in the reference."""
    tr, ref = Trees(R, B, N), PrioritizedRingReference(R, B * N, alpha=1.0, beta=0.4, eps=0.0)
    for s in range(R):
        acted = (rng.random(B * N) < p_acted) & (s not in empty_slots)
        tr.build(s, acted, 1.0)
        ref.store_round(s, acted)
    slot, cell = np.nonzero(ref.leaf > 0)
    td = 2.0 ** rng.integers(-3, 4, size=len(slot)) * rng.choice([-1.0, 1.0], size=len(slot))
    tr.update(slot, cell, td, 1.0, 0.0)
    ref.update(slot, cell, td)
    return tr, ref


@pytest.mark.parametrize("B,N,R", [(1, 1, 5), (3, 4, 1000), (2, 16, 64), (33, 50, 6), (700, 50, 3)])
def test_exact_sampling_matches_the_reference_before_and_after_wrap(B, N, R):
    rng = np.random.default_rng(B * 1000 + N + R)
    tr, ref = _dyadic_ring(rng, R, B, N, empty_slots=(1,) if R > 2 else ())
    np.testing.assert_array_equal(tr.leaves(), ref.leaf)
    tr.check_internal_nodes()
    assert tr.prio.cpu().tolist() == [ref.max_prio, ref.min_prio]
    C = B * N
    for n_step in (1, 2, 3, 4):
        for head in (R - 1, R, 3 * R + 2):
            us = _usable(head, R, n_step) if n_step < R else None
            if us is None:
                continue
            first, n = us
            slots = (first + np.arange(n)) % R
            flat = ref.leaf[slots].reshape(-1)
            u = rng.random(4096)
            if (flat > 0).any():
                S = np.cumsum(flat)
                on = rng.choice(np.flatnonzero(flat > 0), size=min(256, int((flat > 0).sum())), replace=False)
                u = np.concatenate([u, S[on] / S[-1], [0.0, np.nextafter(1.0, 0.0)]])
                s_got, c_got, v_got = tr.sample(u, first, n)
                s_ref, c_ref, v_ref = ref.sample(u, slots)
                np.testing.assert_array_equal(s_got, s_ref, err_msg=f"n_step {n_step} head {head}")
                np.testing.assert_array_equal(c_got, c_ref, err_msg=f"n_step {n_step} head {head}")
                np.testing.assert_array_equal(v_got, v_ref)
                assert (v_got > 0).all() and np.isin(s_got, slots).all()
                assert (ref.leaf[s_got, c_got] > 0).all()                   # acted cells only
            else:                                                           # nothing positive: documented fallback
                s_got, c_got, v_got = tr.sample(u[:64], first, n)
                assert (s_got == first).all() and (c_got == 0).all() and (v_got == 0).all()


def test_u_exactly_on_prefix_sums_of_a_power_of_two_total():
    tr = Trees(3, 1, 4)
    ref = PrioritizedRingReference(3, 4, alpha=1.0, beta=0.4, eps=0.0)
    leaves = np.array([[0.0, 0.5, 0.0, 0.25], [0.0, 0.0, 0.0, 0.0], [1.0, 0.0, 0.25, 0.0]])
    for s in range(3):
        tr.build(s, leaves[s] > 0, 1.0)
        ref.store_round(s, leaves[s] > 0)
    slot, cell = np.nonzero(leaves)
    tr.update(slot, cell, leaves[slot, cell], 1.0, 0.0)
    ref.update(slot, cell, leaves[slot, cell])
    slots = np.array([2, 0, 1])
    flat = leaves[slots].reshape(-1)
    S = np.cumsum(flat)
    assert S[-1] == 2.0                                                     # v = u * T lands exactly on S_i
    u = np.concatenate([S / 2.0, [0.0, S[0] / 2.0 + 1e-12, np.nextafter(1.0, 0.0)]])
    got = tr.sample(u, 2, 3)
    want = ref.sample(u, slots)
    for g, w in zip(got, want):
        np.testing.assert_array_equal(g, w)
    assert list(zip(got[0][:12], got[1][:12])) == [(2, 0), (2, 0), (2, 2), (2, 2), (2, 2), (0, 1), (0, 1), (0, 3),
                                                   (0, 3), (0, 3), (0, 3), (0, 3)]


def test_update_with_duplicate_leaves_last_wins_and_parents_are_sums():
    rng = np.random.default_rng(11)
    R, B, N = 5, 40, 50                                                     # 2000 leaves: 4 levels
    tr, ref = _dyadic_ring(rng, R, B, N)
    for step in range(3):
        s, c, _ = ref.sample(rng.random(3000), np.arange(R))
        dup = rng.integers(0, len(s), size=1500)
        s, c = np.concatenate([s, s[dup]]), np.concatenate([c, c[dup]])
        td = 2.0 ** rng.integers(-6, 6, size=len(s)) * rng.choice([-1.0, 1.0], size=len(s))
        if step == 2:
            td[0] = 0.0                                                     # priority 0: never sampled again
        tr.update(s, c, td, 1.0, 0.0)
        ref.update(s, c, td)
        np.testing.assert_array_equal(tr.leaves(), ref.leaf)
        tr.check_internal_nodes()
        assert tr.prio.cpu().tolist() == [ref.max_prio, ref.min_prio]
    assert ref.min_prio == 0.0
    got_s, got_c, got_v = tr.sample(rng.random(1 << 16), 0, R)
    assert (got_v > 0).all() and (ref.leaf[got_s, got_c] > 0).all()


def test_non_dyadic_roots_and_sampling_away_from_boundaries():
    rng = np.random.default_rng(12)
    R, B, N, alpha = 4, 300, 50, 0.6
    tr = Trees(R, B, N)
    ref = PrioritizedRingReference(R, B * N, alpha=alpha, beta=0.4)
    for s in range(R):
        acted = rng.random(B * N) < 0.7
        tr.build(s, acted, alpha)
        ref.store_round(s, acted)
        s_, c_ = np.full(int(acted.sum()), s), np.flatnonzero(acted)
        td = rng.normal(size=len(s_)).astype(np.float32)
        tr.update(s_, c_, td, alpha, EPS32)
        ref.update(s_, c_, td)
    np.testing.assert_allclose(tr.leaves(), ref.leaf, rtol=1e-14, atol=0)
    np.testing.assert_allclose(tr.prio.cpu().numpy(), [ref.max_prio, ref.min_prio], rtol=0, atol=0)
    tr.check_internal_nodes(exact=False)
    leaves = tr.leaves()
    roots = tr.t[:, -1].cpu().numpy()
    for s in range(R):
        assert abs(roots[s] - math.fsum(leaves[s])) <= 1e-12 * math.fsum(leaves[s])
    ref.leaf[:] = leaves                                                    # same leaves: compare the search alone
    first, n = 1, 3
    slots = (first + np.arange(n)) % R
    u = rng.random(20000)
    got = tr.sample(u, first, n)
    want = ref.sample(u, slots)
    flat = leaves[slots].reshape(-1)
    S = np.cumsum(flat)
    T = S[-1]
    v = u * T
    k = np.searchsorted(S, v)
    near = (np.abs(S[np.minimum(k, len(S) - 1)] - v) <= 1e-9 * T) | (np.abs(S[np.maximum(k - 1, 0)] - v) <= 1e-9 * T)
    assert near.mean() < 0.01
    far = ~near
    np.testing.assert_array_equal(got[0][far], want[0][far])
    np.testing.assert_array_equal(got[1][far], want[1][far])
    assert (got[2] > 0).all()


def test_per_leaf_frequencies_follow_the_priorities():
    """2^22 samples over 3 usable slots of 10 cells; chi-square of the per-leaf counts against M * leaf / T, rejected
    below a p-value of 1e-6 (a fixed seed, so the outcome is deterministic)."""
    from scipy.stats import chi2
    rng = np.random.default_rng(13)
    R, B, N = 4, 2, 5
    tr, ref = _dyadic_ring(rng, R, B, N, p_acted=0.7)
    first, n = 2, 3
    slots = (first + np.arange(n)) % R
    M = 1 << 22
    g = torch.Generator(device="cuda")
    g.manual_seed(123)
    u = torch.rand(M, dtype=torch.float64, device="cuda", generator=g)
    s, c, v = tr.sample(u, first, n)
    flat = ref.leaf[slots].reshape(-1)
    order = np.full(R, -1)
    order[slots] = np.arange(n)
    assert (order[s] >= 0).all()
    idx = order[s] * (B * N) + c
    counts = np.bincount(idx, minlength=len(flat)).astype(np.float64)
    assert counts[flat == 0].sum() == 0
    exp = M * flat / flat.sum()
    keep = flat > 0
    stat = float((((counts - exp) ** 2)[keep] / exp[keep]).sum())
    assert stat < chi2.isf(1e-6, int(keep.sum()) - 1), stat


def _synthetic_round(rng, B, N, p=0.5):
    obs = torch.zeros(B, N, 8, dtype=torch.float32, device="cuda")
    active = torch.as_tensor(rng.random((B, N)) < p, dtype=torch.uint8, device="cuda")
    act = torch.as_tensor(rng.integers(0, 2, size=(B, N)), dtype=torch.int8, device="cuda")
    rew = torch.as_tensor(rng.normal(size=(B, N)), dtype=torch.float64, device="cuda")
    term = torch.as_tensor(rng.random((B, N)) < 0.3, dtype=torch.uint8, device="cuda")
    return obs, active, act, rew, term


def test_unupdated_priorities_sample_like_the_uniform_ring_with_unit_weights_and_no_host_sync():
    from melissa_b200.replay import DevicePrioritizedReplay, DeviceReplay
    rng = np.random.default_rng(14)
    B, N, R, n_step = 16, 20, 6, 2
    per = DevicePrioritizedReplay(B, N, R, alpha=0.6, beta=0.4, seed=3)
    uni = DeviceReplay(B, N, R, seed=4)
    for r in range(2 * R + 1):
        obs, active, act, rew, term = _synthetic_round(rng, B, N, p=0.1 if r == 2 * R - 3 else 0.5)
        for rep in (per, uni):
            rep.begin_round(obs, active)
            rep.end_round(act, rew, term)
    M = 1 << 20
    rho_p, ep_p, ag_p = per.sample_indices(M, n_step)
    rho_u, _, _ = uni.sample_indices(M, n_step)
    first, n = per._usable_rounds(n_step)
    usable = (first + np.arange(n)) % R
    fp = np.bincount(rho_p.cpu().numpy(), minlength=R) / M
    fu = np.bincount(rho_u.cpu().numpy(), minlength=R) / M
    cnt = np.where(np.isin(np.arange(R), usable), per.counts.cpu().numpy(), 0).astype(np.float64)
    np.testing.assert_allclose(fp, cnt / cnt.sum(), atol=3e-3)
    np.testing.assert_allclose(fp, fu, atol=5e-3)
    assert (per.flags[rho_p.long(), ep_p.long(), ag_p.long()] & 1).all()
    got = per.gather(rho_p[:4096], ep_p[:4096], ag_p[:4096], n_step, 0.99)
    assert (got["weight"] == 1.0).all() and got["weight"].dtype == torch.float32
    # after the first sample nothing synchronises with the host
    rounds = [_synthetic_round(rng, B, N) for _ in range(R + 1)]
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for obs, active, act, rew, term in rounds:
            per.begin_round(obs, active)
            per.end_round(act, rew, term)
            rho, ep, ag = per.sample_indices(4096, n_step)
            b = per.gather(rho, ep, ag, n_step, 0.99)
            per.update_weight((rho, ep, ag), b["returns"])
    finally:
        torch.cuda.set_sync_debug_mode(0)
    with pytest.raises(ValueError, match="bootstrap frame"):
        per.sample_indices(16, R)
    with pytest.raises(ValueError):
        per.set_beta(-0.1)
    with pytest.raises(ValueError):
        per.update_weight((rho, ep, ag), b["returns"][:-1])


def test_sampling_refuses_an_empty_ring():
    from melissa_b200.replay import DevicePrioritizedReplay
    per = DevicePrioritizedReplay(4, 3, 4, alpha=0.6, beta=0.4)
    with pytest.raises(RuntimeError, match="not enough rounds"):
        per.sample_indices(8, 1)
    obs = torch.zeros(4, 3, 8, device="cuda")
    for _ in range(3):
        per.begin_round(obs, torch.zeros(4, 3, dtype=torch.uint8, device="cuda"))
        per.end_round(torch.zeros(4, 3, dtype=torch.int8, device="cuda"), torch.zeros(4, 3, dtype=torch.float64, device="cuda"),
                      torch.zeros(4, 3, dtype=torch.uint8, device="cuda"))
    with pytest.raises(RuntimeError, match="no transitions"):
        per.sample_indices(8, 1)


# ---------------------------------------------------------------------------------------------- end to end
DUELING = lambda: ({"hidden_sizes": [128, 128]}, {"hidden_sizes": [128, 128]})
EN, EB, EP, ER = 20, 64, 512, 6


class _Lockstep:
    """Collector over a prioritized ring of ER rounds, run in lockstep with the oracle environment (the pattern of
    tests/test_training_replay_gpu.py); the reference ring stores the oracle's active sets."""

    def __init__(self, policy_cls, n_step, alpha, beta, seed=3):
        from melissa_b200.batched_env import BatchedGraphEnv, ResetTuplesDevice
        from melissa_b200.data_parallel import FlatParameters, FusedAdam
        from melissa_b200.networks import NETWORKS
        from melissa_b200.policy import BatchedCollector, MultiAgentSharedPolicy
        from melissa_b200.replay import DevicePrioritizedReplay
        self.pool = GraphPool.synthetic(EN, 8, first_seed=seed)
        self.gi, self.src, self.inter, self.scr = reset_chain.episode_pool(seed, EP, EN, 8)[:4]
        torch.manual_seed(seed)
        net = NETWORKS["l_dgn"](5, 128, 2, 4, EN, dueling_param=DUELING(), device="cuda").cuda()
        self.pol = policy_cls(net, FusedAdam(FlatParameters(net)), discount_factor=0.99, estimation_step=n_step,
                              target_update_freq=0, eps=0.1)
        self.replay = DevicePrioritizedReplay(EB, EN, ER, alpha=alpha, beta=beta, seed=1)
        self.ref = PrioritizedRingReference(ER, EB * EN, alpha=alpha, beta=beta)
        self.col = BatchedCollector(agents_num=EN, policy=MultiAgentSharedPolicy(self.pol, [str(i) for i in range(EN)]),
                                    env=BatchedGraphEnv(EB, EN, self.pool, want_info=True), buffer=self.replay,
                                    exploration_noise=True,
                                    tuples=ResetTuplesDevice(self.gi, self.src, self.inter, self.scr, EN, "cuda", pool_size=8))
        self.o = BatchedEnvOracle(EB, EN)
        g = self.gi[:EB]
        self.o.reset(np.arange(EB), self.pool.adj[g], self.pool.pos[g], self.src[:EB], self.inter[:EB], self.scr[:EB])
        self.n_resets = np.ones(EB, dtype=np.int64)
        self.head = 0

    def rounds(self, n):
        for _ in range(n):
            self.ref.store_round(self.head % ER, self.o.active)
            self.col.iterate(0.2)
            self.o.step(self.col.act.cpu().numpy())
            ids = np.flatnonzero(~self.o.active.any(axis=1))
            if len(ids):
                t = (ids + self.n_resets[ids] * EB) % EP
                self.o.reset(ids, self.pool.adj[self.gi[t]], self.pool.pos[self.gi[t]], self.src[t], self.inter[t], self.scr[t])
                self.n_resets[ids] += 1
            self.head += 1
        assert self.replay.head == self.head


@pytest.mark.parametrize("policy", ["dqn", "dgn"])
def test_policy_update_weights_loss_and_new_priorities_match_the_reference(policy):
    from melissa_b200.policy import DGNPolicy, DQNPolicy
    alpha, beta, n_step, M = 0.6, 0.4, 2, 2048
    ls = _Lockstep(DQNPolicy if policy == "dqn" else DGNPolicy, n_step, alpha, beta)
    pol, replay, ref = ls.pol, ls.replay, ls.ref
    seen = {}
    learn = pol.learn

    def spy(batch, **kw):
        seen["w"] = batch["weight"].detach().double().cpu().numpy()
        out = learn(batch, **kw)
        seen["td"] = batch.weight.detach().cpu().numpy()
        seen["idx"] = (batch.rho.cpu().numpy().astype(np.int64),
                       (batch.ep.long() * EN + batch.agent.long()).cpu().numpy())
        return out
    pol.learn = spy
    ls.rounds(ER - 1)
    for phase in range(4):
        np.testing.assert_allclose(replay.tree[:, :EB * EN].cpu().numpy(), ref.leaf, rtol=1e-12, atol=0)
        out = pol.update(M, replay)
        s, c = seen["idx"]
        assert (ref.leaf[s, c] > 0).all()
        first, n = replay._usable_rounds(n_step)
        assert np.isin(s, (first + np.arange(n)) % ER).all()
        w_ref = ref.weights(s, c)
        np.testing.assert_allclose(seen["w"], w_ref, rtol=1e-6)
        td = seen["td"].astype(np.float64)
        np.testing.assert_allclose(float(out["loss"]), np.mean(td ** 2 * w_ref), rtol=1e-5)
        ref.update(s, c, seen["td"])
        np.testing.assert_allclose(replay.tree[:, :EB * EN].cpu().numpy(), ref.leaf, rtol=1e-12, atol=0)
        np.testing.assert_allclose(replay.prio.cpu().numpy(), [ref.max_prio, ref.min_prio], rtol=1e-15)
        key = s * (EB * EN) + c
        last = len(key) - 1 - np.unique(key[::-1], return_index=True)[1]       # the last occurrence of every leaf
        np.testing.assert_allclose(replay.tree[s[last], c[last]].cpu().numpy(),
                                   (np.abs(td[last]) + EPS32) ** alpha, rtol=1e-12)
        if phase == 1:                                   # set_beta: the weights follow the formula with the new beta
            replay.set_beta(0.9)
            ref.beta = 0.9
            rho, ep, ag = replay.sample_indices(M, n_step)
            w = replay.gather(rho, ep, ag, n_step, 0.99)["weight"].double().cpu().numpy()
            cell = (ep.long() * EN + ag.long()).cpu().numpy()
            leaf = ref.leaf[rho.cpu().numpy(), cell]
            want = (leaf / ref.min_prio) ** -0.9
            np.testing.assert_allclose(w, want / want.max(), rtol=1e-6)
        ls.rounds(3)                                     # new rounds start at the raised max_prio^alpha
