"""GPU: the device replay ring across wrap-around -- stored rows, n-step returns and, above all, the bootstrap
observations, checked against oracle/env_oracle.py driven in lockstep and indexed by ABSOLUTE round, so that a frame
read from the wrong ring slot (never written yet, or overwritten) cannot match by construction."""
import numpy as np
import pytest
import torch

from melissa_b200 import reset_chain
from melissa_b200.topology import GraphPool
from oracle import train_oracle
from oracle.env_oracle import BatchedEnvOracle

pytestmark = pytest.mark.gpu
DUELING = lambda: ({"hidden_sizes": [128, 128]}, {"hidden_sizes": [128, 128]})
N, B, P, R = 20, 64, 512, 6


def _drive(n_rounds, n_step, seed=3):
    """Collector + replay ring of R rounds, run n_rounds in lockstep with the oracle environment.  -> (setup dict,
    history): per absolute round a < n_rounds obs[a] (what the agents decided on), acted, act, rew, term; obs has one
    more entry, the observation of round n_rounds (not stored in the ring yet)."""
    from melissa_b200.batched_env import BatchedGraphEnv, ResetTuplesDevice
    from melissa_b200.data_parallel import FlatParameters, FusedAdam
    from melissa_b200.networks import NETWORKS
    from melissa_b200.policy import BatchedCollector, DQNPolicy, MultiAgentSharedPolicy
    from melissa_b200.replay import DeviceReplay
    pool = GraphPool.synthetic(N, 8, first_seed=seed)
    gi, src, inter, scr = reset_chain.episode_pool(seed, P, N, 8)[:4]
    torch.manual_seed(seed)
    net = NETWORKS["l_dgn"](5, 128, 2, 4, N, dueling_param=DUELING(), device="cuda").cuda()
    pol = DQNPolicy(net, FusedAdam(FlatParameters(net)), discount_factor=0.99, estimation_step=n_step, target_update_freq=0, eps=0.1)
    replay = DeviceReplay(B, N, R, seed=1)
    col = BatchedCollector(agents_num=N, policy=MultiAgentSharedPolicy(pol, [str(i) for i in range(N)]),
                           env=BatchedGraphEnv(B, N, pool, want_info=True), buffer=replay, exploration_noise=True,
                           tuples=ResetTuplesDevice(gi, src, inter, scr, N, "cuda", pool_size=8))
    o = BatchedEnvOracle(B, N)
    o.reset(np.arange(B), pool.adj[gi[:B]], pool.pos[gi[:B]], src[:B], inter[:B], scr[:B])
    n_resets = np.ones(B, dtype=np.int64)
    h = {k: [] for k in ("obs", "acted", "act", "rew", "term")}
    for _ in range(n_rounds):
        h["obs"].append(o.obs().copy())
        h["acted"].append(o.active.copy())
        col.iterate(0.2)
        acts = col.act.cpu().numpy()
        res = o.step(acts)
        h["act"].append(acts.copy())
        h["rew"].append(np.asarray(res[1]).copy())
        h["term"].append(np.asarray(res[3]).astype(bool))
        ids = np.flatnonzero(~o.active.any(axis=1))
        if len(ids):                                            # the device recycles reset tuples in the same order
            t = (ids + n_resets[ids] * B) % P
            o.reset(ids, pool.adj[gi[t]], pool.pos[gi[t]], src[t], inter[t], scr[t])
            n_resets[ids] += 1
    h["obs"].append(o.obs().copy())
    assert replay.head == n_rounds and int(replay.pack_errors.item()) == 0
    return dict(pol=pol, replay=replay), {k: np.stack(v) for k, v in h.items()}


def _absolute(slot, head):
    """Absolute round stored in ring slot ``slot`` at ``head``: the a with head - R <= a < head and a % R == slot."""
    return head - R + (slot - (head - R)) % R


@pytest.mark.parametrize("n_rounds", [R - 1, 3 * R + 2], ids=["before_wrap", "after_wrap"])
@pytest.mark.parametrize("n_step", [1, 2, 3, 4])
def test_replay_rows_returns_and_bootstrap_frames_match_the_oracle(n_step, n_rounds):
    """Every sampled transition: its row bit for bit, action, n-step return (tianshou's recursion on the agent's chain),
    whether it bootstraps, and the bootstrap row = the observation the agent saw at absolute round rho + n_step.  Then
    process_fn's targets end to end, and uniform sampling over the stored transitions of the usable rounds."""
    from melissa_b200.policy import Batch
    s, h = _drive(n_rounds, n_step)
    pol, replay = s["pol"], s["replay"]
    head = replay.head
    M = 20000
    for gamma in (0.99, 0.5):
        rho, ep, ag = replay.sample_indices(M, n_step)
        raw = replay.gather(rho, ep, ag, n_step, gamma)
        a0 = _absolute(rho.cpu().numpy().astype(np.int64), head)
        e, a = ep.cpu().numpy().astype(np.int64), ag.cpu().numpy().astype(np.int64)
        assert h["acted"][a0, e, a].all()                                               # stored transitions only
        rows = raw["obs"].cpu().numpy()
        np.testing.assert_array_equal(rows[:, :-1].view(np.uint32), h["obs"][a0, e].reshape(M, -1).view(np.uint32))
        np.testing.assert_array_equal(rows[:, -1], a.astype(np.float32))
        np.testing.assert_array_equal(raw["act"].cpu().numpy(), h["act"][a0, e, a])
        # returns and the bootstrap decision: the agent's own chain (its tianshou sub-buffer) from a0 on, built from
        # absolute rounds up to the bootstrap round (stored by construction of the usable rounds)
        ret, boot = raw["returns"].cpu().numpy(), raw["boot_round"].cpu().numpy()
        want_ret, alive = np.empty(M), np.empty(M, dtype=bool)
        memo = {}
        for m in range(M):
            key = (int(a0[m]), int(e[m]), int(a[m]))
            if key not in memo:
                r0, ee, aa = key
                rew_c, term_c = [], []
                for rr in range(r0, min(r0 + n_step, head - 1) + 1):
                    assert h["acted"][rr, ee, aa]
                    rew_c.append(h["rew"][rr, ee, aa]); term_c.append(bool(h["term"][rr, ee, aa]))
                    if term_c[-1]:
                        break
                memo[key] = (train_oracle.nstep_return_chain(np.array(rew_c), np.array(term_c), 0, n_step, gamma, lambda t: 0.0),
                             not any(term_c[:n_step]))
            want_ret[m], alive[m] = memo[key]
        np.testing.assert_allclose(ret, want_ret, rtol=1e-6, atol=1e-6)
        np.testing.assert_array_equal(boot >= 0, alive)
        if n_step == 4:
            assert not alive.any()                              # TTL 4 decisions: a 4-step window always ends the chain
        else:
            assert alive.any()
            ab = a0[alive] + n_step                                 # absolute bootstrap round
            np.testing.assert_array_equal(boot[alive], ab % R)
            got = replay.rows_at(raw["boot_round"][alive], raw["ep"][alive], raw["agent"][alive]).cpu().numpy()
            want = h["obs"][ab, e[alive]].reshape(len(ab), -1)
            bad = np.flatnonzero((got[:, :-1].view(np.uint32) != want.view(np.uint32)).any(axis=1))
            if len(bad):
                zero = int((got[bad, :-1] == 0).all(axis=1).sum())
                old = ab[bad] - R
                stale = int(sum(old[i] >= 0 and np.array_equal(got[b, :-1], h["obs"][old[i], e[alive][b]].reshape(-1))
                                for i, b in enumerate(bad)))
                pytest.fail(f"{len(bad)} of {len(ab)} bootstrap rows differ from the observation at round rho + n_step "
                            f"(all-zero frames: {zero}, frames of R = {R} rounds earlier: {stale}; "
                            f"newest stored round {head - 1}, bad bootstrap rounds {sorted(set(ab[bad].tolist()))})")
            np.testing.assert_array_equal(got[:, -1], a[alive].astype(np.float32))
            # end to end: process_fn's target = reward sum + gamma^n * Q_target(row of the oracle observation)
            want_rows = torch.as_tensor(np.concatenate([want, a[alive, None].astype(np.float32)], axis=1), device="cuda")
            tq = pol._target_q(want_rows).double().cpu().numpy()
            target = want_ret.copy()
            target[alive] += gamma ** n_step * tq
            b = pol.process_fn(Batch(raw), replay)
            np.testing.assert_allclose(b.returns.cpu().numpy(), target, rtol=1e-6, atol=1e-6)
        assert a0.max() == head - 1 - n_step, "sampled a round whose window or bootstrap frame is not stored, or never the newest usable one"
    # uniform over the stored transitions of the usable rounds (coarse check per ring slot)
    rho, _, _ = replay.sample_indices(200000, n_step)
    freq = np.bincount(rho.cpu().numpy(), minlength=R) / 200000
    cnt = replay.counts.cpu().numpy().astype(np.float64)
    usable = np.array([0 <= _absolute(sl, head) <= head - 1 - n_step for sl in range(R)])
    want = np.where(usable, cnt, 0.0)
    np.testing.assert_allclose(freq, want / want.sum(), atol=0.01)
    # a ring that cannot hold a window plus its bootstrap frame refuses to sample
    for n in (R, R + 1):
        with pytest.raises(ValueError, match="bootstrap frame"):
            replay.sample_indices(16, n)
