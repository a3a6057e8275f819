"""GPU: the device episode stream (EpisodeStream, mls_episode_sample, mls_env_reset_sampled / mls_env_step_sampled).

1. The round kernel plays exactly the sampler's tuples: a stream environment and a pool environment fed the
   materialised tuples (row b + r*B = episode r of slot b) agree bit for bit on every output of every round.
2. The draws have the training-reset distribution (chi-square / z-tests with fixed seeds, thresholds set once).
3. Sub-batch views, captured CUDA graphs and rank offsets draw what they should; duplicates stay at chance.
4. The collector and the trainer run on a stream, past the 4*B episodes of the default pool."""
import math

import numpy as np
import pytest
import torch
from scipy import stats

from episode_stream_util import expected_duplicate_pairs, k_probabilities
from melissa_b200 import _lib
from melissa_b200.topology import GraphPool

pytestmark = pytest.mark.gpu

P_MIN = 1e-4           # chi-square p-value floor
Z_MAX = 5.0            # |z| ceiling of the normal-approximation checks


def _bits(words: torch.Tensor, n_nodes: int) -> torch.Tensor:
    """int32 [n, W] bitmasks -> bool [n, N] (on the device)."""
    sh = torch.arange(32, device=words.device, dtype=torch.int32)
    b = (words.unsqueeze(-1) >> sh) & 1
    return b.reshape(words.shape[0], -1)[:, :n_nodes].bool()


def _pool(N, G, seed):
    side = None if N in (20, 50) else min(1.0, (N / 50.0) ** 0.5)
    return GraphPool.synthetic(N, G, first_seed=seed, side=side)


def _snapshot(env):
    """Every output and every state array of the environment, bit patterns of the floats."""
    out = dict(obs=env.obs.view(torch.int32), reward=env.reward.view(torch.int64), active=env.active,
               terminated=env.terminated, done=env.done, info=env.info_buf, episode=env.episode, node=env.node,
               recv_count=env.recv_count, rewards_sum=env.rewards_sum.view(torch.int64))
    if env.dynamic:
        out.update(adj=env.adj, pos=env.pos.view(torch.int64))
    if env.recv_from is not None:
        out.update(recv_from=env.recv_from)
    return {k: t.clone() for k, t in out.items()}


CASES = [(20, 128, False, None, 0.0), (50, 128, False, None, 0.0), (100, 64, False, None, 0.0), (200, 32, False, None, 0.0),
         (20, 128, True, None, 0.0), (50, 64, True, None, 0.0), (100, 32, True, None, 0.0),
         (20, 128, False, "mpr", 0.4), (50, 64, True, "mpr", 0.4)]


@pytest.mark.parametrize("N,B,dynamic,heuristic,ratio", CASES)
def test_round_kernel_plays_exactly_the_sampled_tuples(N, B, dynamic, heuristic, ratio):
    from melissa_b200.batched_env import BatchedGraphEnv, EpisodeStream, ResetTuplesDevice
    G, rounds = 12, 30
    pool = _pool(N, G + 4, 300 + N)
    stream = EpisodeStream(N, G, seed=1234 + N, scripted_agents_ratio=ratio)
    mk = lambda: BatchedGraphEnv(B, N, pool, dynamic_graph=dynamic, heuristic=heuristic, want_info=True)
    env = mk()
    env.reset(stream)
    env.set_recycling(stream)
    rng = np.random.default_rng(N)
    actions, snaps, restarts = [], [_snapshot(env)], []
    for t in range(rounds):
        a = rng.integers(0, 2, size=(B, N)).astype(np.int8)
        r_before = env.episode[:, _lib.MLS_EP_N_RESETS].cpu().numpy()
        env.step(a)
        done = env.done.cpu().numpy().astype(bool)
        restarts += [(int(b), int(r_before[b])) for b in np.flatnonzero(done)]
        actions.append(a)
        snaps.append(_snapshot(env))
    assert len(restarts) > B // 2, "too few restarts to test the recycle branch"
    n_resets = env.episode[:, _lib.MLS_EP_N_RESETS].cpu().numpy()
    assert sorted(restarts) == sorted((b, r) for b in range(B) for r in range(1, n_resets[b]))
    R = int(n_resets.max())
    tup = stream.sample(np.tile(np.arange(B), R), np.repeat(np.arange(R), B))    # row b + r*B
    first = ResetTuplesDevice.__new__(ResetTuplesDevice)
    first.count = B
    for k in ("graph_index", "source", "interested", "scripted"):
        setattr(first, k, getattr(tup, k)[:B])
    ref = mk()
    ref.reset(first)
    ref.set_recycling(tup)
    for t in range(rounds + 1):
        if t:
            ref.step(actions[t - 1])
        got = _snapshot(ref)
        for name, x in snaps[t].items():
            assert torch.equal(x, got[name]), f"round {t}: {name} differs between the stream and the materialised pool"


def _draw(N, G, n, seed, ratio=0.0, slot_offset=0, slots=None, eps=None):
    from melissa_b200.batched_env import EpisodeStream
    s = EpisodeStream(N, G, seed, scripted_agents_ratio=ratio, slot_offset=slot_offset)
    if slots is None:
        slots, eps = np.arange(n) % 4096, np.arange(n) // 4096
    t = s.sample(slots, eps)
    return t, _bits(t.interested, N), _bits(t.scripted, N)


def _chi2(counts, probs, n):
    exp = probs * n
    keep = exp >= 5
    assert counts[~keep].sum() <= max(5.0, 5 * exp[~keep].sum()), "mass where the law has (almost) none"
    return stats.chisquare(counts[keep], exp[keep] * counts[keep].sum() / exp[keep].sum()).pvalue


@pytest.mark.parametrize("G", [1024, 1000])
def test_graph_source_and_density_follow_the_training_law(G):
    N, n = 50, 1 << 20
    t, inter, _ = _draw(N, G, n, seed=11 + G)
    gi = t.graph_index.cpu().numpy()
    src = t.source.cpu().numpy()
    k = inter.sum(1).cpu().numpy()
    assert gi.min() >= 0 and gi.max() < G and src.min() >= 0 and src.max() < N
    assert _chi2(np.bincount(gi, minlength=G), np.full(G, 1.0 / G), n) > P_MIN
    assert _chi2(np.bincount(src, minlength=N), np.full(N, 1.0 / N), n) > P_MIN
    assert _chi2(np.bincount(k, minlength=N + 1), k_probabilities(N), n) > P_MIN


def _z(obs, exp, var):
    return (obs - exp) / np.sqrt(np.maximum(var, 1e-12))


def test_interest_sets_are_uniform_k_subsets_independent_of_the_source():
    N, n = 50, 1 << 20
    t, inter, _ = _draw(N, 64, n, seed=5)
    X = inter.double()
    k = X.sum(1)
    p1 = (k / N).cpu().numpy()
    p2 = (k * (k - 1) / (N * (N - 1))).cpu().numpy()
    # per-node inclusion: node i is in with probability k/N
    node = X.sum(0).cpu().numpy()
    assert np.abs(_z(node, p1.sum(), (p1 * (1 - p1)).sum())).max() < Z_MAX
    # pairwise inclusion: i and j are both in with probability k(k-1)/(N(N-1))
    pair = (X.T @ X).cpu().numpy()
    iu = np.triu_indices(N, 1)
    assert np.abs(_z(pair[iu], p2.sum(), (p2 * (1 - p2)).sum())).max() < Z_MAX
    # per k: every node equally likely (chi-square over the nodes, for the well-populated k)
    kk = k.long().cpu().numpy()
    Xc = inter.cpu().numpy()
    for m in (5, 12, 25, 38, 49):
        rows = Xc[kk == m]
        assert len(rows) > 1000
        c = rows.sum(0)
        assert stats.chisquare(c).pvalue > P_MIN, m
    # the source is interested with probability k/N (the two draws are independent)
    src = t.source.long()
    hit = X.gather(1, src[:, None]).squeeze(1).sum().item()
    assert abs(_z(hit, p1.sum(), (p1 * (1 - p1)).sum())) < Z_MAX


def test_scripted_sets_have_the_drawn_size_without_the_source():
    N, n = 50, 1 << 18
    from melissa_b200.batched_env import scripted_count
    ns = scripted_count(0.4, N)
    t, inter, scr = _draw(N, 8, n, seed=21, ratio=0.4)
    cnt = scr.sum(1).cpu().numpy()
    src = t.source.long()
    src_scr = scr.long().gather(1, src[:, None]).squeeze(1).bool()
    assert not src_scr.any(), "the source is never scripted when ratio < 1"
    assert set(np.unique(cnt).tolist()) <= {ns - 1, ns}
    # one fewer exactly when the source was among the drawn n_scripted: probability n_scripted / N
    short = int((cnt == ns - 1).sum())
    p = ns / N
    assert abs(_z(short, n * p, n * p * (1 - p))) < Z_MAX
    # per-node inclusion of the scripted set (before the source is removed every node has n_scripted/N)
    node = scr.double().sum(0).cpu().numpy()
    s_node = np.bincount(t.source.cpu().numpy(), minlength=N)
    # P(i scripted) = P(i drawn) * P(i not source) = ns/N * (N-1)/N; conditional on the sources actually drawn:
    exp = ns / N * (n - s_node)
    assert np.abs(_z(node, exp, exp * (1 - ns / N))).max() < Z_MAX
    # independent of the interest set: P(i interested and scripted) = E[k]/N * P(i scripted)
    both = (scr & inter).double().sum().item()
    exp_both = (inter.double().sum(1) * scr.double().sum(1) / N).sum().item()     # sum over episodes of k * |S| / N
    assert abs(both - exp_both) / math.sqrt(exp_both) < Z_MAX
    _, _, scr0 = _draw(N, 8, 4096, seed=21, ratio=0.0)
    assert not scr0.any()
    _, _, scr1 = _draw(N, 8, 4096, seed=21, ratio=1.0)
    assert scr1.all(), "ratio = 1: every node is scripted, the source included"


def test_sub_batch_views_draw_what_the_full_batch_draws():
    from melissa_b200.batched_env import BatchedGraphEnv, EpisodeStream
    N, B = 20, 256
    pool = _pool(N, 8, 44)
    stream = EpisodeStream(N, 8, seed=3)
    a, b = (BatchedGraphEnv(B, N, pool, dynamic_graph=True, want_info=True) for _ in range(2))
    for e in (a, b):
        e.reset(stream)
        e.set_recycling(stream)
    rng = np.random.default_rng(0)
    for t in range(25):
        act = torch.as_tensor(rng.integers(0, 2, size=(B, N)).astype(np.int8), device="cuda")
        a.step_device(act)
        b.step_device_slice(act[: B // 2], 0, B // 2)
        b.step_device_slice(act[B // 2:], B // 2, B)
        sa, sb = _snapshot(a), _snapshot(b)
        for name in sa:
            assert torch.equal(sa[name], sb[name]), f"round {t}: {name}"
    assert int(a.episode[:, _lib.MLS_EP_N_RESETS].min()) >= 2


def test_captured_rollout_replays_fresh_sampled_episodes():
    from melissa_b200.batched_env import BatchedGraphEnv, EpisodeStream
    from melissa_b200.rollout import Rollout
    N, B = 50, 512
    pool = _pool(N, 16, 8)
    stream = EpisodeStream(N, 16, seed=17)
    env = BatchedGraphEnv(B, N, pool)
    ro = Rollout(env, None)
    ro.start(stream)
    ro.capture()
    for _ in range(40):
        ro.round()
    torch.cuda.synchronize()
    ep = env.episode.cpu().numpy()
    r = ep[:, _lib.MLS_EP_N_RESETS]
    assert r.min() >= 3, "every slot restarted under replay"
    t = stream.sample(np.arange(B), r - 1)                         # the episode each slot plays now
    np.testing.assert_array_equal(ep[:, _lib.MLS_EP_GRAPH], t.graph_index.cpu().numpy())
    np.testing.assert_array_equal(ep[:, _lib.MLS_EP_SOURCE], t.source.cpu().numpy())
    fl = env.flags()
    np.testing.assert_array_equal(fl["interested"], _bits(t.interested, N).cpu().numpy())
    np.testing.assert_array_equal(fl["scripted"], _bits(t.scripted, N).cpu().numpy())


def _rows(t, N):
    return np.concatenate([t.graph_index.cpu().numpy()[:, None], t.source.cpu().numpy()[:, None],
                           t.interested.cpu().numpy().reshape(t.count, -1), t.scripted.cpu().numpy().reshape(t.count, -1)],
                          axis=1)


def test_rank_offsets_give_disjoint_sequences_and_duplicates_stay_at_chance():
    from melissa_b200.sharding import rank_slot_offset
    N, G, B, R = 20, 8, 512, 64
    slots, eps = np.tile(np.arange(B), R), np.repeat(np.arange(R), B)
    seqs = []
    for rank in range(2):
        t, _, _ = _draw(N, G, B * R, seed=99, slot_offset=rank_slot_offset(rank, B), slots=slots, eps=eps)
        seqs.append(_rows(t, N).reshape(R, B, -1).transpose(1, 0, 2).reshape(B, -1))     # [slot][episodes ...]
    common = {s.tobytes() for s in seqs[0]} & {s.tobytes() for s in seqs[1]}
    assert not common, "two ranks play the same episode sequence"
    # the key is the global slot: rank 1's slot b is slot B + b of rank 0's numbering
    t0, _, _ = _draw(N, G, B, seed=99, slots=np.arange(B, 2 * B), eps=np.zeros(B, dtype=int))
    t1, _, _ = _draw(N, G, B, seed=99, slot_offset=B, slots=np.arange(B), eps=np.zeros(B, dtype=int))
    np.testing.assert_array_equal(_rows(t0, N), _rows(t1, N))
    # duplicate tuples among the 64 episodes x B slots of one rank: no more than independent draws give
    rows = seqs[0].reshape(B * R, -1)
    _, cnt = np.unique(rows, axis=0, return_counts=True)
    pairs = float((cnt * (cnt - 1) // 2).sum())
    lam = expected_duplicate_pairs(B * R, N, G)
    assert pairs <= lam + Z_MAX * math.sqrt(lam) + 5, (pairs, lam)


def test_collector_and_trainer_run_on_a_stream():
    from melissa_b200.batched_env import BatchedGraphEnv, EpisodeStream
    from melissa_b200.data_parallel import FlatParameters, FusedAdam
    from melissa_b200.networks import NETWORKS
    from melissa_b200.policy import BatchedCollector, DQNPolicy, MultiAgentSharedPolicy
    from melissa_b200.replay import DeviceReplay
    from melissa_b200.trainer import OffpolicyTrainer
    N, B = 20, 64
    pool = _pool(N, 8, 3)
    torch.manual_seed(3)
    net = NETWORKS["l_dgn"](5, 128, 2, 4, N, dueling_param=({"hidden_sizes": [128, 128]}, {"hidden_sizes": [128, 128]}),
                            device="cuda").cuda()
    net.set_precision("bf16")
    pol = DQNPolicy(net, FusedAdam(FlatParameters(net), lr=1e-3), discount_factor=0.99, estimation_step=4,
                    target_update_freq=4, eps=0.3)
    masp = MultiAgentSharedPolicy(pol, [str(i) for i in range(N)])
    env = BatchedGraphEnv(B, N, pool, want_info=True)
    stream = EpisodeStream(N, 8, seed=5)
    col = BatchedCollector(agents_num=N, policy=masp, env=env, buffer=DeviceReplay(B, N, 12, seed=1),
                           exploration_noise=True, tuples=stream)
    res = col.collect(n_episode=4 * B + 1)
    assert res.n_collected_episodes > 4 * B and np.isfinite(res.returns).all()
    r = env.episode[:, _lib.MLS_EP_N_RESETS].cpu().numpy()
    assert r.max() > 4
    tr = OffpolicyTrainer(policy=masp, train_collector=col, max_epoch=1, step_per_epoch=3000, step_per_collect=1000,
                          batch_size=256, update_per_step=0.003)
    out = tr.run()
    assert out["env_step"] >= 3000 and out["gradient_step"] >= 3 and np.isfinite(out["loss"])
