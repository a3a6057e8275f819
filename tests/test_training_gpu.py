"""GPU: training step of the data-parallel DQN path -- packed frames, device replay with the MultiAgentCollector
completion rule, n-step returns, the fused Adam kernel, DQNPolicy / DGNPolicy.learn, and the tianshou-shaped
policy / collector surfaces.  Checkers: oracle/env_oracle.py driven in lockstep (pinned to the reference) and
oracle/train_oracle.py (tianshou's published n-step / Adam arithmetic, parity unpinned)."""
import numpy as np
import pytest
import torch

from melissa_b200 import reset_chain
from melissa_b200.topology import GraphPool
from oracle import net_oracle as no
from oracle import train_oracle
from oracle.env_oracle import BatchedEnvOracle

pytestmark = pytest.mark.gpu
DUELING = lambda: ({"hidden_sizes": [128, 128]}, {"hidden_sizes": [128, 128]})


def _setup(kind="l_dgn", N=20, B=64, P=512, seed=3, ring=12, n_step=4, target_freq=0, policy_cls=None, lr=1e-3, heads=4, **kw):
    from melissa_b200.batched_env import BatchedGraphEnv, ResetTuplesDevice
    from melissa_b200.data_parallel import FlatParameters, FusedAdam
    from melissa_b200.networks import NETWORKS
    from melissa_b200.policy import BatchedCollector, DQNPolicy, MultiAgentSharedPolicy
    from melissa_b200.replay import DeviceReplay
    pool = GraphPool.synthetic(N, 8, first_seed=seed)
    tup = reset_chain.episode_pool(seed, P, N, 8)
    torch.manual_seed(seed)
    net = NETWORKS[kind](5, 128, 2, heads, N, dueling_param=DUELING(), device="cuda", **kw).cuda()
    flat = FlatParameters(net)
    optim = FusedAdam(flat, lr=lr)
    pol = (policy_cls or DQNPolicy)(net, optim, discount_factor=0.99, estimation_step=n_step, target_update_freq=target_freq, eps=0.1)
    env = BatchedGraphEnv(B, N, pool, want_info=True)
    replay = DeviceReplay(B, N, ring, seed=1)
    masp = MultiAgentSharedPolicy(pol, [str(i) for i in range(N)])
    col = BatchedCollector(agents_num=N, policy=masp, env=env, buffer=replay, exploration_noise=True,
                           tuples=ResetTuplesDevice(*tup[:4], N, "cuda", pool_size=8))
    return dict(pool=pool, tup=tup, net=net, flat=flat, optim=optim, pol=pol, masp=masp, env=env, replay=replay, col=col, N=N, B=B, P=P)


def test_obs_pack_unpack_is_lossless_and_counts_bad_rows():
    from melissa_b200 import _lib
    s = _setup()
    env, L = s["env"], _lib.lib()
    for _ in range(5):
        s["col"].iterate(0.3)
    rows = env.B * env.N
    packed = torch.zeros(rows, 12, dtype=torch.uint8, device="cuda")
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    _lib.check(L.mls_obs_pack(env.obs.data_ptr(), rows, packed.data_ptr(), err.data_ptr(), _lib.current_stream_ptr()))
    out = torch.full((env.B, env.N * 8), -7.0, dtype=torch.float32, device="cuda")
    _lib.check(L.mls_obs_unpack(packed.data_ptr(), None, None, env.N, env.B, env.N * 8, out.data_ptr(), _lib.current_stream_ptr()))
    assert int(err.item()) == 0
    assert torch.equal(out.view(env.B, env.N, 8).view(torch.int32), env.obs.view(torch.int32))     # bit for bit
    bad = env.obs.clone()
    bad[0, 0, 3] = 0.5
    _lib.check(L.mls_obs_pack(bad.data_ptr(), rows, packed.data_ptr(), err.data_ptr(), _lib.current_stream_ptr()))
    assert int(err.item()) == 1
    # agent rows: frame selection + controlling index in the last column
    frames = torch.tensor([3, 0, 3], dtype=torch.int64, device="cuda")
    agents = torch.tensor([5, 1, 19], dtype=torch.int32, device="cuda")
    _lib.check(L.mls_obs_pack(env.obs.data_ptr(), rows, packed.data_ptr(), None, _lib.current_stream_ptr()))
    ar = torch.zeros(3, env.N * 8 + 1, dtype=torch.float32, device="cuda")
    _lib.check(L.mls_obs_unpack(packed.data_ptr(), frames.data_ptr(), agents.data_ptr(), env.N, 3, env.N * 8 + 1, ar.data_ptr(),
                                _lib.current_stream_ptr()))
    assert torch.equal(ar[:, :-1], env.obs.view(env.B, -1)[frames]) and ar[:, -1].tolist() == [5.0, 1.0, 19.0]


def test_replay_stores_what_the_multi_agent_collector_would_and_samples_only_windows_with_a_stored_bootstrap_frame():
    """The oracle environment is driven in lockstep with the device's actions.  Every agent transition of a round must be
    in the ring with: the observation the agent decided on, its action, the reward of the world step that followed,
    terminated exactly when its TTL ended -- the completion rule of multi_agent_collector.py:240-308 -- and the sampled
    n-step returns must equal tianshou's compute_nstep_return on the agent's own chain.  Sampling never starts a window
    in the newest n_step rounds: the bootstrap observation of round rho + n_step must already be stored."""
    N, B, P, R = 20, 64, 512, 12
    s = _setup(N=N, B=B, P=P, ring=R)
    env, replay, col, pool = s["env"], s["replay"], s["col"], s["pool"]
    gi, src, inter, scr = s["tup"][:4]
    o = BatchedEnvOracle(B, N)
    o.reset(np.arange(B), pool.adj[gi[:B]], pool.pos[gi[:B]], src[:B], inter[:B], scr[:B])
    n_resets = np.ones(B, dtype=np.int64)
    hist = []                                                   # per round: obs, acted, act, reward, terminated
    for r in range(R):
        obs_before, acted = o.obs().copy(), o.active.copy()
        col.iterate(0.2)
        acts = col.act.cpu().numpy()
        res = o.step(acts)
        rew, term = np.asarray(res[1]), np.asarray(res[3]).astype(bool)
        hist.append((obs_before, acted, acts.copy(), rew.copy(), term.copy()))
        ids = np.flatnonzero(~o.active.any(axis=1))
        if len(ids):
            t = (ids + n_resets[ids] * B) % P
            o.reset(ids, pool.adj[gi[t]], pool.pos[gi[t]], src[t], inter[t], scr[t])
            n_resets[ids] += 1
    assert replay.head == R and int(replay.pack_errors.item()) == 0
    flags = replay.flags.cpu().numpy()
    for r, (obs_b, acted, acts, rew, term) in enumerate(hist):
        np.testing.assert_array_equal((flags[r] & 1).astype(bool), acted)
        np.testing.assert_array_equal((flags[r] & 2).astype(bool), term & acted)
        np.testing.assert_array_equal(replay.act[r].cpu().numpy()[acted], acts[acted])
        np.testing.assert_array_equal(replay.rew[r].cpu().numpy()[acted].view(np.uint64), rew[acted].view(np.uint64))
        assert int(replay.counts[r].item()) == int(acted.sum())
    assert len(replay) == sum(int(h[1].sum()) for h in hist)
    # sampling: uniform over complete windows, rows = the reference's agent observation
    for n_step in (4, 2, 1):
        rho, ep, ag = replay.sample_indices(4000, n_step)
        b = replay.gather(rho, ep, ag, n_step, 0.99)
        rho_n, ep_n, ag_n = rho.cpu().numpy(), ep.cpu().numpy(), ag.cpu().numpy()
        assert rho_n.max() == R - 1 - n_step and len(np.unique(rho_n)) > 1     # window + bootstrap frame stored
        rows, ret, boot = b["obs"].cpu().numpy(), b["returns"].cpu().numpy(), b["boot_round"].cpu().numpy()
        for m in range(0, 4000, 37):
            r0, e, a = int(rho_n[m]), int(ep_n[m]), int(ag_n[m])
            assert hist[r0][1][e, a]                                             # a stored transition
            np.testing.assert_array_equal(rows[m, :-1].view(np.uint32), hist[r0][0][e].reshape(-1).view(np.uint32))
            assert rows[m, -1] == a and int(b["act"][m].item()) == int(hist[r0][2][e, a])
            # the agent's own chain from r0 on (its tianshou sub-buffer): consecutive rounds until terminated
            rew_c, term_c = [], []
            rr = r0
            while rr < R:
                assert hist[rr][1][e, a]
                rew_c.append(hist[rr][3][e, a]); term_c.append(bool(hist[rr][4][e, a]))
                if term_c[-1]:
                    break
                rr += 1
            want = train_oracle.nstep_return_chain(np.array(rew_c), np.array(term_c), 0, n_step, 0.99, lambda t: 0.0)
            assert ret[m] == pytest.approx(want, rel=1e-6, abs=1e-6)
            alive = not any(term_c[:n_step])
            assert (boot[m] >= 0) == alive and (not alive or boot[m] == (r0 + n_step) % R)
    # uniformity: every stored transition whose window and bootstrap frame are stored is equally likely (coarse check
    # per ring round; with n_step 1 that is every round but the newest)
    rho, _, _ = replay.sample_indices(200000, 1)
    freq = np.bincount(rho.cpu().numpy(), minlength=R) / 200000
    cnt = replay.counts.cpu().numpy().astype(np.float64)
    cnt[R - 1] = 0.0
    np.testing.assert_allclose(freq, cnt / cnt.sum(), atol=0.01)


def test_fused_adam_matches_torch_adam():
    from melissa_b200.data_parallel import FlatParameters, FusedAdam
    torch.manual_seed(0)
    lin = torch.nn.Sequential(torch.nn.Linear(37, 53), torch.nn.Linear(53, 11)).cuda()
    ref = torch.nn.Sequential(torch.nn.Linear(37, 53), torch.nn.Linear(53, 11)).cuda()
    ref.load_state_dict(lin.state_dict())
    flat = FlatParameters(lin)
    opt, opt_ref = FusedAdam(flat, lr=3e-3, weight_decay=0.01), torch.optim.Adam(ref.parameters(), lr=3e-3, weight_decay=0.01)
    p0 = flat.flat.double().cpu().numpy()
    grads = []
    for it in range(12):
        x = torch.randn(64, 37, device="cuda")
        opt.zero_grad(); opt_ref.zero_grad()
        lin(x).pow(2).mean().backward()
        ref(x).pow(2).mean().backward()
        grads.append(flat.grad.double().cpu().numpy().copy())
        opt.step(); opt_ref.step()
    got = torch.cat([p.detach().reshape(-1) for p in lin.parameters()])
    want = torch.cat([p.detach().reshape(-1) for p in ref.parameters()])
    assert float((got - want).abs().max()) <= 2e-6
    assert all(p.data_ptr() == flat.flat.data_ptr() + 4 * o for p, o in zip(lin.parameters(), flat.offsets))   # views of the flat buffer
    del p0, grads
    # grad_scale = 1 / world: half the gradient
    flat2 = FlatParameters(torch.nn.Linear(5, 3).cuda())
    o2 = FusedAdam(flat2, lr=1e-2)
    flat2.grad.fill_(2.0)
    before = flat2.flat.clone()
    o2.step(grad_scale=0.5)
    want = train_oracle.adam_reference(before.cpu().numpy(), [np.ones(flat2.numel)], lr=1e-2)
    assert flat2.numel % 16 == 0
    np.testing.assert_allclose(flat2.flat.cpu().numpy(), want, rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("kind,kw", [("l_dgn", {}), ("dgn_r", {}), ("hl_dgn", {"aggregator": "max"})])
def test_training_forward_agrees_with_the_rollout_kernels(kind, kw):
    """The autograd forward used by learn() and the CUDA forward used by the rollout must be the same function of the
    parameters: fp32 kernels within 1e-5, bf16 kernels within the stated bf16 tolerance."""
    from melissa_b200.networks.autograd import q_values
    s = _setup(kind=kind, N=20, **kw)
    for _ in range(6):
        s["col"].iterate(0.3)
    env, net = s["env"], s["net"]
    b_idx, a_idx = torch.nonzero(env.active, as_tuple=True)
    rows = torch.cat([env.obs.view(env.B, -1)[b_idx], a_idx.float()[:, None]], dim=1)[:300]
    with torch.no_grad():
        q_t = q_values(net, rows)
    q_c, _ = net(rows)
    scale = max(1.0, float(q_t.abs().max()))
    assert float((q_c - q_t).abs().max()) <= 1e-5 * scale
    net.set_precision("bf16")
    q_b, _ = net(rows)
    assert float((q_b - q_t).abs().max()) <= 1e-2 * scale


def _rows(s, n, synthetic):
    """Agent-observation rows: from a short rollout, or synthetic (one complete-graph sample, one isolated controlling
    node)."""
    if synthetic:
        return train_oracle.agent_rows(s["N"], n, seed=s["N"] + n, complete=(0,), isolated=(1,)).cuda()
    for _ in range(6):
        s["col"].iterate(0.3)
    env = s["env"]
    b_idx, a_idx = torch.nonzero(env.active, as_tuple=True)
    return torch.cat([env.obs.view(env.B, -1)[b_idx], a_idx.float()[:, None]], dim=1)[:n]


@pytest.mark.parametrize("agg,synthetic,heads", [("max", False, 4), ("mean", False, 4), ("add", False, 4),
                                                 ("max", True, 1), ("add", True, 2), ("mean", True, 4)],
                         ids=["max", "mean", "add", "max-synthetic-h1", "add-synthetic-h2", "mean-synthetic-h4"])
def test_fused_hl_dgn_training_forward_backward_matches_the_torch_path(agg, synthetic, heads):
    from melissa_b200.networks import autograd as ag
    s = _setup(kind="hl_dgn", N=20, aggregator=agg, heads=heads)
    net = s["net"]
    rows = _rows(s, 200, synthetic)
    assert ag.fused_training_available(net, rows)
    target = torch.linspace(-1, 1, rows.shape[0], device=rows.device)
    res = []
    for fn in (ag.q_values_torch, ag.q_values_hl_dgn_fused):
        s["optim"].zero_grad()
        q = fn(net, rows)
        ((q[:, 0] - target).pow(2).mean() + q[:, 1].mean()).backward()
        res.append((q.detach().clone(), {k: p.grad.detach().clone() for k, p in net.named_parameters()}))
    (q_t, g_t), (q_f, g_f) = res
    assert float((q_t - q_f).abs().max()) <= 1e-5 * max(1.0, float(q_t.abs().max()))
    for k in g_t:
        assert float((g_t[k] - g_f[k]).abs().max()) <= 1e-4 * max(float(g_t[k].abs().max()), 1e-6), k


@pytest.mark.parametrize("kind,N,synthetic,heads", [("l_dgn", 20, False, 4), ("l_dgn", 50, False, 4), ("dgn_r", 20, False, 4),
                                                    ("dgn_r", 50, False, 4), ("l_dgn", 50, True, 1), ("l_dgn", 20, True, 2),
                                                    ("dgn_r", 50, True, 2), ("dgn_r", 20, True, 4)],
                         ids=["l_dgn-20", "l_dgn-50", "dgn_r-20", "dgn_r-50", "l_dgn-50-synthetic-h1", "l_dgn-20-synthetic-h2",
                              "dgn_r-50-synthetic-h2", "dgn_r-20-synthetic-h4"])
def test_fused_gatv2_training_kernels_match_the_torch_autograd_path(kind, N, synthetic, heads):
    """mls_train_lists + mls_gatv2_edge_fwd / _bwd (the L-DGN training forward / backward) against the plain torch-op
    formulation of the same math (autograd.q_values_torch, itself pinned to the oracle on the CPU): Q-values to 1e-5 and
    every parameter gradient to 1e-4 of the gradient's scale (fp32, different summation orders and atomics)."""
    from melissa_b200.networks import autograd as ag
    s = _setup(kind=kind, N=N, heads=heads)
    net = s["net"]
    rows = _rows(s, 400, synthetic)
    assert rows.shape[0] >= 50 and ag.fused_training_available(net, rows)
    target = torch.linspace(-1, 1, rows.shape[0], device=rows.device)
    grads = []
    for fn in (ag.q_values_torch, ag.q_values_l_dgn_fused):
        s["optim"].zero_grad()
        q = fn(net, rows)
        ((q[:, 0] - target).pow(2).mean() + q[:, 1].mean()).backward()
        grads.append((q.detach().clone(), {k: p.grad.detach().clone() for k, p in net.named_parameters() if "lin_skip" not in k}))
    (q_t, g_t), (q_f, g_f) = grads
    assert float((q_t - q_f).abs().max()) <= 1e-5 * max(1.0, float(q_t.abs().max()))
    assert set(g_t) == set(g_f)
    for k in g_t:
        scale = max(float(g_t[k].abs().max()), 1e-6)
        assert float((g_t[k] - g_f[k]).abs().max()) <= 1e-4 * scale, k
    # the edge lists themselves: slots of a sample = controlling node first, then its radius neighbours in index order
    slot_base, s1_cnt, tgt_row, src_row, src_cnt, used = ag.train_lists(rows, N)
    assert bool(used.bool()[tgt_row.long()].all())
    pos, _, _, ctrl = ag.split_rows(rows, N, net.input_dim)
    mask = ag.radius_mask(pos)
    for b in (0, rows.shape[0] // 2, rows.shape[0] - 1):
        c = int(ctrl[b])
        want = [c] + torch.nonzero(mask[b, c]).flatten().tolist()
        lo = int(slot_base[b])
        assert (tgt_row[lo:lo + int(s1_cnt[b])] - b * N).tolist() == want
        for k, i in enumerate(want):
            srcs = [i] + torch.nonzero(mask[b, i]).flatten().tolist()
            assert int(src_cnt[lo + k]) == len(srcs)
            assert (src_row[lo + k, :len(srcs)] - b * N).tolist() == srcs


def test_learn_reduces_td_error_and_refreshes_the_rollout_weights():
    s = _setup(N=20, B=128, ring=10, lr=5e-4)
    col, replay, pol, net = s["col"], s["replay"], s["pol"], s["net"]
    net.set_precision("bf16")
    for _ in range(10):
        col.iterate(0.5)
    from melissa_b200.policy import Batch
    rho, ep, ag = replay.sample_indices(2048, 4)
    fixed = replay.gather(rho, ep, ag, 4, 0.99)
    assert bool((fixed["boot_round"] < 0).all())             # TTL 4 decisions, n_step 4: the window always reaches the terminal
    q_before, _ = net(fixed["obs"])
    losses = []
    for it in range(25):
        out = pol.learn(Batch(fixed))
        losses.append(float(out["loss"]))
    assert losses[-1] < 0.85 * losses[0] and losses[12] < losses[0], losses
    assert pol._iter == 25 and s["optim"].step_count == 25
    # the bf16 rollout forward sees the new weights (prepared copy is re-packed on the version bump)
    q_after, _ = net.forward_graphs(s["env"].obs, s["env"].active, discrete_features=True, prepared=True)
    q_again, _ = net.forward_graphs(s["env"].obs, s["env"].active, discrete_features=True)
    assert torch.equal(q_after, q_again)
    q_now, _ = net(fixed["obs"])
    assert not torch.equal(q_now, q_before)
    # update() = sample + process_fn + learn
    out = s["masp"].update(512, replay)
    assert np.isfinite(float(out["loss"]))


def test_bootstrap_path_with_short_windows_and_target_network():
    s = _setup(N=20, B=64, ring=10, n_step=2, target_freq=3)
    col, replay, pol = s["col"], s["replay"], s["pol"]
    for _ in range(8):
        col.iterate(0.5)
    from melissa_b200.policy import Batch
    rho, ep, ag = replay.sample_indices(600, 2)
    raw = replay.gather(rho, ep, ag, 2, 0.99)
    alive = raw["boot_round"] >= 0
    assert bool(alive.any()) and bool((~alive).any())
    base = raw["returns"].clone()
    b = pol.process_fn(Batch(raw), replay)
    # double DQN on the bootstrap rows; that rows_at returns the observation of round rho + n_step is checked against
    # the oracle environment in test_training_replay_gpu.py
    rows = replay.rows_at(raw["boot_round"][alive], raw["ep"][alive], raw["agent"][alive])
    q_on, _ = pol.model(rows)
    q_old, _ = pol.model_old(rows)
    want = base.clone()
    want[alive] += 0.99 ** 2 * q_old.gather(1, q_on.argmax(1, keepdim=True)).squeeze(1)       # double DQN
    assert torch.allclose(b.returns, want, rtol=1e-6, atol=1e-6)
    assert torch.equal(b.returns[~alive], base[~alive])
    # target network follows the online one every target_update_freq learn() calls
    w_old = pol.model_old.conv2.lin_l.weight.clone()
    for it in range(4):
        pol.update(256, replay)
    assert not torch.equal(pol.model_old.conv2.lin_l.weight, w_old)
    assert not torch.equal(pol.model_old.conv2.lin_l.weight, pol.model.conv2.lin_l.weight)       # synced at iter 3, one more step since


def test_dgn_policy_sum_of_q_loss():
    """policies/dgn.py:22-71: per experience, the Q-values at the taken actions of all agents active in that round."""
    from melissa_b200.networks.autograd import q_values
    from melissa_b200.policy import Batch, DGNPolicy
    s = _setup(kind="dgn_r", N=12, B=32, ring=8, policy_cls=DGNPolicy, lr=0.0)
    col, replay, pol, net = s["col"], s["replay"], s["pol"], s["net"]
    for _ in range(8):
        col.iterate(0.5)
    rho, ep, ag = replay.sample_indices(24, 4)
    b = Batch(replay.gather(rho, ep, ag, 4, 0.99))
    b.rho = rho
    out = pol.learn(b, buffer=replay)
    want = []
    for m in range(24):
        r0, e = int(rho[m]), int(ep[m])
        acted = torch.nonzero(replay.flags[r0, e] & 1)[:, 0]
        rows = replay.rows_at(torch.full_like(acted, r0, dtype=torch.int32), torch.full_like(acted, e, dtype=torch.int32), acted.to(torch.int32))
        with torch.no_grad():
            q = q_values(net, rows)
        want.append(float(q.gather(1, replay.act[r0, e, acted].long()[:, None]).sum()))
    td = b.returns.cpu().numpy() - np.array(want)
    assert float(out["loss"]) == pytest.approx(float((td ** 2).mean()), rel=1e-4)
    np.testing.assert_allclose(b.weight.cpu().numpy(), td, rtol=1e-4, atol=1e-4)


def test_tianshou_shaped_policy_surface_follows_the_collector_call_sequence():
    """multi_agent_collector.py:150-200: ``result = policy(data, last_state)``; ``act = to_numpy(result.act)``;
    ``act = policy.exploration_noise(act, data)``; ``env.step(act)`` -- driven through the AEC facade (one agent
    observation at a time, as tianshou's PettingZooEnv presents them)."""
    from melissa_b200 import graph_env_v0, topology
    from melissa_b200.networks import LDGNNetwork
    from melissa_b200.policy import Batch, DQNPolicy, MultiAgentSharedPolicy, to_numpy
    N = 12
    env = graph_env_v0.env(graph=topology.make_connected_graph(N, 5), number_of_agents=N)
    sd = no.init_state_dict("l_dgn", seed=2)
    net = LDGNNetwork(5, 128, 2, 4, N, dueling_param=DUELING(), device="cuda")
    net.load_state_dict(sd)
    net = net.cuda()
    masp = MultiAgentSharedPolicy(DQNPolicy(net, None, 0.99, 4, 500, eps=0.0), env)
    assert masp.agents == [str(i) for i in range(N)]
    env.reset(seed=4)
    steps = 0
    while env.agents and steps < 60:
        agent = env.agent_selection
        ob = env.observe(agent)
        dead = env.terminations[agent] or env.truncations[agent]
        data = Batch(obs=Batch(agent_id=np.array([agent]), obs=ob["observation"][None], mask=(ob["action_mask"] == 1)[None]),
                     info=Batch(env_id=np.array([0])), rew=np.zeros((1, N)))
        result = masp(data, None)
        act = to_numpy(result.act)
        want_q = no.l_dgn_forward(sd, torch.as_tensor(ob["observation"][None]), N).numpy()
        assert np.abs(to_numpy(result.logits) - want_q).max() <= 1e-5 * max(1.0, np.abs(want_q).max())
        if abs(want_q[0, 1] - want_q[0, 0]) > 1e-4 and not dead:
            assert act[0] == int(want_q[0, 1] > want_q[0, 0])
        assert set(result.out.keys()) == set(masp.agents) and not result.out[agent].is_empty()
        masp.policy.set_eps(0.5)
        noisy = masp.exploration_noise(act.copy(), data, rng=np.random.default_rng(steps))
        masp.policy.set_eps(0.0)
        assert noisy.shape == act.shape and set(noisy.tolist()) <= {0, 1}
        assert masp.exploration_noise(act, data) is act
        env.step(None if dead else int(act[0]))
        steps += 1
    assert steps > N // 2
    # batched form: rows of several agents at once, grouped masking like the reference's per-id call
    rows = np.stack([env.observe(str(i))["observation"] for i in range(N)]) if env.agents else None
    ck = masp.policy.state_dict()
    assert "model.conv1.lin_l.weight" in ck and "model_old.conv1.lin_l.weight" in ck
    del rows


def test_offpolicy_trainer_runs_epochs_and_tracks_the_best_test_return():
    from melissa_b200.batched_env import BatchedGraphEnv, ResetTuplesDevice
    from melissa_b200.policy import BatchedCollector
    from melissa_b200.trainer import OffpolicyTrainer
    s = _setup(kind="hl_dgn", N=20, B=64, ring=12, aggregator="max", target_freq=4)
    s["net"].set_precision("bf16")
    gi, src, inter, scr, mv, dens = reset_chain.testing_episode_pool(64, 20, 8, num_test_episodes=10, seed=1)
    tenv = BatchedGraphEnv(16, 20, s["pool"], is_testing=True, want_info=True)
    tcol = BatchedCollector(agents_num=20, policy=s["masp"], env=tenv, tuples=ResetTuplesDevice(gi, src, inter, scr, 20, "cuda"))
    seen = []
    tr = OffpolicyTrainer(policy=s["masp"], train_collector=s["col"], test_collector=tcol, max_epoch=2, step_per_epoch=6000,
                          step_per_collect=1500, episode_per_test=20, batch_size=256, update_per_step=0.002,
                          train_fn=lambda e, st: s["pol"].set_eps(0.3), test_fn=lambda e, st: s["pol"].set_eps(0.001),
                          save_best_fn=lambda p: seen.append(1), test_in_train=False)
    out = tr.run()
    assert out["env_step"] >= 12000 and out["gradient_step"] >= 6 and np.isfinite(out["loss"])
    assert seen and np.isfinite(out["best_reward"]) and out["test_result"].n_collected_episodes >= 20
