"""CPU: host logic of the training path -- the differentiable forward against the oracle, the Batch container, the flat
parameter / gradient buffers and the world-size-2 (gloo) gradient all-reduce."""
import os

import numpy as np
import pytest
import torch

from oracle import net_oracle as no
from oracle import train_oracle

DUELING = lambda: ({"hidden_sizes": [128, 128]}, {"hidden_sizes": [128, 128]})


def _rows(N, bs, seed):
    rng = np.random.default_rng(seed)
    om = np.zeros((bs, N, 8), dtype=np.float32)
    om[:, :, :2] = rng.random((bs, N, 2)) * (0.6 if N <= 20 else 1.0)
    om[:, :, 2] = rng.integers(0, 8, size=(bs, N))
    om[:, :, 3] = rng.integers(0, 5, size=(bs, N))
    om[:, :, 4:7] = rng.integers(0, 2, size=(bs, N, 3))
    om[:, :, 7] = rng.random((bs, N)) >= 0.3
    ctrl = rng.integers(0, N, size=bs).astype(np.float32)
    ctrl[0] = -3.0
    return torch.as_tensor(np.concatenate([om.reshape(bs, -1), ctrl[:, None]], axis=1))


@pytest.mark.parametrize("kind,kw", [("l_dgn", {}), ("dgn_r", {}), ("hl_dgn", {"aggregator": "max"}),
                                      ("hl_dgn", {"aggregator": "mean"}), ("hl_dgn", {"aggregator": "add"})])
@pytest.mark.parametrize("N", [12, 50])
def test_autograd_forward_equals_oracle_and_reaches_every_parameter(kind, kw, N):
    from melissa_b200.networks import NETWORKS
    from melissa_b200.networks.autograd import q_values
    sd = no.init_state_dict(kind, seed=5)
    rows = _rows(N, 12, 3)
    want = no.FORWARDS[kind](sd, rows, N, **kw)
    m = NETWORKS[kind](5, 128, 2, 4, N, dueling_param=DUELING(), device="cpu", **kw)
    m.load_state_dict(sd)
    got = q_values(m, rows)
    assert float((got - want).abs().max()) <= 1e-5 * max(1.0, float(want.abs().max()))
    got.pow(2).sum().backward()
    for name, p in m.named_parameters():
        if "lin_skip" in name:
            assert p.grad is None                       # constructed by PyG, never used (SURVEY B.4)
        else:
            assert p.grad is not None and torch.isfinite(p.grad).all(), name


@pytest.mark.parametrize("kind,kw", [("l_dgn", {}), ("dgn_r", {}), ("hl_dgn", {"aggregator": "add"})])
def test_network_without_dueling_heads_on_the_host(kind, kw):
    """dueling_param=None builds ``out_linear`` (l_dgn.py:88-90,149): checkpoint keys, the differentiable forward against
    the oracle, gradients reaching it."""
    from melissa_b200.networks import NETWORKS
    from melissa_b200.networks.autograd import q_values
    N = 12
    sd = no.init_state_dict(kind, seed=6, dueling=False)
    assert "out_linear.weight" in sd and not any(k.startswith(("Q.", "V.")) for k in sd)
    m = NETWORKS[kind](5, 128, 2, 4, N, dueling_param=None, device="cpu", **kw)
    assert sorted(m.state_dict()) == sorted(sd)
    m.load_state_dict(sd)
    rows = _rows(N, 10, 4)
    want = no.FORWARDS[kind](sd, rows, N, **kw)
    got = q_values(m, rows)
    assert float((got - want).abs().max()) <= 1e-5 * max(1.0, float(want.abs().max()))
    got.pow(2).sum().backward()
    assert m.out_linear.weight.grad is not None and float(m.out_linear.weight.grad.abs().sum()) > 0


def test_batch_container_operations():
    from melissa_b200.policy import Batch
    b = Batch(obs=Batch(obs=np.arange(12).reshape(4, 3), mask=np.ones((4, 2), bool), agent_id=np.array(["0", "1", "0", "2"])),
              info={"env_id": np.arange(4)}, rew=np.zeros((4, 3)))
    assert len(b) == 4 and b.obs.agent_id[3] == "2" and b["info"].env_id[2] == 2
    sub = b[np.array([0, 2])]
    assert len(sub) == 2 and sub.obs.obs.tolist() == [[0, 1, 2], [6, 7, 8]] and sub.info.env_id.tolist() == [0, 2]
    b.update(act=np.array([1, 0, 1, 0]))
    assert b.get("act").sum() == 2 and b.get("missing", 7) == 7 and b.pop("rew").shape == (4, 3) and "rew" not in b
    c = Batch.cat([sub, sub])
    assert len(c) == 4 and c.obs.agent_id.tolist() == ["0", "0", "0", "0"]
    assert Batch().is_empty() and not b.is_empty()


def test_adam_restatement_is_pinned_on_torch_optim_adam():
    """The reference optimises with torch.optim.Adam (l_dgn.py:66) and torch IS installed here, so this part of
    oracle/train_oracle.py is pinned on the real thing: 25 steps in float64 with and without weight decay."""
    rng = np.random.default_rng(3)
    for wd in (0.0, 0.01):
        p0 = rng.standard_normal(257)
        grads = [rng.standard_normal(257) * (10.0 ** rng.integers(-3, 2)) for _ in range(25)]
        want_p = torch.tensor(p0, dtype=torch.float64, requires_grad=True)
        opt = torch.optim.Adam([want_p], lr=1e-3, weight_decay=wd)
        for g in grads:
            want_p.grad = torch.tensor(g, dtype=torch.float64)
            opt.step()
        got = train_oracle.adam_reference(p0, grads, lr=1e-3, weight_decay=wd)
        np.testing.assert_allclose(got, want_p.detach().numpy(), rtol=1e-12, atol=1e-14)


def test_nstep_restatement_on_hand_cases():
    rew = np.array([1.0, 2.0, 3.0, 4.0])
    term = np.array([False, False, False, True])
    g = 0.9
    # window reaches the terminal: pure discounted sum, no bootstrap
    assert train_oracle.nstep_return_chain(rew, term, 0, 4, g, lambda t: 100.0) == pytest.approx(1 + g * 2 + g * g * 3 + g ** 3 * 4)
    assert train_oracle.nstep_return_chain(rew, term, 2, 4, g, lambda t: 100.0) == pytest.approx(3 + g * 4)
    # shorter window: bootstrap from the observation after the window's last transition
    assert train_oracle.nstep_return_chain(rew, term, 0, 2, g, lambda t: 10.0 * t) == pytest.approx(1 + g * 2 + g * g * 10.0)
    assert train_oracle.nstep_return_chain(rew, term, 3, 1, g, lambda t: 10.0) == pytest.approx(4.0)


def test_adam_restatement_continues_from_a_given_state():
    rng = np.random.default_rng(4)
    p0 = rng.standard_normal(33)
    grads = [rng.standard_normal(33) for _ in range(5)]
    want = train_oracle.adam_reference(p0, grads, lr=1e-2, weight_decay=0.01)
    p, m, v = train_oracle.adam_reference(p0, grads[:2], lr=1e-2, weight_decay=0.01, state=(np.zeros(33), np.zeros(33), 0))
    for t, g in enumerate(grads[2:], start=2):
        p, m, v = train_oracle.adam_reference(p, [g], lr=1e-2, weight_decay=0.01, state=(m, v, t))
    np.testing.assert_allclose(p, want, rtol=1e-14, atol=1e-15)


def _dense_lists(edges):
    """Fixed-capacity lists (self first, then the sources in index order) of every node of dense masks [B, i, j]."""
    B, N, _ = edges.shape
    cap = 36
    tgt, src, cnt = [], [], []
    for b in range(B):
        for i in range(N):
            s = [i] + torch.nonzero(edges[b, i]).flatten().tolist()
            tgt.append(b * N + i)
            src.append([b * N + j for j in s] + [0] * (cap - len(s)))
            cnt.append(len(s))
    as_i32 = lambda x: torch.tensor(x, dtype=torch.int32)
    return as_i32(tgt), as_i32(src), as_i32(cnt)


@pytest.mark.parametrize("heads", [1, 3, 4])
@pytest.mark.parametrize("seed", [0, 1])
def test_edge_references_equal_the_dense_oracle_convolutions(heads, seed):
    """oracle/train_oracle.py's list-based float64 references of the training edge kernels against net_oracle's dense
    GATv2Conv / TransformerConv (bias removed) on random radius graphs, isolated nodes included."""
    torch.manual_seed(seed)
    B, N, D, HC = 3, 12, 16, heads * 128
    pos = torch.rand(B, N, 2, dtype=torch.float64) * 0.5
    pos[0, 0] = 5.0                                                # an isolated node
    edges = no.radius_graph_mask(pos)
    x = torch.randn(B, N, D, dtype=torch.float64)
    w = lambda *s: torch.randn(*s, dtype=torch.float64) * 0.3
    sd = {"c.lin_l.weight": w(HC, D), "c.lin_l.bias": w(HC), "c.lin_r.weight": w(HC, D), "c.lin_r.bias": w(HC),
          "c.att": w(1, heads, 128), "c.bias": torch.zeros(HC, dtype=torch.float64),
          "c.lin_query.weight": w(HC, D), "c.lin_query.bias": w(HC), "c.lin_key.weight": w(HC, D), "c.lin_key.bias": w(HC),
          "c.lin_value.weight": w(HC, D), "c.lin_value.bias": w(HC)}
    lin = lambda k: torch.nn.functional.linear(x, sd[f"c.{k}.weight"], sd[f"c.{k}.bias"]).reshape(B * N, HC)
    tgt, src, cnt = _dense_lists(edges)
    want = no.gatv2_conv(sd, "c", x, edges, heads).reshape(B * N, HC)
    got, alpha = train_oracle.gatv2_edge_reference(lin("lin_l"), lin("lin_r"), sd["c.att"].view(-1), tgt, src, cnt, heads)
    torch.testing.assert_close(got, want, rtol=1e-12, atol=1e-12)
    torch.testing.assert_close(alpha.sum(1), torch.ones(B * N, heads, dtype=torch.float64), rtol=1e-12, atol=1e-12)
    want = no.transformer_conv(sd, "c", x, edges, heads).reshape(B * N, HC)
    got, alpha = train_oracle.transformer_edge_reference(lin("lin_query"), lin("lin_key"), lin("lin_value"), tgt, src, cnt, heads)
    torch.testing.assert_close(got, want, rtol=1e-12, atol=1e-12)
    assert float(got[0].abs().max()) == 0.0 and float(alpha[:, 0].abs().max()) == 0.0   # isolated node; entry 0 skipped


def _dp_worker(rank, world, port, out_dir):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from melissa_b200.data_parallel import FlatParameters, GradSync
    from melissa_b200.networks import LDGNNetwork
    from melissa_b200.networks.autograd import q_values
    N = 12
    torch.manual_seed(100 + rank)                          # different initial weights per rank on purpose
    net = LDGNNetwork(5, 128, 2, 4, N, dueling_param=DUELING(), device="cpu")
    flat = FlatParameters(net)
    sync = GradSync(flat.grad)
    sync.broadcast_parameters(flat.flat, src=0)
    start = flat.flat.clone()
    opt = torch.optim.Adam([flat.flat], lr=1e-3)
    flat.flat.grad = flat.grad                             # the flat buffer is the single optimised tensor
    grads = []
    for it in range(3):
        rows = _rows(N, 6, 10 * rank + it)                 # every rank its own minibatch
        flat.zero_grad()
        loss = q_values(net, rows).pow(2).mean()
        loss.backward()
        local = flat.grad.clone()
        sync.start()
        sync.finish()
        flat.grad.mul_(sync.grad_scale)
        grads.append((local, flat.grad.clone()))
        opt.step()
    torch.save({"start": start, "end": flat.flat.clone(), "grads": grads, "w": net.conv2.lin_l.weight.detach().clone()},
               os.path.join(out_dir, f"dp{rank}.pt"))
    dist.destroy_process_group()


def test_world_size_2_gradient_allreduce_keeps_weights_identical(tmp_path):
    import torch.multiprocessing as mp
    port = 29600 + (os.getpid() % 1000)
    mp.spawn(_dp_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = torch.load(tmp_path / "dp0.pt"), torch.load(tmp_path / "dp1.pt")
    assert torch.equal(r0["start"], r1["start"])                       # broadcast from rank 0
    assert torch.equal(r0["end"], r1["end"]) and not torch.equal(r0["start"], r0["end"])
    for (l0, a0), (l1, a1) in zip(r0["grads"], r1["grads"]):
        assert not torch.equal(l0, l1)                                 # different minibatches ...
        assert torch.equal(a0, a1)                                     # ... one averaged gradient
        assert torch.allclose(a0, (l0 + l1) / 2, rtol=0, atol=1e-7)
    assert torch.equal(r0["w"], r1["w"])                               # parameters are views of the flat buffer
