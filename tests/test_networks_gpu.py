"""GPU parity of mls_dgn_forward (through the nn.Module mirrors and the C ABI) against the
pure-torch fp32 restatement in oracle/net_oracle.py.

Tolerance (fp32 mode), as BASELINE.json states: Q-values within 1e-5 relative.  Written
here as  max|q_cuda - q_ref| <= 1e-5 * max(1, max|q_ref|)  per batch, plus greedy-action
agreement wherever the reference's own margin |q1 - q0| exceeds 1e-4.
"""
import numpy as np
import pytest
import torch

from melissa_b200 import reset_chain
from melissa_b200.topology import GraphPool
from oracle import net_oracle as no

pytestmark = pytest.mark.gpu

DUELING = lambda: ({"hidden_sizes": [128, 128]}, {"hidden_sizes": [128, 128]})
REL_TOL = 1e-5


def _module(kind, N, sd, **kw):
    from melissa_b200.networks import NETWORKS
    m = NETWORKS[kind](5, 128, 2, 4, N, dueling_param=DUELING(), device="cuda", **kw)
    m.load_state_dict(sd)
    return m.cuda()


def _random_sd(kind, seed):
    sd = no.init_state_dict(kind, seed=seed)
    g = torch.Generator().manual_seed(seed + 1)
    for k in sd:                      # non-zero biases everywhere so a dropped bias cannot hide
        if k.endswith("bias"):
            sd[k] = (torch.rand(sd[k].shape, generator=g) - 0.5) * 0.2
    return sd


def _obs_matrix(N, B, seed, scripted_ratio=0.3):
    """Plausible obs matrices: positions of real synthetic graphs + random feature columns."""
    pool = GraphPool.synthetic(N, min(B, 8), first_seed=seed, side=None if N in (20, 50) else min(1.0, (N / 50) ** 0.5))
    rng = np.random.default_rng(seed)
    gi = rng.integers(0, len(pool), size=B)
    om = np.zeros((B, N, 8), dtype=np.float32)
    om[:, :, :2] = pool.pos[gi]
    om[:, :, 2] = pool.adj[gi].sum(2)
    om[:, :, 3] = rng.integers(0, 5, size=(B, N))
    om[:, :, 4] = rng.integers(0, 2, size=(B, N))
    om[:, :, 5] = rng.integers(0, 2, size=(B, N))
    om[:, :, 6] = rng.integers(0, 2, size=(B, N))
    om[:, :, 7] = rng.random((B, N)) >= scripted_ratio
    return om


def _assert_q(got, want, what=""):
    got, want = np.asarray(got, dtype=np.float64), np.asarray(want, dtype=np.float64)
    scale = max(1.0, float(np.abs(want).max()) if want.size else 1.0)
    err = float(np.abs(got - want).max()) if want.size else 0.0
    assert err <= REL_TOL * scale, f"{what}: max abs err {err:.3e} > {REL_TOL} * {scale:.3f}"


@pytest.mark.parametrize("kind,kw", [("l_dgn", {}), ("dgn_r", {}), ("hl_dgn", {"aggregator": "mean"})])
@pytest.mark.parametrize("precision", ["fp32", "bf16", "bf16-tables"])
@pytest.mark.parametrize("N,B", [(20, 48), (50, 500), (100, 40)])
def test_network_without_dueling_heads(kind, kw, precision, N, B):
    """dueling_param=None: q = out_linear(latent) (l_dgn.py:88-90,149), agent rows and obs-matrix batches, every precision.
    In bf16 the head reads a controlling node's conv1 columns from its x1 row: conv2's tensor-core path and the record-based
    conv1 kernel (N = 20, 50), the gather paths (N = 100)."""
    from melissa_b200.networks import NETWORKS
    sd = no.init_state_dict(kind, seed=31, dueling=False)
    sd["out_linear.bias"] = torch.tensor([0.3, -0.2])
    m = NETWORKS[kind](5, 128, 2, 4, N, dueling_param=None, device="cuda", **kw)
    assert sorted(m.state_dict()) == sorted(sd) and not m.use_dueling
    m.load_state_dict(sd)
    m = m.cuda().set_precision("fp32" if precision == "fp32" else "bf16")
    tol = REL_TOL if precision == "fp32" else BF16_TOL
    om = _obs_matrix(N, B, 13)
    cm = np.random.default_rng(3).random((B, N)) < 0.3
    want = no.forward_graphs(kind, sd, torch.as_tensor(om), torch.as_tensor(cm), N, **kw).numpy()
    q, act = m.forward_graphs(torch.as_tensor(om, device="cuda"), torch.as_tensor(cm, device="cuda").to(torch.uint8),
                              discrete_features=precision == "bf16-tables")
    q, act = q.cpu().numpy(), act.cpu().numpy()
    scale = max(1.0, float(np.abs(want).max()))
    assert float(np.abs(q - want).max()) <= tol * scale
    assert np.all(q[~cm] == 0) and np.all(act[~cm] == -1)
    np.testing.assert_array_equal(act[cm], (q[..., 1] > q[..., 0]).astype(np.int8)[cm])
    ctrl = np.random.default_rng(1).integers(0, N, size=B).astype(np.float32)
    rows = np.concatenate([om.reshape(B, -1), ctrl[:, None]], axis=1)
    want_r = no.FORWARDS[kind](sd, torch.as_tensor(rows), N, **kw).numpy()
    q_r, _ = m(rows)
    assert float(np.abs(q_r.cpu().numpy() - want_r).max()) <= tol * max(1.0, float(np.abs(want_r).max()))


@pytest.mark.parametrize("kind", ["l_dgn", "dgn_r", "hl_dgn"])
@pytest.mark.parametrize("N", [20, 50])
def test_forward_agent_rows_matches_oracle(kind, N):
    """Drop-in call: obs [bs, 8N+1] with the controlling index in the last column."""
    bs = 24
    sd = _random_sd(kind, 11)
    om = _obs_matrix(N, bs, 5)
    ctrl = np.random.default_rng(1).integers(0, N, size=bs).astype(np.float32)
    ctrl[0], ctrl[1] = -4.0, N + 7.0                      # clamped (common.py:63)
    rows = np.concatenate([om.reshape(bs, -1), ctrl[:, None]], axis=1)
    kw = dict(aggregator="max") if kind == "hl_dgn" else {}
    want = no.FORWARDS[kind](sd, torch.as_tensor(rows), N, **kw).numpy()
    m = _module(kind, N, sd, **kw)
    q, state = m(rows)                                    # numpy in, like tianshou feeds it
    assert q.shape == (bs, 2) and q.dtype == torch.float32
    _assert_q(q.cpu().numpy(), want, f"{kind} N={N}")
    q2, _ = m(torch.as_tensor(rows, device="cuda"))
    np.testing.assert_array_equal(q.cpu().numpy(), q2.cpu().numpy())
    with pytest.raises(ValueError):
        m(rows[:, :-1])
    with pytest.raises(ValueError):
        m(rows[0])


@pytest.mark.parametrize("kind,kw", [("l_dgn", {}), ("dgn_r", {}), ("hl_dgn", {"aggregator": "max"}),
                                      ("hl_dgn", {"aggregator": "mean"}), ("hl_dgn", {"aggregator": "add"})])
@pytest.mark.parametrize("N,B", [(20, 40), (50, 20)])
def test_forward_graphs_matches_oracle(kind, kw, N, B):
    sd = _random_sd(kind, 21)
    om = _obs_matrix(N, B, 9)
    rng = np.random.default_rng(2)
    cm = rng.random((B, N)) < 0.25
    cm[0] = False                                         # a graph without controlling agents
    cm[1] = True
    want = no.forward_graphs(kind, sd, torch.as_tensor(om), torch.as_tensor(cm), N, **kw).numpy()
    m = _module(kind, N, sd, **kw)
    q, act = m.forward_graphs(torch.as_tensor(om, device="cuda"), torch.as_tensor(cm, device="cuda").to(torch.uint8))
    q, act = q.cpu().numpy(), act.cpu().numpy()
    _assert_q(q, want, f"{kind} N={N}")
    assert np.all(q[~cm] == 0) and np.all(act[~cm] == -1)
    margin = np.abs(want[..., 1] - want[..., 0])
    sure = cm & (margin > 1e-4)
    np.testing.assert_array_equal(act[sure], (want[..., 1] > want[..., 0]).astype(np.int8)[sure])


def test_chunked_batches_and_many_graphs():
    """More graphs than one workspace chunk (32768 rows: 1638 graphs of 20 nodes): three passes, the last one partial;
    results must not depend on chunking.  The oracle checks graphs on both sides of each pass boundary."""
    import ctypes
    from melissa_b200 import _lib
    N, B = 20, 3400
    sd = _random_sd("l_dgn", 3)
    om = _obs_matrix(N, B, 13)
    cm = np.random.default_rng(3).random((B, N)) < 0.2
    m = _module("l_dgn", N, sd)
    gc = _lib.lib().mls_dgn_chunk_graphs(ctypes.byref(m._desc()), B)
    assert 2 * gc < B < 3 * gc, gc
    q, act = m.forward_graphs(torch.as_tensor(om, device="cuda"), torch.as_tensor(cm, device="cuda").to(torch.uint8))
    sel = np.r_[0:16, gc - 16:gc + 16, 2 * gc - 16:2 * gc + 16, B - 16:B]
    want = no.forward_graphs("l_dgn", sd, torch.as_tensor(om[sel]), torch.as_tensor(cm[sel]), N).numpy()
    _assert_q(q.cpu().numpy()[sel], want, "chunked")


@pytest.mark.parametrize("kind", ["l_dgn", "dgn_r"])
def test_degenerate_graphs(kind):
    """All nodes at one point (reference test fixture: pos=(0,0)) -> complete graph, capped at
    32 neighbours in index order for N > 33; plus fully isolated nodes."""
    for N in (12, 50):
        sd = _random_sd(kind, 31)
        B = 6
        om = _obs_matrix(N, B, 17)
        om[:3, :, :2] = 0.0
        om[3:, :, 0] = np.arange(N)[None, :] * 1.0       # far apart: no edges at all
        om[3:, :, 1] = 0.0
        cm = np.ones((B, N), dtype=bool)
        want = no.forward_graphs(kind, sd, torch.as_tensor(om), torch.as_tensor(cm), N).numpy()
        m = _module(kind, N, sd)
        q, _ = m.forward_graphs(torch.as_tensor(om, device="cuda"), torch.as_tensor(cm, device="cuda").to(torch.uint8))
        _assert_q(q.cpu().numpy(), want, f"{kind} degenerate N={N}")


def test_epsilon_greedy_with_host_fed_uniforms_and_philox():
    N, B = 20, 64
    sd = _random_sd("l_dgn", 41)
    om = _obs_matrix(N, B, 19)
    rng = np.random.default_rng(4)
    cm = rng.random((B, N)) < 0.5
    m = _module("l_dgn", N, sd)
    om_d, cm_d = torch.as_tensor(om, device="cuda"), torch.as_tensor(cm, device="cuda").to(torch.uint8)
    q, greedy = m.forward_graphs(om_d, cm_d)
    rand3 = rng.random((B * N, 3))
    eps = 0.3
    _, act = m.forward_graphs(om_d, cm_d, eps=eps, rand3=torch.as_tensor(rand3, device="cuda"))
    qn = q.cpu().numpy().reshape(B * N, 2)
    want = no.exploration_noise(no.dqn_act(qn, np.ones((B * N, 2))), eps, rand3[:, 0], rand3[:, 1:], np.ones((B * N, 2)))
    got = act.cpu().numpy().reshape(-1)
    flat = cm.reshape(-1)
    np.testing.assert_array_equal(got[flat], want[flat].astype(np.int8))
    np.testing.assert_array_equal(greedy.cpu().numpy().reshape(-1)[flat], no.dqn_act(qn, None)[flat].astype(np.int8))
    # Philox stream: deterministic in (seed, offset), explores at roughly the requested rate
    _, a1 = m.forward_graphs(om_d, cm_d, eps=0.5, philox_seed=9, philox_offset=1)
    _, a2 = m.forward_graphs(om_d, cm_d, eps=0.5, philox_seed=9, philox_offset=1)
    _, a3 = m.forward_graphs(om_d, cm_d, eps=0.5, philox_seed=9, philox_offset=2)
    assert torch.equal(a1, a2) and not torch.equal(a1, a3)
    changed = (a1 != greedy).cpu().numpy().reshape(-1)[flat].mean()
    assert 0.15 < changed < 0.35                          # eps/2 of the draws flip a binary action


def test_checkpoint_keys_and_cpu_module_fails_loudly():
    from melissa_b200 import _lib
    from melissa_b200.networks import LDGNNetwork
    m = LDGNNetwork(5, 128, 2, 4, 20, dueling_param=DUELING())
    assert set(m.state_dict()) == set(no.init_state_dict("l_dgn"))
    with pytest.raises(_lib.MelissaLibraryError):
        m(np.zeros((1, 161), dtype=np.float32))           # parameters on the CPU: no fallback


# ----------------------------------------------------------------------------- bf16 tensor-core path
# Stated tolerance of the bf16 mode (BASELINE.json: "or a stated bf16 tolerance"): activations and
# weights are rounded to bf16 (8 mantissa bits) between layers, accumulation is fp32.  Against the
# fp32 oracle:  max|q_bf16 - q_ref| <= 1e-2 * max(1, max|q_ref|)  and the greedy action agrees
# wherever the reference margin |q1 - q0| exceeds 2e-2 * max(1, max|q_ref|).
BF16_TOL = 1e-2


@pytest.mark.parametrize("kind,kw", [("l_dgn", {}), ("dgn_r", {}), ("hl_dgn", {"aggregator": "max"}),
                                      ("hl_dgn", {"aggregator": "mean"}), ("hl_dgn", {"aggregator": "add"})])
@pytest.mark.parametrize("N,B", [(20, 64), (50, 40), (12, 9)])
def test_bf16_forward_graphs_within_stated_tolerance(kind, kw, N, B):
    sd = _random_sd(kind, 51)
    om = _obs_matrix(N, B, 23)
    rng = np.random.default_rng(5)
    cm = rng.random((B, N)) < 0.3
    cm[0] = False
    cm[1] = True
    want = no.forward_graphs(kind, sd, torch.as_tensor(om), torch.as_tensor(cm), N, **kw).numpy()
    m = _module(kind, N, sd, **kw).set_precision("bf16")
    q, act = m.forward_graphs(torch.as_tensor(om, device="cuda"), torch.as_tensor(cm, device="cuda").to(torch.uint8))
    q, act = q.cpu().numpy(), act.cpu().numpy()
    scale = max(1.0, float(np.abs(want).max()))
    err = float(np.abs(q - want).max())
    print(f"bf16 {kind} N={N}: max abs err {err:.4f} (scale {scale:.2f})")
    assert err <= BF16_TOL * scale, f"{kind}: {err} > {BF16_TOL} * {scale}"
    assert np.all(q[~cm] == 0) and np.all(act[~cm] == -1)
    sure = cm & (np.abs(want[..., 1] - want[..., 0]) > 2 * BF16_TOL * scale)
    np.testing.assert_array_equal(act[sure], (want[..., 1] > want[..., 0]).astype(np.int8)[sure])
    # greedy action is consistent with the kernel's own Q-values everywhere
    np.testing.assert_array_equal(act[cm], (q[..., 1] > q[..., 0]).astype(np.int8)[cm])


# runs in a child process: MLS_BF16_CHUNK_TILES is read once per process.  Prints the pass size, writes Q.
_BF16_CHUNK_CHILD = """
import sys, ctypes, numpy as np, torch
sys.path.insert(0, sys.argv[1])
from melissa_b200 import _lib
from melissa_b200.networks import NETWORKS
kind, N, d = sys.argv[2], int(sys.argv[3]), sys.argv[4]
kw = dict(aggregator="max") if kind == "hl_dgn" else {}
dueling = ({"hidden_sizes": [128, 128]}, {"hidden_sizes": [128, 128]})
m = NETWORKS[kind](5, 128, 2, 4, N, dueling_param=dueling, device="cuda", **kw)
m.load_state_dict(torch.load(d + "/sd.pt"))
m = m.cuda().set_precision("bf16")
rows = np.load(d + "/rows.npy")
q, _ = m(rows)
np.save(d + "/q.npy", q.cpu().numpy())
print(_lib.lib().mls_dgn_chunk_graphs(ctypes.byref(m._desc()), rows.shape[0]))
"""


@pytest.mark.parametrize("kind", ["l_dgn", "dgn_r", "hl_dgn"])
def test_bf16_agent_rows_and_chunking(kind, tmp_path):
    """Agent rows through the bf16 path, in one pass and, in a child process with 40-tile passes (102 graphs of 50 nodes),
    in nine: every pass computes its graphs with the same kernels, tiles and reductions, so Q must not change in any bit."""
    import ctypes
    import os
    import subprocess
    import sys
    from melissa_b200 import _lib
    N, bs = 50, 900
    kw = dict(aggregator="max") if kind == "hl_dgn" else {}
    sd = _random_sd(kind, 61)
    om = _obs_matrix(N, bs, 29)
    ctrl = np.random.default_rng(7).integers(0, N, size=bs).astype(np.float32)
    rows = np.concatenate([om.reshape(bs, -1), ctrl[:, None]], axis=1)
    sel = np.r_[0:16, 94:110, 196:212, 884:900]
    want = no.FORWARDS[kind](sd, torch.as_tensor(rows[sel]), N, **kw).numpy()
    m = _module(kind, N, sd, **kw).set_precision("bf16")
    assert _lib.lib().mls_dgn_chunk_graphs(ctypes.byref(m._desc()), bs) == bs      # one pass in this process
    q, _ = m(rows)
    q = q.cpu().numpy()
    scale = max(1.0, float(np.abs(want).max()))
    assert float(np.abs(q[sel] - want).max()) <= BF16_TOL * scale
    assert np.isfinite(q).all()
    torch.save(sd, tmp_path / "sd.pt")
    np.save(tmp_path / "rows.npy", rows)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, MLS_BF16_CHUNK_TILES="40")
    res = subprocess.run([sys.executable, *(["-s"] if sys.flags.no_user_site else []), "-c", _BF16_CHUNK_CHILD, root, kind, str(N),
                          str(tmp_path)], env=env, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    gc = int(res.stdout.split()[-1])
    assert gc < bs and gc == 40 * 128 // N, gc
    q_chunked = np.load(tmp_path / "q.npy")
    assert np.array_equal(q_chunked.view(np.uint32), q.view(np.uint32)), float(np.abs(q_chunked - q).max())


def test_large_graphs_200_nodes():
    """BASELINE config 5 stress: 200-node graphs (mean degree ~21, max > 32 -> the 32-neighbour cap of
    radius_graph is exercised).  fp32 and bf16 paths for every model (the attention kernels stage the
    source rows as bf16, so even the three-operand Transformer conv fits one CTA's shared memory at N = 200)."""
    from melissa_b200 import _lib
    N, B = 200, 3
    om = _obs_matrix(N, B, 71)
    cm = np.random.default_rng(8).random((B, N)) < 0.1
    for kind, kw in (("l_dgn", {}), ("dgn_r", {}), ("hl_dgn", {"aggregator": "max"})):
        sd = _random_sd(kind, 73)
        want = no.forward_graphs(kind, sd, torch.as_tensor(om), torch.as_tensor(cm), N, **kw).numpy()
        m = _module(kind, N, sd, **kw)
        q, _ = m.forward_graphs(torch.as_tensor(om, device="cuda"), torch.as_tensor(cm, device="cuda").to(torch.uint8))
        _assert_q(q.cpu().numpy(), want, f"{kind} N=200 fp32")
        m.set_precision("bf16")
        q, _ = m.forward_graphs(torch.as_tensor(om, device="cuda"), torch.as_tensor(cm, device="cuda").to(torch.uint8))
        scale = max(1.0, float(np.abs(want).max()))
        assert float(np.abs(q.cpu().numpy() - want).max()) <= BF16_TOL * scale, kind


@pytest.mark.parametrize("kind", ["l_dgn", "dgn_r"])
@pytest.mark.parametrize("N,B", [(50, 300), (20, 64), (12, 9), (64, 17), (7, 500)])
def test_conv2_tensor_core_attention_matches_gather_kernel(kind, N, B):
    """conv2_attn.cu (default for graphs of <= 64 nodes): packed-half logits, fp16 softmax weights, tcgen05 aggregation
    over the compacted needed rows.  Against the gather kernel (option conv2_mma = 0, bf16 operands, fp32 SIMT math) and
    the fp32 oracle: within the stated bf16 tolerance; targets with many / no neighbours, graphs without controlling
    nodes and all-controlling graphs included."""
    from melissa_b200 import _lib
    assert _lib.get_option("conv2_mma") == 1
    sd = _random_sd(kind, 81)
    om = _obs_matrix(N, B, 31)
    if B > 4:
        om[2, :, :2] = 0.0                                  # complete graph: every target has min(N-1, 32) sources
        om[3, :, 0] = np.arange(N) * 1.0                    # no edges at all
    cm = np.random.default_rng(9).random((B, N)) < 0.3
    cm[0] = False
    cm[1] = True
    want = no.forward_graphs(kind, sd, torch.as_tensor(om), torch.as_tensor(cm), N).numpy()
    m = _module(kind, N, sd).set_precision("bf16")
    args = (torch.as_tensor(om, device="cuda"), torch.as_tensor(cm, device="cuda").to(torch.uint8))
    q1, a1 = m.forward_graphs(*args)
    _lib.set_option("conv2_mma", 0)
    try:
        q0, _ = m.forward_graphs(*args)
    finally:
        _lib.set_option("conv2_mma", 1)
    scale = max(1.0, float(np.abs(want).max()))
    e_or, e_g = float(np.abs(q1.cpu().numpy() - want).max()), float((q1 - q0).abs().max())
    print(f"conv2 mma {kind} N={N}: vs oracle {e_or:.4f}, vs gather {e_g:.4f} (scale {scale:.2f})")
    assert e_or <= BF16_TOL * scale, (e_or, scale)
    assert e_g <= 0.5 * BF16_TOL * scale, (e_g, scale)
    assert not torch.equal(q0, q1)                          # really the other kernel
    assert torch.equal(a1 >= 0, torch.as_tensor(cm, device="cuda"))
    q2, _ = m.forward_graphs(*args)
    assert torch.equal(q1, q2)                              # deterministic, scratch state left clean


@pytest.mark.parametrize("kind,kw", [("l_dgn", {}), ("dgn_r", {}), ("hl_dgn", {"aggregator": "max"})])
@pytest.mark.parametrize("N", [20, 50, 100])
def test_topology_cache_and_prepared_weights_are_bit_identical(kind, kw, N):
    """Static pools: radius_graph lists from the per-pool cache (selected by graph id, strided like the
    environment's episode array) and parameters packed once (MLS_FWD_PREPARED) give exactly the results of the
    per-call path; after the parameters change, the prepared copy is refreshed."""
    B, G = 48, 8
    pool = GraphPool.synthetic(N, G, first_seed=3, side=None if N in (20, 50) else min(1.0, (N / 50) ** 0.5))
    rng = np.random.default_rng(12)
    gi = rng.integers(0, G, size=B).astype(np.int32)
    om = _obs_matrix(N, B, 5)
    om[:, :, :2] = pool.pos[gi]
    om[:, :, 2] = pool.adj[gi].sum(2)
    cm = rng.random((B, N)) < 0.35
    sd = _random_sd(kind, 14)
    m = _module(kind, N, sd, **kw).set_precision("bf16")
    args = (torch.as_tensor(om, device="cuda"), torch.as_tensor(cm, device="cuda").to(torch.uint8))
    q0, a0 = m.forward_graphs(*args, discrete_features=True)
    cache = m.build_topology_cache(pool.pos)
    ids = torch.zeros(B, 8, dtype=torch.int32, device="cuda")
    ids[:, 3] = torch.as_tensor(gi, device="cuda")
    q1, a1 = m.forward_graphs(*args, discrete_features=True, graph_ids=ids.view(-1)[3:], graph_id_stride=8, topology_cache=cache,
                              prepared=True)
    assert torch.equal(q0, q1) and torch.equal(a0, a1)
    q2, _ = m.forward_graphs(*args, discrete_features=True, graph_ids=ids.view(-1)[3:], graph_id_stride=8, topology_cache=cache,
                             prepared=True)
    assert torch.equal(q1, q2)
    with torch.no_grad():
        for p in m.parameters():
            p.mul_(1.01)
    q3, _ = m.forward_graphs(*args, discrete_features=True)
    q4, _ = m.forward_graphs(*args, discrete_features=True, graph_ids=ids.view(-1)[3:], graph_id_stride=8, topology_cache=cache,
                             prepared=True)
    assert torch.equal(q3, q4) and not torch.equal(q3, q0)


@pytest.fixture
def gather_attention():
    """Discrete-feature mode with the gather kernel only (no pair-logit table / tensor-core aggregation)."""
    from melissa_b200 import _lib
    old = _lib.get_option("attn_mma")
    _lib.set_option("attn_mma", 0)
    yield
    _lib.set_option("attn_mma", old)


@pytest.mark.parametrize("kind,kw", [("l_dgn", {}), ("dgn_r", {}), ("hl_dgn", {"aggregator": "max"}),
                                     ("hl_dgn", {"aggregator": "mean"})])
@pytest.mark.parametrize("N,B", [(50, 40), (20, 64), (12, 9), (200, 6)])
def test_discrete_feature_table_path_is_bit_identical(kind, kw, N, B, gather_attention):
    """MLS_FWD_DISCRETE_FEATURES: encoder + conv1 projections looked up per distinct feature vector.  The
    table rows are produced by the same kernels on the same inputs, so Q-values and actions must equal the
    per-node bf16 path bit for bit; the violation counter stays 0 on environment observations."""
    sd = _random_sd(kind, 5)
    om = _obs_matrix(N, B, 77)
    cm = np.random.default_rng(3).random((B, N)) < 0.4
    m = _module(kind, N, sd, **kw).set_precision("bf16")
    args = (torch.as_tensor(om, device="cuda"), torch.as_tensor(cm, device="cuda").to(torch.uint8))
    q0, a0 = m.forward_graphs(*args, eps=0.2, philox_seed=4, philox_offset=1)
    err = torch.full((1,), 7, dtype=torch.int32, device="cuda")
    q1, a1 = m.forward_graphs(*args, eps=0.2, philox_seed=4, philox_offset=1, discrete_features=True, feature_errors=err)
    assert int(err.item()) == 0
    assert torch.equal(q0, q1) and torch.equal(a0, a1)
    # a non-integer feature is counted (and that row evaluated with key 0), never silently accepted
    bad = om.copy()
    bad[0, 0, 3] = 0.5
    bad[B - 1, N - 1, 2] = -1.0
    m.forward_graphs(torch.as_tensor(bad, device="cuda"), args[1], discrete_features=True, feature_errors=err)
    assert int(err.item()) == 2


@pytest.mark.parametrize("kind,kw", [("l_dgn", {}), ("dgn_r", {}), ("hl_dgn", {"aggregator": "max"}),
                                     ("hl_dgn", {"aggregator": "mean"}), ("hl_dgn", {"aggregator": "add"})])
@pytest.mark.parametrize("N,B", [(50, 300), (20, 64), (12, 9), (62, 33), (7, 1000), (60, 64)])
def test_tensor_core_table_attention_within_tolerance(kind, kw, N, B):
    """attn_table.cu (default in discrete-feature mode, graphs of <= 62 nodes): softmax weights from the
    pair-logit table, aggregation on tcgen05 (HL-DGN: graph pooling in the epilogue).  Differs from the gather
    kernel only by bf16 rounding of the softmax weights: within the stated bf16 tolerance of the fp32 oracle,
    and close to the gather path.  Tiles of 1..5 graphs; N = 60 leaves no room for the bias rows in the weight
    matrix (the epilogue adds the bias)."""
    from melissa_b200 import _lib
    assert _lib.get_option("attn_mma") == 1
    sd = _random_sd(kind, 6)
    om = _obs_matrix(N, B, 78)
    cm = np.random.default_rng(4).random((B, N)) < 0.4
    want = no.forward_graphs(kind, sd, torch.as_tensor(om), torch.as_tensor(cm), N, **kw).numpy()
    m = _module(kind, N, sd, **kw).set_precision("bf16")
    args = (torch.as_tensor(om, device="cuda"), torch.as_tensor(cm, device="cuda").to(torch.uint8))
    q0, _ = m.forward_graphs(*args)
    err = torch.zeros(1, dtype=torch.int32, device="cuda")
    q1, a1 = m.forward_graphs(*args, discrete_features=True, feature_errors=err)
    assert int(err.item()) == 0
    scale = max(1.0, float(np.abs(want).max()))
    e_or = float(np.abs(q1.cpu().numpy() - want).max())
    e_g = float((q1 - q0).abs().max())
    assert e_or <= BF16_TOL * scale, (e_or, scale)
    assert e_g <= 0.5 * BF16_TOL * scale, (e_g, scale)
    assert not torch.equal(q0, q1)                          # really the other kernel
    assert torch.equal(a1 >= 0, torch.as_tensor(cm, device="cuda"))
    # same call again (scratch state such as the used-key flags is left clean)
    q2, _ = m.forward_graphs(*args, discrete_features=True)
    assert torch.equal(q1, q2)


def test_tensor_core_table_attention_falls_back_when_keys_overflow():
    """More than 1024 distinct feature keys in one pass: the pair-logit table cannot hold them, the gather
    kernel takes the pass (decided on the device) -- bit-identical to the per-node path."""
    N, B = 50, 200
    sd = _random_sd("l_dgn", 8)
    om = _obs_matrix(N, B, 79)
    rng = np.random.default_rng(0)
    om[:, :, 2] = rng.integers(0, 64, size=(B, N))
    om[:, :, 3] = rng.integers(0, 64, size=(B, N))
    cm = rng.random((B, N)) < 0.4
    m = _module("l_dgn", N, sd).set_precision("bf16")
    args = (torch.as_tensor(om, device="cuda"), torch.as_tensor(cm, device="cuda").to(torch.uint8))
    q0, a0 = m.forward_graphs(*args)
    q1, a1 = m.forward_graphs(*args, discrete_features=True)
    assert torch.equal(q0, q1) and torch.equal(a0, a1)


@pytest.mark.parametrize("kind,kw", [("l_dgn", {}), ("dgn_r", {}), ("hl_dgn", {"aggregator": "max"})])
def test_bf16_product_path_on_environment_observations_flip_rate(kind, kw):
    """The headline configuration's inputs, not synthetic feature columns: 4096 episodes of 50-node graphs rolled out for
    36 rounds with the bf16 product path (discrete-feature tables, tensor-core attention, topology cache); on the
    observations the environment then holds, the bf16 path and the fp32 CUDA path (the <= 1e-5 parity anchor) are
    compared decision by decision: max |dq| within the stated bf16 tolerance, and every greedy-action flip sits on a
    decision whose fp32 margin |q1 - q0| is below 2 * max|dq| (a flip needs both Q-values to move across the gap)."""
    from melissa_b200.batched_env import BatchedGraphEnv, ResetTuplesDevice
    from melissa_b200.rollout import Rollout
    N, B, G = 50, 4096, 64
    pool = GraphPool.synthetic(N, G, first_seed=0)
    gi, src, inter, scr, _ = reset_chain.episode_pool(9, 2 * B, N, G)
    sd = _random_sd(kind, 9)
    net = _module(kind, N, sd, **kw).set_precision("bf16")
    env = BatchedGraphEnv(B, N, pool)
    ro = Rollout(env, net, eps=0.05, seed=9)
    ro.start(ResetTuplesDevice(gi, src, inter, scr, N, "cuda", pool_size=G))
    for _ in range(36):
        ro.round()
    assert ro.feature_violations() == 0
    obs, active = env.obs.clone(), env.active.clone()
    q_b, a_b = net.forward_graphs(obs, active, discrete_features=True, graph_ids=ro.graph_ids, graph_id_stride=8,
                                  topology_cache=ro.topology_cache, prepared=True)
    ref = _module(kind, N, sd, **kw)                                  # fp32 kernels
    q_f, a_f = ref.forward_graphs(obs, active)
    m = active.bool()
    n_dec = int(m.sum())
    assert n_dec > 2 * B
    dq = float((q_b - q_f).abs()[m].max())
    scale = max(1.0, float(q_f[m].abs().max()))
    flips = (a_b != a_f) & m
    rate = float(flips.sum()) / n_dec
    margin = (q_f[..., 1] - q_f[..., 0]).abs()
    worst = float(margin[flips].max()) if bool(flips.any()) else 0.0
    print(f"{kind}: {n_dec} decisions, max|dq| {dq:.5f} (scale {scale:.2f}), flip rate {rate:.5f}, largest flipped margin {worst:.5f}, "
          f"median margin {float(margin[m].median()):.4f}")
    assert dq <= BF16_TOL * scale
    assert worst <= 2.0 * dq + 1e-7
    assert rate <= 0.02


@pytest.mark.parametrize("kind,kw", [("l_dgn", {}), ("dgn_r", {}), ("hl_dgn", {"aggregator": "mean"})])
def test_fp32_tensor_core_route_meets_the_fp32_bar(kind, kw):
    """precision fp32 runs its dense layers on tcgen05 through 3-way bf16 operand splits concatenated along K
    (option fp32_tc, default on): same <= 1e-5 bar against the fp32 oracle as the SIMT sgemm route, on a batch large
    enough for several 128-row GEMM tiles and with trained-scale (x8) weights in one layer to stress the split."""
    from melissa_b200 import _lib
    N, B = 50, 60
    sd = _random_sd(kind, 33)
    sd["conv1.lin_l.weight" if kind != "dgn_r" else "conv1.lin_key.weight"] *= 8.0
    om = _obs_matrix(N, B, 41)
    cm = np.random.default_rng(6).random((B, N)) < 0.3
    want = no.forward_graphs(kind, sd, torch.as_tensor(om), torch.as_tensor(cm), N, **kw).numpy()
    m = _module(kind, N, sd, **kw)
    args = (torch.as_tensor(om, device="cuda"), torch.as_tensor(cm, device="cuda").to(torch.uint8))
    assert _lib.get_option("fp32_tc") == 1
    q1, a1 = m.forward_graphs(*args)
    _assert_q(q1.cpu().numpy(), want, f"{kind} fp32 tensor-core route")
    _lib.set_option("fp32_tc", 0)
    try:
        q0, a0 = m.forward_graphs(*args)
    finally:
        _lib.set_option("fp32_tc", 1)
    _assert_q(q0.cpu().numpy(), want, f"{kind} fp32 SIMT route")
    scale = max(1.0, float(np.abs(want).max()))
    print(f"{kind}: tensor-core route err {float(np.abs(q1.cpu().numpy() - want).max()):.2e}, SIMT route err "
          f"{float(np.abs(q0.cpu().numpy() - want).max()):.2e} (scale {scale:.2f})")
    assert not torch.equal(q0, q1)                          # really another code path
