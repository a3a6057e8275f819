"""bf16 training precision (``DGNBase.set_train_precision("bf16")``): the dense-layer Function ``_LinearBF16`` on the tcgen05
GEMM (``csrc/train_linear.cu``) against float64 references, its determinism, and the Q-values, gradients and updates of every
network family against the fp32 training path."""
import numpy as np
import pytest
import torch

from test_persistent_tiles_gpu import _Cap

pytestmark = pytest.mark.gpu
U32 = 2.0 ** -24                                            # unit roundoff of fp32
DUELING = lambda: ({"hidden_sizes": [128, 128]}, {"hidden_sizes": [128, 128]})


def _bf16(t):
    return t.to(torch.bfloat16).to(torch.float32)


def _run(x, w, b, dy, need_dx=True):
    """y, dx, dW, db of _LinearBF16 through autograd.  ``x`` may be a column slice of a wider matrix (row stride > in)."""
    from melissa_b200.networks.autograd import _LinearBF16
    x = x.detach().requires_grad_(need_dx)
    w = w.detach().requires_grad_(True)
    b = b.detach().requires_grad_(True)
    y = _LinearBF16.apply(x, w, b)
    y.backward(dy)
    return y.detach(), (x.grad if need_dx else None), w.grad, b.grad


def _ints(g, shape, lim=8):
    return torch.randint(-lim, lim + 1, shape, generator=g, dtype=torch.int32).to(torch.float32).cuda()


def _exact_case(rows, k_in, k_out, seed, strided=False):
    g = torch.Generator().manual_seed(seed)
    x = _ints(g, (rows, k_in + 3))[:, :k_in] if strided else _ints(g, (rows, k_in))
    w, b, dy = _ints(g, (k_out, k_in)), _ints(g, (k_out,)), _ints(g, (rows, k_out))
    y, dx, dw, db = _run(x, w, b, dy)
    x64, w64, dy64 = x.double(), w.double(), dy.double()
    want = {"y": x64 @ w64.T + b.double(), "dx": dy64 @ w64, "dW": dy64.T @ x64, "db": dy64.sum(0)}
    for name, got in (("y", y), ("dx", dx), ("dW", dw), ("db", db)):
        assert got.dtype == torch.float32 and got.shape == want[name].shape, name
        bad = int((got.double() != want[name]).sum())
        assert bad == 0, f"{name}: {bad} of {got.numel()} entries differ from the exact result (rows {rows}, in {k_in}, out {k_out})"


@pytest.mark.parametrize("k_out", [1, 2, 128, 512])
@pytest.mark.parametrize("k_in", [5, 128, 512, 1152])
def test_integer_operands_are_exact(k_in, k_out):
    """Integers |v| <= 8: every operand is a bf16 value and every fp32 partial sum (at most 8 * 8 * 4097 < 2^24) is exact, so
    forward, dx, dW and db must equal float64 bit for bit.  A wrong pad, K block, row clip or transposition shows here."""
    for i, rows in enumerate((1, 63, 64, 127, 128, 129, 4097)):
        _exact_case(rows, k_in, k_out, seed=1000 * k_in + 10 * k_out + i, strided=(i % 2 == 1))


def test_integer_operands_are_exact_at_several_tiles_per_cta():
    with _Cap(2):
        for k_in, k_out in ((1152, 512), (5, 128), (512, 2)):
            _exact_case(4097, k_in, k_out, seed=k_in + k_out)


def test_zero_rows():
    from melissa_b200.networks.autograd import _LinearBF16
    x = torch.zeros(0, 5, device="cuda", requires_grad=True)
    w = torch.randn(128, 5, device="cuda", requires_grad=True)
    b = torch.randn(128, device="cuda", requires_grad=True)
    y = _LinearBF16.apply(x, w, b)
    assert y.shape == (0, 128)
    y.sum().backward()
    assert x.grad.shape == (0, 5)
    assert bool((w.grad == 0).all()) and bool((b.grad == 0).all())


def _dot_bound(a64, b64, K):
    """fp32 accumulation of exact bf16 products over K: the GEMM adds one K = 16 slice per MMA step into an fp32 accumulator.
    Allow 2u (one truncating alignment plus one rounding) per step, K / 16 steps plus four for the additions inside a slice,
    on the sum of |products|: |err| <= 2u (K / 16 + 4) sum_k |a_k b_k|."""
    return 2 * U32 * (K / 16 + 4) * (a64.abs() @ b64.abs().T)


def test_random_operands_within_the_fp32_accumulation_bound():
    """Normal operands against float64 on the bf16-rounded operands.  The bound must be >= 100x tighter than what two likely
    mistakes cost: one operand rounded once more or once less (the unrounded fp32 value in place of its bf16 rounding), and
    one dropped 64-wide K block.  Sizes keep K <= 192 so that this holds for every product."""
    g = torch.Generator().manual_seed(5)
    rows, k_in, k_out = 129, 128, 192
    x = torch.randn(rows, k_in, generator=g).cuda()
    w = torch.randn(k_out, k_in, generator=g).cuda() * 0.1
    b = torch.randn(k_out, generator=g).cuda()
    dy = torch.randn(rows, k_out, generator=g).cuda()
    y, dx, dw, db = _run(x, w, b, dy)
    xb, wb, dyb = _bf16(x).double(), _bf16(w).double(), _bf16(dy).double()
    # (output, A, B^T as [N][K], the unrounded A, bias)
    cases = {"y": (y, xb, wb, x.double(), b.double()), "dx": (dx, dyb, wb.T, dy.double(), None),
             "dW": (dw, dyb.T, xb.T, dy.double().T, None)}
    for name, (got, a, bt, a_raw, bias) in cases.items():
        K = a.shape[1]
        want = a @ bt.T + (bias if bias is not None else 0)
        tol = _dot_bound(a, bt, K) + (U32 * want.abs() if bias is not None else 0)
        err = (got.double() - want).abs()
        assert bool((err <= tol).all()), f"{name}: worst err/tol {float((err / tol).max()):.3g}"
        once_more = ((a_raw @ bt.T) - (a @ bt.T)).abs().max()
        dropped = (a[:, :64] @ bt[:, :64].T).abs().max()
        assert float(once_more) >= 100 * float(tol.max()) and float(dropped) >= 100 * float(tol.max()), name
    want_db = dy.double().sum(0)
    tol_db = U32 * (64 + (rows + 63) // 64) * dy.double().abs().sum(0)
    assert bool(((db.double() - want_db).abs() <= tol_db).all())


def test_backward_is_bitwise_reproducible():
    g = torch.Generator().manual_seed(8)
    x = torch.randn(4097, 512, generator=g).cuda()
    w = torch.randn(128, 512, generator=g).cuda()
    b = torch.randn(128, generator=g).cuda()
    dy = torch.randn(4097, 128, generator=g).cuda()
    first = _run(x, w, b, dy)
    for _ in range(2):
        again = _run(x, w, b, dy)
        for u, v in zip(first, again):
            assert torch.equal(u.view(torch.int32), v.view(torch.int32))


def _setup(kind, N=20, B=64, seed=3, ring=8, dueling=True, replay_cls=None, policy_cls=None, **kw):
    from melissa_b200 import reset_chain
    from melissa_b200.batched_env import BatchedGraphEnv, ResetTuplesDevice
    from melissa_b200.data_parallel import FlatParameters, FusedAdam
    from melissa_b200.networks import NETWORKS
    from melissa_b200.policy import BatchedCollector, DQNPolicy
    from melissa_b200.replay import DeviceReplay
    from melissa_b200.topology import GraphPool
    pool = GraphPool.synthetic(N, 8, first_seed=seed)
    tup = reset_chain.episode_pool(seed, 512, N, 8)
    torch.manual_seed(seed)
    net = NETWORKS[kind](5, 128, 2, 4, N, dueling_param=DUELING() if dueling else None, device="cuda", **kw).cuda()
    flat = FlatParameters(net)
    optim = FusedAdam(flat, lr=1e-3)
    pol = (policy_cls or DQNPolicy)(net, optim, discount_factor=0.99, estimation_step=4, target_update_freq=5, eps=0.1)
    env = BatchedGraphEnv(B, N, pool, want_info=True)
    replay = (replay_cls or DeviceReplay)(B, N, ring, seed=1)
    col = BatchedCollector(agents_num=N, policy=pol, env=env, buffer=replay, exploration_noise=True,
                           tuples=ResetTuplesDevice(*tup[:4], N, "cuda", pool_size=8))
    for _ in range(ring):
        col.iterate(0.3)
    return net, flat, pol, replay


NETS = [("l_dgn", {}, True), ("dgn_r", {}, True), ("hl_dgn", {"aggregator": "max"}, True), ("hl_dgn", {"aggregator": "mean"}, True),
        ("l_dgn", {}, False)]


# How far a bf16 gradient may sit from the fp32 one depends on where the parameter sits relative to the attention logits.
# The forward rounds the projections' operands to bf16, so every logit carries a relative rounding error of about 2^-9 of
# its terms, and the logits' gradient is the softmax Jacobian a_e (g_e - sum_f a_f g_f): a difference of near-equal terms
# in which that error is amplified.  Parameters that reach the loss only through the logits (GATv2's target projection and
# attention vector, TransformerConv's query and key projections) see it most; every other parameter below an attention
# layer receives part of its gradient through a logit; the dueling heads / out_linear after the last aggregation see none.
LOGIT_ONLY = (".lin_r.", ".att", ".lin_query.", ".lin_key.weight")
HEADS = ("Q.", "V.", "out_linear.")
BARS = {"heads": 2e-2, "graph": 5e-2, "logit-only": 1e-1}


def _grad_class(name):
    if name.startswith(HEADS):
        return "heads"
    return "logit-only" if any(a in name for a in LOGIT_ONLY) else "graph"


def _q_and_grads(net, rows, prec):
    from melissa_b200.networks.autograd import q_values
    target = torch.linspace(-1, 1, rows.shape[0], device="cuda")
    net.set_train_precision(prec)
    net.zero_grad(set_to_none=True)
    q = q_values(net, rows)
    ((q[:, 0] - target).pow(2).mean() + q[:, 1].mean()).backward()
    return q.detach(), {k: p.grad.detach().clone() for k, p in net.named_parameters() if p.grad is not None}


def _rel_errors(g_test, g_ref):
    """Relative L2 error per parameter, except TransformerConv's key bias: its exact gradient is zero (adding <q, b> to every
    logit of a target leaves the softmax unchanged), so both values are rounding noise, measured against the key weights'
    gradient instead."""
    rel, key_bias = {}, {}
    for k, g in g_ref.items():
        err = float((g_test[k] - g).norm())
        if k.endswith("lin_key.bias"):
            key_bias[k] = max(err, float(g_test[k].norm())) / float(g_ref[k[:-4] + "weight"].norm())
        elif float(g.norm()) > 0:
            rel[k] = err / float(g.norm())
    return rel, key_bias


def _replay_rows(kind, dueling, kw, n=1024):
    from melissa_b200.policy import Batch
    net, _, _, replay = _setup(kind, N=50, dueling=dueling, **kw)
    rho, ep, ag = replay.sample_indices(n, 4)
    return net, Batch(replay.gather(rho, ep, ag, 4, 0.99)).obs


@pytest.mark.parametrize("fused", [True, False], ids=["fused", "torch"])
@pytest.mark.parametrize("kind,kw,dueling", NETS, ids=["l_dgn", "dgn_r", "hl_dgn-max", "hl_dgn-mean", "l_dgn-no-dueling"])
def test_network_q_and_gradients_match_fp32(kind, kw, dueling, fused, monkeypatch):
    """Q within the project's bf16 bar 1e-2 max(1, |q|) and every parameter gradient within its class's relative (L2) bar
    (BARS) of the fp32 training path, on 50-node rows sampled from a replay a collector filled; the same parameters get
    gradients; TransformerConv's key bias stays at rounding level, 1e-2 of the key weights' gradient."""
    from melissa_b200.networks.autograd import fused_training_available
    monkeypatch.setenv("MLS_TRAIN_FUSED", "1" if fused else "0")
    net, rows = _replay_rows(kind, dueling, kw)
    assert fused_training_available(net, rows) == fused
    (q32, g32), (q16, g16) = _q_and_grads(net, rows, "fp32"), _q_and_grads(net, rows, "bf16")
    dq = float((q16 - q32).abs().max())
    assert dq <= 1e-2 * max(1.0, float(q32.abs().max())), dq
    assert set(g16) == set(g32) and not any("lin_skip" in k for k in g32)
    rel, key_bias = _rel_errors(g16, g32)
    worst = {}
    for k, v in rel.items():
        c = _grad_class(k)
        if v > worst.get(c, ("-", 0.0))[1]:
            worst[c] = (k, v)
    worst_kb = max(key_bias.items(), key=lambda kv: kv[1]) if key_bias else ("-", 0.0)
    print(f"\n{kind}{kw} dueling={dueling} fused={fused}: max|dq| {dq:.2e}; worst relative gradient error per class {worst}; "
          f"key bias / key weights {worst_kb}")
    assert "heads" in worst
    for c, (k, v) in worst.items():
        assert v <= BARS[c], (c, k, v)
    assert worst_kb[1] <= 1e-2, worst_kb


@pytest.mark.parametrize("kind,kw,dueling", NETS, ids=["l_dgn", "dgn_r", "hl_dgn-max", "hl_dgn-mean", "l_dgn-no-dueling"])
def test_bf16_fused_and_torch_paths_agree(kind, kw, dueling, monkeypatch):
    """Both training paths hand the same operands to the same bf16 dense layers; they differ only in the fp32 summation order
    of the edge phase.  So their bf16 Q and gradients must agree far more closely than either agrees with fp32: the
    distance to fp32 measured above is the precision of the definition, not a defect of one path."""
    net, rows = _replay_rows(kind, dueling, kw)
    monkeypatch.setenv("MLS_TRAIN_FUSED", "1")
    q_f, g_f = _q_and_grads(net, rows, "bf16")
    monkeypatch.setenv("MLS_TRAIN_FUSED", "0")
    q_t, g_t = _q_and_grads(net, rows, "bf16")
    assert float((q_f - q_t).abs().max()) <= 1e-3 * max(1.0, float(q_t.abs().max()))
    assert set(g_f) == set(g_t)
    rel, key_bias = _rel_errors(g_f, g_t)
    worst = max(rel.items(), key=lambda kv: kv[1])
    print(f"\n{kind}{kw} dueling={dueling}: bf16 fused vs torch, worst relative gradient difference {worst}")
    assert worst[1] <= 5e-3, worst
    assert all(v <= 1e-2 for v in key_bias.values()), key_bias


@pytest.mark.parametrize("policy", ["dqn", "dgn"])
def test_policy_updates_with_prioritized_replay(policy):
    from melissa_b200.policy import DGNPolicy, DQNPolicy
    from melissa_b200.replay import DevicePrioritizedReplay
    per = lambda B, N, R, seed: DevicePrioritizedReplay(B, N, R, alpha=0.6, beta=0.4, seed=seed)
    net, flat, pol, replay = _setup("l_dgn", N=12, B=32, replay_cls=per, policy_cls=DGNPolicy if policy == "dgn" else DQNPolicy)
    net.set_train_precision("bf16")
    w0 = flat.flat.clone()
    for _ in range(20):
        loss = float(pol.update(64, replay)["loss"])
        assert np.isfinite(loss)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(flat.flat).all()) and bool(torch.isfinite(replay.tree).all()) and bool(torch.isfinite(replay.prio).all())
    assert float(flat.grad.abs().sum()) > 0 and not torch.equal(flat.flat, w0)
