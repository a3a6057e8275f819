"""GPU: the training kernels called directly through the ABI on hand-built inputs, against float64 references --
the GATv2 / TransformerConv edge phases and their backward (oracle/train_oracle.py, pinned on net_oracle by
tests/test_training_host.py), the per-sample edge lists (net_oracle.radius_graph_mask) and one Adam step at a time.
Every index stays in bounds: list slots past a target's count point at a row filled with 1e6, and row -1 of the
target-side inputs is NaN, so a kernel that reads what it must not gives wrong numbers rather than a fault."""
import numpy as np
import pytest
import torch

from oracle import net_oracle as no
from oracle import train_oracle

pytestmark = pytest.mark.gpu
C = 128
POISON = 1e6


def _lib():
    from melissa_b200 import _lib
    return _lib, _lib.lib()


def _edge_case(T, H, seed):
    """Lists of T targets over S = T + 64 source rows.  Target t: entry 0 = source row t (its own row), entry 1 = the
    shared row S - 1 (every target with cnt >= 2), the rest random; cnt from 1 to 34 with 1 and 34 always present.
    Targets t % 7 == 3 have cnt = 1; t % 11 == 5: every source row holds the same values (all-equal logits);
    t % 13 == 6: sources from a block of scaled rows (peaked logits, about +-60); t % 17 == 9 (t > 0): tgt_row = -1.
    Target 0 is a plain target with cnt 34, so T = 1 is one full list."""
    g = torch.Generator().manual_seed(seed)
    S = T + 64
    cap = 36
    cnt = torch.randint(1, 35, (T,), generator=g)
    t = torch.arange(T)
    cnt[0] = 34
    cnt[t % 7 == 3] = 1
    src = torch.randint(0, S - 1, (T, cap), generator=g)
    src[:, 0] = t
    src[:, 1] = S - 1
    flat = t % 11 == 5
    peak = t % 13 == 6
    src[flat, 1:] = S - 9 + torch.randint(0, 8, (int(flat.sum()), cap - 1), generator=g)     # rows S-9 .. S-2: equal
    src[flat, 0] = S - 9
    src[peak, 1:] = S - 33 + torch.randint(0, 24, (int(peak.sum()), cap - 1), generator=g)   # rows S-33 .. S-10: scaled
    src[torch.arange(cap)[None, :] >= cnt[:, None]] = S                                        # row S = poison
    tgt = t.clone()
    tgt[(t % 17 == 9) & (t > 0)] = -1
    return tgt.int(), src.int(), cnt.int(), S


def _inputs(S, T, H, seed, scale_rows):
    """Source-side [S + 1, ld] (row S = poison) and target-side [1 + T, ld] (row 0 = row -1 = NaN) fp32 buffers,
    ld = 128 H + 4 with poisoned padding."""
    g = torch.Generator().manual_seed(seed)
    HC, ld = H * C, H * C + 4

    def src_buf():
        x = torch.randn(S + 1, ld, generator=g)
        x[S - 9:S - 1, :HC] = x[S - 9, :HC]
        x[S - 33:S - 9, :HC] *= scale_rows
        x[S] = POISON
        x[:, HC:] = POISON
        return x.cuda()

    def tgt_buf():
        x = torch.randn(T + 1, ld, generator=g)
        x[0] = float("nan")
        x[:, HC:] = POISON
        return x.cuda()
    return src_buf, tgt_buf


def _close(name, got, want, errs):
    # fp32 kernels, <= 34-term softmaxes and 128-term dot products: the largest error measured on a B200 (1000 W) was
    # 2.5e-6 of max(1, max |ref|), for d_v; 1e-5 leaves room for other atomic orders
    scale = max(1.0, float(want.abs().max()))
    err = float((got.double() - want).abs().max()) / scale
    errs[name] = err
    assert err <= 1e-5, f"{name}: max error {err:.3e} of max(1, max |ref|) = {scale:.3e}"


EDGE_CASES = [(H, 300) for H in (1, 2, 3, 4)] + [(4, T) for T in (1, 1183, 1184, 1185)] + [(3, 10000)]


@pytest.mark.parametrize("H,T", EDGE_CASES)
def test_gatv2_edge_kernels_match_the_float64_reference(H, T):
    _l, L = _lib()
    torch.manual_seed(T + H)
    tgt, src, cnt, S = _edge_case(T, H, seed=H * 7919 + T)
    src_buf, tgt_buf = _inputs(S, T, H, seed=T + H, scale_rows=6.0)
    HC, ld = H * C, H * C + 4
    xl_b, xr_b = src_buf(), tgt_buf()
    att = (torch.randn(HC, generator=torch.Generator().manual_seed(H)) * 0.3).cuda()
    tgt_d, src_d, cnt_d = tgt.cuda(), src.cuda().contiguous(), cnt.cuda()
    xr_ptr = xr_b.data_ptr() + ld * 4                                  # row -1 of the kernel's xr = the NaN row
    out = torch.full((T, HC), float("nan"), device="cuda")
    alpha = torch.full((T, 36, H), float("nan"), device="cuda")
    st = _l.current_stream_ptr()
    _l.check(L.mls_gatv2_edge_fwd(xl_b.data_ptr(), ld, xr_ptr, ld, att.data_ptr(), tgt_d.data_ptr(), src_d.data_ptr(),
                                  cnt_d.data_ptr(), T, H, out.data_ptr(), alpha.data_ptr(), st))
    dout = torch.randn(T, HC, device="cuda")
    d_xl = torch.zeros(S + 1, HC, device="cuda")
    d_xr = torch.zeros(T + 1, HC, device="cuda")                       # row 0 = row -1 of the kernel: must stay 0
    nb = L.mls_gatv2_edge_bwd_blocks(T)
    part = torch.empty(nb, HC, device="cuda")
    _l.check(L.mls_gatv2_edge_bwd(xl_b.data_ptr(), ld, xr_ptr, ld, att.data_ptr(), tgt_d.data_ptr(), src_d.data_ptr(),
                                  cnt_d.data_ptr(), T, H, alpha.data_ptr(), dout.data_ptr(), d_xl.data_ptr(),
                                  d_xr.data_ptr() + HC * 4, part.data_ptr(), st))
    # float64 reference on the dense columns (xr row r of the kernel = buffer row r + 1)
    xl = xl_b[:, :HC].double().requires_grad_()
    xr = xr_b[1:, :HC].double().requires_grad_()
    at = att.double().requires_grad_()
    r_out, r_alpha = train_oracle.gatv2_edge_reference(xl, xr, at, tgt_d, src_d, cnt_d, H)
    (r_out * dout.double()).sum().backward()
    errs = {}
    _close("out", out, r_out.detach(), errs)
    valid = (torch.arange(36, device="cuda")[None, :] < cnt_d[:, None]) & (tgt_d >= 0)[:, None]
    _close("alpha", alpha[valid], r_alpha.detach()[valid], errs)
    _close("d_xl", d_xl, xl.grad, errs)
    _close("d_xr", d_xr[1:], xr.grad, errs)
    _close("d_att", part.double().sum(0), at.grad, errs)
    assert float(d_xr[0].abs().max()) == 0.0 and float(d_xl[S].abs().max()) == 0.0
    one = (cnt_d == 1) & (tgt_d >= 0)                                  # a single source: alpha = 1, out = its row
    assert bool((alpha[one, 0] == 1.0).all())
    assert torch.equal(out[one], xl_b[src_d[one, 0].long(), :HC])
    if bool((tgt_d < 0).any()):                                       # absent targets: zeros
        assert float(out[tgt_d < 0].abs().max()) == 0.0
    print(f"gatv2 H={H} T={T}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))


@pytest.mark.parametrize("H,T", EDGE_CASES)
def test_transformer_edge_kernels_match_the_float64_reference(H, T):
    _l, L = _lib()
    torch.manual_seed(T + H)
    tgt, src, cnt, S = _edge_case(T, H, seed=H * 104729 + T)
    src_buf, tgt_buf = _inputs(S, T, H, seed=3 * T + H, scale_rows=15.0)
    HC, ld = H * C, H * C + 4
    k_b, v_b, q_b = src_buf(), src_buf(), tgt_buf()
    tgt_d, src_d, cnt_d = tgt.cuda(), src.cuda().contiguous(), cnt.cuda()
    q_ptr = q_b.data_ptr() + ld * 4
    out = torch.full((T, HC), float("nan"), device="cuda")
    alpha = torch.full((T, 36, H), float("nan"), device="cuda")
    st = _l.current_stream_ptr()
    _l.check(L.mls_transformer_edge_fwd(k_b.data_ptr(), v_b.data_ptr(), ld, q_ptr, ld, tgt_d.data_ptr(), src_d.data_ptr(),
                                        cnt_d.data_ptr(), T, H, out.data_ptr(), alpha.data_ptr(), st))
    dout = torch.randn(T, HC, device="cuda")
    d_k = torch.zeros(S + 1, HC, device="cuda")
    d_v = torch.zeros(S + 1, HC, device="cuda")
    d_q = torch.zeros(T + 1, HC, device="cuda")
    _l.check(L.mls_transformer_edge_bwd(k_b.data_ptr(), v_b.data_ptr(), ld, q_ptr, ld, tgt_d.data_ptr(), src_d.data_ptr(),
                                        cnt_d.data_ptr(), T, H, alpha.data_ptr(), dout.data_ptr(), d_k.data_ptr(),
                                        d_v.data_ptr(), d_q.data_ptr() + HC * 4, st))
    k, v = k_b[:, :HC].double().requires_grad_(), v_b[:, :HC].double().requires_grad_()
    q = q_b[1:, :HC].double().requires_grad_()
    r_out, r_alpha = train_oracle.transformer_edge_reference(q, k, v, tgt_d, src_d, cnt_d, H)
    (r_out * dout.double()).sum().backward()
    errs = {}
    _close("out", out, r_out.detach(), errs)
    e = torch.arange(36, device="cuda")[None, :]
    valid = (e >= 1) & (e < cnt_d[:, None]) & (tgt_d >= 0)[:, None]
    _close("alpha", alpha[valid], r_alpha.detach()[valid], errs)
    _close("d_k", d_k, k.grad, errs)
    _close("d_v", d_v, v.grad, errs)
    _close("d_q", d_q[1:], q.grad, errs)
    assert float(d_q[0].abs().max()) == 0.0 and float(d_k[S].abs().max()) == 0.0 and float(d_v[S].abs().max()) == 0.0
    lone = (cnt_d == 1) & (tgt_d >= 0)                                 # no sources: out = 0, no gradient
    if lone.any():
        assert float(out[lone].abs().max()) == 0.0 and float(d_q[1:][tgt_d[lone].long()].abs().max()) == 0.0
    print(f"transformer H={H} T={T}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs.items()))


@pytest.mark.parametrize("N", [1, 31, 32, 33, 50, 64, 65, 200])
def test_train_lists_follow_the_radius_rule_at_the_edges(N):
    """mls_train_lists modes 0, 1, 2 against net_oracle.radius_graph_mask: complete graphs (lists capped at 32
    neighbours, 33 for nodes outside the first 33 hits), an isolated controlling node, controlling indices below 0,
    past N - 1 and fractional (clamped and truncated like the network's split_rows)."""
    _l, L = _lib()
    bs = 12
    ctrl = np.random.default_rng(N).integers(0, N, size=bs).astype(np.float32)
    ctrl[:4] = [-4.0, N + 7.0, min(3.7, N - 0.3), N - 1]
    rows = train_oracle.agent_rows(N, bs, seed=N, complete=(1, 3, 5), isolated=(2, 6), ctrl=ctrl).cuda()
    pos = rows[:, :-1].view(bs, N, 8)[..., :2]
    mask = no.radius_graph_mask(pos.cpu())
    c = rows[:, -1].cpu().clamp(0, N - 1).long()
    cap, st, r2 = L.mls_train_list_capacity(), _l.current_stream_ptr(), no.r2_threshold()
    want_lists = lambda b, i: [b * N + i] + [b * N + j for j in torch.nonzero(mask[b, i]).flatten().tolist()]
    s1_cnt = torch.full((bs,), -1, dtype=torch.int32, device="cuda")
    _l.check(L.mls_train_lists(rows.data_ptr(), rows.shape[1], bs, N, r2, 0, s1_cnt.data_ptr(), None, None, None, None, None, st))
    assert s1_cnt.tolist() == [1 + int(mask[b, c[b]].sum()) for b in range(bs)]
    if N > 33:
        assert int(s1_cnt[3]) == 34                                             # node N-1 of a complete graph: 33 neighbours
    assert int(s1_cnt[2]) == 1 and int(s1_cnt[6]) == 1                          # isolated controlling node
    base = (torch.cumsum(s1_cnt.long(), 0) - s1_cnt.long()).contiguous()
    n_slots = int(s1_cnt.sum())
    tgt_row = torch.full((n_slots,), -7, dtype=torch.int32, device="cuda")
    src_row = torch.full((n_slots, cap), -7, dtype=torch.int32, device="cuda")
    src_cnt = torch.full((n_slots,), -7, dtype=torch.int32, device="cuda")
    used = torch.zeros(bs * N, dtype=torch.uint8, device="cuda")
    _l.check(L.mls_train_lists(rows.data_ptr(), rows.shape[1], bs, N, r2, 1, None, base.data_ptr(), tgt_row.data_ptr(),
                               src_row.data_ptr(), src_cnt.data_ptr(), used.data_ptr(), st))
    want_used = torch.zeros(bs * N, dtype=torch.uint8)
    tgt_row, src_row, src_cnt = tgt_row.cpu(), src_row.cpu(), src_cnt.cpu()
    for b in range(bs):
        s1 = [int(c[b])] + torch.nonzero(mask[b, c[b]]).flatten().tolist()
        lo = int(base[b])
        assert (tgt_row[lo:lo + len(s1)] - b * N).tolist() == s1
        for k, i in enumerate(s1):
            want = want_lists(b, i)
            assert int(src_cnt[lo + k]) == len(want) and src_row[lo + k, :len(want)].tolist() == want
            want_used[want] = 1
    assert torch.equal(used.cpu(), want_used)
    # mode 2: every node's list, slot = node row
    tgt2 = torch.full((bs * N,), -7, dtype=torch.int32, device="cuda")
    src2 = torch.full((bs * N, cap), -7, dtype=torch.int32, device="cuda")
    cnt2 = torch.full((bs * N,), -7, dtype=torch.int32, device="cuda")
    _l.check(L.mls_train_lists(rows.data_ptr(), rows.shape[1], bs, N, r2, 2, None, None, tgt2.data_ptr(), src2.data_ptr(),
                               cnt2.data_ptr(), None, st))
    assert tgt2.cpu().tolist() == list(range(bs * N))
    assert cnt2.cpu().tolist() == (1 + mask.sum(2)).flatten().tolist()
    src2_h = src2.cpu()
    for b in range(bs):
        for i in range(N):
            want = want_lists(b, i)
            assert src2_h[b * N + i, :len(want)].tolist() == want


@pytest.mark.parametrize("wd", [0.0, 0.01])
@pytest.mark.parametrize("n", [1, 255, 257, (1 << 20) + 13])
def test_adam_kernel_one_step_at_a_time_in_float64(n, wd):
    """mls_adam_step on raw buffers: sizes around a block and past three grid passes of 148 * 8 * 256; steps with bias
    corrections near 0 and near 1.  Each step is compared with float64 Adam started from the kernel's own fp32 state, so
    errors do not accumulate (largest measured on a B200: 7.3e-7 for p, a few fp32 ulps).  The ABI takes fp32 hyperparameters: the reference uses those values (fp32(0.999) makes
    1 - beta2 differ from 0.001 by 1.3e-5 relative, far more than the kernel's rounding)."""
    _l, L = _lib()
    f32 = lambda x: float(np.float32(x))
    lr, b1, b2, eps, gs = f32(1e-3), f32(0.9), f32(0.999), f32(1e-8), 0.125
    wd = f32(wd)
    rng = np.random.default_rng(n)
    pad = 64                                                           # sentinel tail: nothing past n may change
    p = torch.full((n + pad,), 7.0, device="cuda")
    m, v = torch.full_like(p, 7.0), torch.full_like(p, 7.0)
    p[:n] = torch.as_tensor(rng.standard_normal(n).astype(np.float32))
    m[:n] = 0.0
    v[:n] = 0.0
    st = _l.current_stream_ptr()
    worst = {"p": 0.0, "m": 0.0, "v": 0.0}
    for step in (1, 2, 10, 1000, 10 ** 6):
        g = (rng.standard_normal(n) * 10.0 ** rng.integers(-3, 3, size=n)).astype(np.float32)
        special = np.array([0.0, 1e-20, -1e-20, 1e4, -1e4], dtype=np.float32)
        g[: min(n, 5)] = special[: min(n, 5)]
        g[rng.integers(0, n, size=min(n, 64))] = special[rng.integers(0, 5, size=min(n, 64))]
        grad = torch.full((n + pad,), 7.0, device="cuda")
        grad[:n] = torch.as_tensor(g)
        p0, m0, v0 = (x[:n].double().cpu().numpy() for x in (p, m, v))
        _l.check(L.mls_adam_step(p.data_ptr(), grad.data_ptr(), m.data_ptr(), v.data_ptr(), n, lr, b1, b2, eps, wd, step, gs, st))
        wp, wm, wv = train_oracle.adam_reference(p0, [g.astype(np.float64) * gs], lr=lr, betas=(b1, b2), eps=eps,
                                                 weight_decay=wd, state=(m0, v0, step - 1))
        gp, gm, gv = (x[:n].double().cpu().numpy() for x in (p, m, v))
        gw = g.astype(np.float64) * gs + wd * p0
        # bounds scale with the magnitudes of each update's terms (no cancellation can hide behind a small result)
        with np.errstate(invalid="ignore"):                                # 0 / 0 where both terms are exactly 0
            em = np.nan_to_num(np.abs(gm - wm) / (b1 * np.abs(m0) + (1 - b1) * np.abs(gw)), nan=0.0)
        ev = np.abs(gv - wv) / np.maximum(wv, 1e-30 / 1e-6)
        ep = np.abs(gp - wp) / (np.abs(p0) + np.abs(p0 - wp))
        for k, e in (("p", ep), ("m", em), ("v", ev)):
            worst[k] = max(worst[k], float(e.max()))
            assert float(e.max()) <= 1e-6, f"{k} at step {step}: relative error {float(e.max()):.3e}"
        for x in (p, m, v):
            assert bool((x[n:] == 7.0).all())
    print(f"adam n={n} wd={wd}: " + ", ".join(f"{k} {e:.2e}" for k, e in worst.items()))
