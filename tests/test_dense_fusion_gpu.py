"""GPU: the fused dense layers around conv2 (csrc/gemm_tcgen05.cu) against the launches they replace, bit for bit.

* Both conv2 projections in one split launch vs two calls of the plain GEMM entry (source columns on the needed rows,
  target columns on the controlling rows): Psrc, Ptgt and both dot arrays.
* The fused 128-wide dueling heads vs head0 (MODE 2) -> head1 (MODE 3) through the GEMM entry, then the output layer,
  dueling combination and epsilon-greedy action in torch / numpy (Philox4x32-10 re-implemented here): Q and actions.
Both fusions keep every MMA shape, K order and rounding point, so nothing may differ in any bit."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

vp = C.c_void_p
HC, NODES = 512, 50


def _L():
    from melissa_b200 import _lib
    L = _lib.lib()
    L.mls_test_gemm_bf16_ex.argtypes = [vp, vp, vp, vp, C.c_longlong, C.c_int, vp, vp, vp, vp, vp, C.c_int, vp,
                                        C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]
    L.mls_test_gemm_bf16_ex.restype = C.c_int
    L.mls_test_conv2_proj.argtypes = [vp, C.c_int, vp, C.c_int, vp, vp, vp, C.c_longlong, C.c_int, vp, vp, vp, vp, vp, vp, vp,
                                      C.c_int, C.c_int, C.c_int, vp, vp, vp]
    L.mls_test_conv2_proj.restype = C.c_int
    L.mls_test_head_dueling.argtypes = [vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp,
                                        vp, vp, vp, C.c_longlong, C.c_int, vp, vp, C.c_int, C.c_float, C.c_ulonglong,
                                        C.c_ulonglong, vp, vp]
    L.mls_test_head_dueling.restype = C.c_int
    return _lib, L


def _gemm_ex(A, B, bias, C_out, M, m_dev, obs=None, row_index=None, dotvec=None, dots=None, dotvec2=None, dots2=None,
             dot_relu=0, relu=0):
    _lib, L = _L()
    N, K = B.shape
    _lib.check(L.mls_test_gemm_bf16_ex(A.data_ptr(), B.data_ptr(), bias.data_ptr(), _lib.ptr(obs), NODES * 8 if obs is not None else 0,
                                       NODES, _lib.ptr(row_index), _lib.ptr(dotvec), _lib.ptr(dotvec2), _lib.ptr(dots), _lib.ptr(dots2),
                                       dot_relu, _lib.ptr(C_out), M, N, K, relu, _lib.ptr(m_dev), _lib.current_stream_ptr()))


def _bits_equal(a, b):
    a, b = a.contiguous(), b.contiguous()
    if a.dtype == torch.bfloat16:
        return torch.equal(a.view(torch.int16), b.view(torch.int16))
    return torch.equal(a.view(torch.int32), b.view(torch.int32))


# ---------------------------------------------------------------------------------------------- conv2 projections
@pytest.mark.parametrize("nproj", [2, 3], ids=["gatv2", "transformer"])
@pytest.mark.parametrize("count", [0, 700, 256, 301], ids=["count0", "count_eq_ntotal", "count_x128", "count_odd"])
@pytest.mark.parametrize("scaled", [False, True], ids=["noscale", "rowscale"])
@pytest.mark.parametrize("a2", [False, True], ids=["x1", "a2"])
def test_split_projection_matches_two_launches(nproj, count, scaled, a2):
    _lib, L = _L()
    M, ntotal, graphs = 1000, 700, 40                 # device-side row counts below M; node rows = 40 graphs x 50 nodes
    g = torch.Generator(device="cuda").manual_seed(nproj * 1000 + count + 7 * scaled + 13 * a2)
    x1 = (torch.randn(M, HC, device="cuda", generator=g) * 0.5).to(torch.bfloat16)
    W = (torch.randn(nproj * HC, HC, device="cuda", generator=g) / 16).to(torch.bfloat16)
    bias = torch.randn(nproj * HC, device="cuda", generator=g)
    att = torch.randn(nproj * HC, device="cuda", generator=g) if nproj == 2 else None
    obs = torch.rand(graphs, NODES, 8, device="cuda", generator=g) if scaled else None
    if scaled:
        obs[:, :, 7] = (torch.rand(graphs, NODES, device="cuda", generator=g) < 0.6).float()
    nidx = torch.randint(0, graphs * NODES, (M,), device="cuda", dtype=torch.int32, generator=g) if scaled else None
    idx = torch.randint(0, graphs * NODES, (M,), device="cuda", dtype=torch.int32, generator=g) if scaled else None
    # target rows: x1 itself, or (controlling rows kept apart) the snapshot columns of a wider matrix
    z = (torch.randn(M, 128 + 2 * HC, device="cuda", generator=g) * 0.5).to(torch.bfloat16) if a2 else None
    tgt_A = z[:, 128:128 + HC].contiguous() if a2 else x1
    m_src = torch.tensor([ntotal], dtype=torch.int32, device="cuda")
    m_tgt = torch.tensor([count], dtype=torch.int32, device="cuda")
    nsrc = nproj - 1
    src = slice(HC, 3 * HC) if nproj == 3 else slice(0, HC)
    tgt = slice(0, HC) if nproj == 3 else slice(HC, 2 * HC)

    def outs():
        return (torch.full((M, nsrc * HC), float("nan"), dtype=torch.bfloat16, device="cuda"),
                torch.full((M, HC), float("nan"), dtype=torch.bfloat16, device="cuda"),
                torch.full((M, nsrc * HC // 128), float("nan"), device="cuda") if att is not None else None,
                torch.full((M, HC // 128), float("nan"), device="cuda") if att is not None else None)

    Ps_ref, Pt_ref, ab_ref, dt_ref = outs()
    _gemm_ex(x1, W[src].contiguous(), bias[src].contiguous(), Ps_ref, M, m_src, obs, nidx,
             att[src].contiguous() if att is not None else None, ab_ref)
    _gemm_ex(tgt_A, W[tgt].contiguous(), bias[tgt].contiguous(), Pt_ref, M, m_tgt, obs, idx,
             att[tgt].contiguous() if att is not None else None, dt_ref)
    Ps, Pt, ab, dt = outs()
    _lib.check(L.mls_test_conv2_proj(x1.data_ptr(), HC, z[:, 128:].data_ptr() if a2 else None, z.shape[1] if a2 else 0, W.data_ptr(),
                                     bias.data_ptr(), _lib.ptr(obs), NODES * 8 if scaled else 0, NODES, _lib.ptr(nidx), _lib.ptr(idx),
                                     _lib.ptr(att), _lib.ptr(ab), _lib.ptr(dt), Ps.data_ptr(), Pt.data_ptr(), M, HC, nproj,
                                     m_src.data_ptr(), m_tgt.data_ptr(), _lib.current_stream_ptr()))
    torch.cuda.synchronize()
    assert _bits_equal(Ps, Ps_ref)
    assert _bits_equal(Pt, Pt_ref)
    assert torch.isnan(Pt[(count + 127) // 128 * 128:].float()).all()     # no target rows past the device-side count
    if att is not None:
        assert _bits_equal(ab, ab_ref)
        assert _bits_equal(dt, dt_ref)


# ---------------------------------------------------------------------------------------------- dueling heads
def _philox(key, ctr_lo, ctr_hi):
    m32 = np.uint64(0xFFFFFFFF)
    key, ctr_hi = np.uint64(key), np.uint64(ctr_hi)
    k0, k1 = key & m32, key >> np.uint64(32)
    c0, c1 = ctr_lo & m32, ctr_lo >> np.uint64(32)
    c2 = np.full_like(ctr_lo, ctr_hi & m32)
    c3 = np.full_like(ctr_lo, ctr_hi >> np.uint64(32))
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & m32, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & m32
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & m32, (k1 + np.uint64(0xBB67AE85)) & m32
    return c0, c1, c2, c3


def _actions(q, orow, eps, seed, offset, rand3):
    q = q.cpu().numpy()
    act = (q[:, 1] > q[:, 0]).astype(np.int8)
    eps32 = float(np.float32(eps))
    if abs(eps32) > 1e-8:
        if rand3 is not None:
            r = rand3.cpu().numpy()[orow]
            ue, u0, u1 = r[:, 0], r[:, 1], r[:, 2]
        else:
            v0, v1, v2, v3 = _philox(seed, orow.astype(np.uint64), offset)
            ue = ((v0 >> np.uint64(5)) << np.uint64(26) | (v1 >> np.uint64(6))).astype(np.float64) * (1.0 / 9007199254740992.0)
            u0, u1 = v2.astype(np.float64) / 4294967296.0, v3.astype(np.float64) / 4294967296.0
        act = np.where(ue < eps32, ((u1 + 1.0) > (u0 + 1.0)).astype(np.int8), act)
    return act


@pytest.mark.parametrize("rows", [0, 1, 127, 128, 129, 9001])
@pytest.mark.parametrize("out_mode", [0, 1, 2])
@pytest.mark.parametrize("a2", [False, True], ids=["z", "z_x1"])
@pytest.mark.parametrize("eps", ["greedy", "rand3", "philox"])
def test_fused_head_matches_gemm_chain(rows, out_mode, a2, eps):
    _lib, L = _L()
    hid, K, hh = 128, 128 + 2 * HC, 128
    M = rows + 64                                     # device-side row count below M
    g = torch.Generator(device="cuda").manual_seed(rows * 31 + out_mode * 7 + a2)
    z = (torch.randn(M, K, device="cuda", generator=g) * 0.5).to(torch.bfloat16)
    x1 = (torch.randn(M, HC, device="cuda", generator=g) * 0.5).to(torch.bfloat16) if a2 else None
    if a2:
        z[:, hid:hid + HC] = float("nan")             # the kernel must take these columns from x1
    A_ref = z.clone()
    if a2:
        A_ref[:, hid:hid + HC] = x1
    w_h0 = (torch.randn(2 * hh, K, device="cuda", generator=g) / K ** 0.5).to(torch.bfloat16)
    w_h1 = torch.zeros(2 * hh, 2 * hh, device="cuda")
    w_h1[:hh, :hh] = torch.randn(hh, hh, device="cuda", generator=g) / hh ** 0.5
    w_h1[hh:, hh:] = torch.randn(hh, hh, device="cuda", generator=g) / hh ** 0.5
    w_h1 = w_h1.to(torch.bfloat16)
    b_h0, b_h1 = torch.randn(2 * hh, device="cuda", generator=g) * 0.1, torch.randn(2 * hh, device="cuda", generator=g) * 0.1
    q_w2, v_w2 = torch.randn(2, hh, device="cuda", generator=g) * 0.1, torch.randn(hh, device="cuda", generator=g) * 0.1
    hv1 = torch.cat([q_w2[0], v_w2]).contiguous()
    hv2 = torch.cat([q_w2[1], torch.zeros(hh, device="cuda")]).contiguous()
    bq, bv = torch.randn(2, device="cuda", generator=g), torch.randn(1, device="cuda", generator=g)
    m_dev = torch.tensor([rows], dtype=torch.int32, device="cuda")
    graphs = max(rows, 1) + 5
    row0 = 3 * NODES
    if out_mode == 0:
        idx = torch.randperm(graphs * NODES, device="cuda", generator=g)[:M].to(torch.int32)
        n_out = row0 + graphs * NODES
    elif out_mode == 1:
        idx = (torch.arange(M, device="cuda") * NODES + torch.randint(0, NODES, (M,), device="cuda", generator=g)).to(torch.int32)
        n_out = row0 // NODES + M
    else:
        idx, n_out = None, M
    eps_v = 0.0 if eps == "greedy" else 0.3
    seed, offset = 0x1234ABCD5678, 977
    rand3 = torch.rand(n_out, 3, device="cuda", dtype=torch.float64, generator=g) if eps == "rand3" else None

    # reference: head0 (MODE 2) -> head1 (MODE 3) -> output layer, dueling mean and action
    hid1 = torch.full((M, 2 * hh), float("nan"), dtype=torch.bfloat16, device="cuda")
    _gemm_ex(A_ref, w_h0, b_h0, hid1, M, m_dev, relu=1)
    dots = torch.full((M, 2), float("nan"), device="cuda")
    dots2 = torch.full((M, 2), float("nan"), device="cuda")
    _gemm_ex(hid1, w_h1, b_h1, None, M, m_dev, dotvec=hv1, dots=dots, dotvec2=hv2, dots2=dots2, dot_relu=1, relu=1)
    s0, sv, s1 = dots[:rows, 0] + bq[0], dots[:rows, 1] + bv[0], dots2[:rows, 0] + bq[1]
    mean = (s0 + s1) / 2.0
    o = torch.stack([(s0 - mean) + sv, (s1 - mean) + sv], 1)
    t = torch.arange(rows, device="cuda")
    orow = (row0 + idx[:rows].long() if out_mode == 0 else row0 // NODES + idx[:rows].long() // NODES if out_mode == 1 else t)
    q_ref = torch.full((n_out, 2), float("nan"), device="cuda")
    q_ref[orow] = o
    act_ref = torch.full((n_out,), 77, dtype=torch.int8, device="cuda")
    if out_mode != 2 and rows:
        act_ref[orow] = torch.from_numpy(_actions(o, orow.cpu().numpy(), eps_v, seed, offset, rand3)).cuda()

    q = torch.full((n_out, 2), float("nan"), device="cuda")
    act = torch.full((n_out,), 77, dtype=torch.int8, device="cuda")
    _lib.check(L.mls_test_head_dueling(z.data_ptr(), K, _lib.ptr(x1), HC, hid if a2 else 0, hid + HC if a2 else 0, M, K, m_dev.data_ptr(),
                                       w_h0.data_ptr(), b_h0.data_ptr(), w_h1.data_ptr(), b_h1.data_ptr(), hv1.data_ptr(), hv2.data_ptr(),
                                       bq.data_ptr(), bv.data_ptr(), _lib.ptr(idx), row0 if out_mode != 2 else 0, NODES, q.data_ptr(),
                                       act.data_ptr() if out_mode != 2 else None, out_mode, eps_v, seed, offset, _lib.ptr(rand3),
                                       _lib.current_stream_ptr()))
    torch.cuda.synchronize()
    assert _bits_equal(q, q_ref)
    assert torch.equal(act, act_ref)
