"""GPU: the persistent tensor-core kernels past one tile per CTA.

Every hot kernel of the rollout round walks tiles (or items) blockIdx.x, blockIdx.x + gridDim.x, ... and carries state from one
to the next: double-buffered TMEM accumulators and column slices, a row scale fetched a tile ahead, prefetched graph metadata,
stage rings that wrap after several items.  At the sizes of the other tests most CTAs see one tile.  Here the test-only option
"max_ctas" caps the grid of every persistent launcher, so that small inputs give every CTA many tiles, with tile counts
cap * k + r (k >= 4, r != 0 where the layout allows it) so that CTAs end on both accumulator parities; one uncapped run per family
has at least two tiles per SM.

* The GEMM (every instantiation the dispatcher in gemm_bf16_launch picks) and the fused dueling head against float64 references
  of the same bf16 operands, with a first-order error bound computed from the data.  Inputs make a wrong-tile read visible:
  distinct non-binary row scales through a permuted row index, bias and dot vectors that differ per 256-column slice, device row
  counts in the middle of a tile, NaN in the outputs the kernel must not write.
* The forward is invariant to the grid: Q-values and actions bit for bit at caps H, 2H, 3H, 7H and uncapped, on inputs that reach
  the item boundaries of conv2 and the conv1 table kernels.  Every kernel's arithmetic for an item belongs to one CTA, and the
  GEMM's two-term dot atomics onto a zeroed cell are order-free, so nothing may differ.
* The fp32 tensor-core route (the parity anchor) at caps 1 and 2 against the fp32 oracle at its 1e-5 bar.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from test_dense_fusion_gpu import _actions
from test_dense_fusion_gpu import test_fused_head_matches_gemm_chain as _head_chain_bits
from test_dense_fusion_gpu import test_split_projection_matches_two_launches as _split_bits

pytestmark = pytest.mark.gpu

vp = C.c_void_p
CAPS = [1, 2, 3, 5]
U23 = 2.0 ** -23
NODES = 50


def _L():
    from melissa_b200 import _lib
    L = _lib.lib()
    L.mls_test_gemm_bf16_full.argtypes = [vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp, C.c_longlong, C.c_int, vp, vp, vp,
                                          vp, vp, C.c_int, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]
    L.mls_test_gemm_bf16_full.restype = C.c_int
    L.mls_test_conv2_proj.argtypes = [vp, C.c_int, vp, C.c_int, vp, vp, vp, C.c_longlong, C.c_int, vp, vp, vp, vp, vp, vp, vp,
                                      C.c_int, C.c_int, C.c_int, vp, vp, vp]
    L.mls_test_conv2_proj.restype = C.c_int
    L.mls_test_head_dueling.argtypes = [vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp,
                                        vp, vp, vp, C.c_longlong, C.c_int, vp, vp, C.c_int, C.c_float, C.c_ulonglong,
                                        C.c_ulonglong, vp, vp]
    L.mls_test_head_dueling.restype = C.c_int
    return _lib, L


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


class _Cap:
    """Option max_ctas for the duration of a with-block (0 = uncapped), restored even when the block fails."""

    def __init__(self, cap):
        self.cap = cap

    def __enter__(self):
        from melissa_b200 import _lib
        self.old = _lib.get_option("max_ctas")
        _lib.set_option("max_ctas", self.cap)

    def __exit__(self, *exc):
        from melissa_b200 import _lib
        _lib.set_option("max_ctas", self.old)


def _tile_count(cap, ok):
    """Smallest tile count cap * k + r (k >= 4, 0 < r < cap; cap 1: k >= 5) that the layout can form (ok(T)); when no such
    count exists (a layout whose tile count is a multiple of cap), the smallest T >= 4 cap + 1 it can form."""
    lo = 4 * cap + 1
    for T in range(lo, lo + 64 * cap):
        if (cap == 1 or T % cap) and ok(T):
            return T
    return next(T for T in range(lo, lo + 64 * cap) if ok(T))


def _bf16(x):
    return x.to(torch.bfloat16)


def _scales(rows, g):
    """Distinct non-binary row scales 1 + r / rows in a random order: obs[graph, node, 7]."""
    graphs = (rows + NODES - 1) // NODES
    dm = 1.0 + torch.randperm(graphs * NODES, device="cuda", generator=g).float() / (graphs * NODES)
    obs = torch.rand(graphs, NODES, 8, device="cuda", generator=g)
    obs[:, :, 7] = dm.view(graphs, NODES)
    return obs


def _slice_vec(n, g, scale=1.0):
    """A vector whose 256-column slices differ by far more than any tolerance below."""
    return (torch.randn(n, device="cuda", generator=g) * 0.1 + (torch.arange(n, device="cuda") // 256 + 1).float() * 0.5) * scale


def _ratio(err, tol):
    return float((err / tol).max()) if err.numel() else 0.0


class _Worst:
    """Largest err / tol per case, printed at the end of each test (run with -s to see it)."""

    def __init__(self, what):
        self.what, self.r = what, {}

    def add(self, key, err, tol):
        r = _ratio(err, tol)
        self.r[key] = max(self.r.get(key, 0.0), r)
        assert r <= 1.0, f"{self.what} {key}: err / tol = {r:.3f} (max err {float(err.max()):.3e})"

    def report(self):
        print(f"\n{self.what}: largest err/tol " + ", ".join(f"{k} {v:.3f}" for k, v in self.r.items()))


def _check_segment(worst, key, out, x64, S64, K, live, relu, fp32=False):
    """out rows [0, live) against the float64 epilogue value x64 (pre-ReLU) with accumulation bound K 2^-23 S64; rows past
    live must still hold the NaN they started with."""
    ref = x64.clamp_min(0) if relu else x64
    acc = K * U23 * S64[:live]
    got = out[:live].double()
    tol = (U23 if fp32 else 2.0 ** -8) * (ref[:live].abs() + acc) + acc + 1e-30    # rounding of a value up to |ref| + acc
    worst.add(key, (got - ref[:live]).abs(), tol)
    assert torch.isnan(out[live:].float()).all(), f"{key}: rows past the device row count were written"


def _check_dots(worst, key, dots, x64, S64, K, dv, live, dot_relu):
    """dots[m][g] = sum over the 128 columns of group g of y * dv, y = relu?(x): each column's bound K 2^-23 S (+ the fp32
    rounding of y) through |dv|, plus the fp32 accumulation of the 128 products; rows past live stay 0."""
    y = x64.clamp_min(0) if dot_relu else x64
    M, N = x64.shape
    want = (y * dv.double()[None, :]).view(M, N // 128, 128).sum(2)
    ey = (K * U23 * S64 + U23 * x64.abs()) * dv.double().abs()[None, :]
    prod = (y * dv.double()[None, :]).abs()
    tol = ey.view(M, N // 128, 128).sum(2) + 130 * 2.0 ** -24 * prod.view(M, N // 128, 128).sum(2) + 1e-30
    worst.add(key, (dots[:live].double() - want[:live]).abs(), tol[:live])
    assert (dots[live:] == 0).all(), f"{key}: dots past the device row count"


# ---------------------------------------------------------------------------------------------- GEMM, plain launch
# mode name -> (BN, flags).  The flag combination is what gemm_bf16_launch's dispatcher maps to each instantiation.
PLAIN = {
    "bn256_mode0": dict(bn=256, c=True, cf=True, relu=1, dot=True, dot2=False, dot_relu=0),   # Cf: run-time options
    "bn256_mode1": dict(bn=256, c=True, cf=False, relu=0, dot=True, dot2=False, dot_relu=0),  # C + one dot on raw values
    "bn256_mode2": dict(bn=256, c=True, cf=False, relu=1, dot=False, dot2=False, dot_relu=0),  # hidden layer
    "bn256_mode3": dict(bn=256, c=False, cf=False, relu=1, dot=True, dot2=True, dot_relu=1),   # dots only, on relu(x)
    "bn128_mode0": dict(bn=128, c=True, cf=True, relu=1, dot=False, dot2=False, dot_relu=0),   # N not a multiple of 256
}


def _plain_case(mode, cap, T_min=None, seed=0):
    _lib, L = _L()
    o = PLAIN[mode]
    K, k2_lo, k2_hi = 256, 64, 192
    # column tiles per M tile: 3, or when cap is a multiple of 3, 2 (BN 256) / 5 (BN 128: N must not be a multiple of 256),
    # so that consecutive tiles of a CTA take different column slices (a slice read from the wrong buffer changes the values)
    n_n = 3 if cap % 3 else (2 if o["bn"] == 256 else 5)
    if T_min is None:
        T = _tile_count(cap, lambda T: T % n_n == 0)
    else:
        T = (T_min + n_n - 1) // n_n * n_n
    n_m = T // n_n
    N = n_n * o["bn"]
    live = (n_m - 1) * 128 + 77                           # device row count in the middle of the last M tile
    M = n_m * 128 + 150                                   # tiles past it are never computed
    g = torch.Generator(device="cuda").manual_seed(seed * 7919 + cap * 31 + len(mode))
    A = _bf16(torch.randn(M, K, device="cuda", generator=g) * 0.5)
    A2 = _bf16(torch.randn(M, 200, device="cuda", generator=g) * 0.5)       # row stride 200: columns [k2_lo, k2_hi) of A
    A[:, k2_lo:k2_hi] = float("nan")                       # ... which the kernel must take from A2
    B = _bf16(torch.randn(N, K, device="cuda", generator=g) / 16)
    bias = _slice_vec(N, g)
    obs = _scales(M, g)
    ridx = torch.randperm(obs.shape[0] * NODES, device="cuda", generator=g)[:M].to(torch.int32)
    dv = _slice_vec(N, g, 0.1) if o["dot"] else None
    dv2 = -_slice_vec(N, g, 0.1) if o["dot2"] else None
    Cb = torch.full((M, N), float("nan"), dtype=torch.bfloat16, device="cuda") if o["c"] else None
    Cf = torch.full((M, N), float("nan"), device="cuda") if o["cf"] else None
    dots = torch.full((M, N // 128), float("nan"), device="cuda") if o["dot"] else None
    dots2 = torch.full((M, N // 128), float("nan"), device="cuda") if o["dot2"] else None
    m_dev = torch.tensor([live], dtype=torch.int32, device="cuda")
    with _Cap(cap):
        _lib.check(L.mls_test_gemm_bf16_full(A.data_ptr(), K, A2.data_ptr(), 200, k2_lo, k2_hi, B.data_ptr(), bias.data_ptr(),
                                             obs.data_ptr(), NODES * 8, NODES, ridx.data_ptr(), _lib.ptr(dv), _lib.ptr(dv2),
                                             _lib.ptr(dots), _lib.ptr(dots2), o["dot_relu"], _lib.ptr(Cb), _lib.ptr(Cf), M, N, K,
                                             o["relu"], m_dev.data_ptr(), _lib.current_stream_ptr()))
        torch.cuda.synchronize()
    Al = A.clone()
    Al[:, k2_lo:k2_hi] = A2[:, :k2_hi - k2_lo]
    scale = obs.reshape(-1, 8)[ridx.long(), 7].double()[:, None]
    x64 = scale * (Al.double() @ B.double().T) + bias.double()[None, :]
    S64 = scale.abs() * (Al.double().abs() @ B.double().abs().T)
    worst = _Worst(f"GEMM {mode} cap {cap} ({T} tiles)")
    if Cb is not None:
        _check_segment(worst, "C", Cb, x64, S64, K, live, o["relu"])
    if Cf is not None:
        _check_segment(worst, "Cf", Cf, x64, S64, K, live, o["relu"], fp32=True)
    if dots is not None:
        _check_dots(worst, "dots", dots, x64, S64, K, dv, live, o["dot_relu"])
    if dots2 is not None:
        _check_dots(worst, "dots2", dots2, x64, S64, K, dv2, live, o["dot_relu"])
    worst.report()


@pytest.mark.parametrize("cap", CAPS)
@pytest.mark.parametrize("mode", list(PLAIN))
def test_gemm_plain_modes_many_tiles_per_cta(mode, cap):
    _plain_case(mode, cap)


@pytest.mark.parametrize("mode", list(PLAIN))
def test_gemm_plain_modes_uncapped_two_tiles_per_sm(mode):
    _plain_case(mode, 0, T_min=2 * _sms() + 5, seed=1)


# ---------------------------------------------------------------------------------------------- GEMM, split launch
# (HC, nproj) -> instantiation: GATv2 HC 512 -> <256, 4>; Transformer HC 512 -> <256, 5>; Transformer HC 384 -> <128, 5>
SPLIT = {"bn256_mode4": (512, 2), "bn256_mode5": (512, 3), "bn128_mode5": (384, 3)}


def _split_case(mode, cap, T_min=None, seed=0):
    _lib, L = _L()
    HC, nproj = SPLIT[mode]
    BN = 128 if HC % 256 else 256
    N = nproj * HC
    n_n, n_ns = N // BN, (N - HC) // BN

    def count(n_m, n_mt):
        return n_mt * n_n + (n_m - n_mt) * n_ns

    # both row ranges end mid-tile, target rows below source rows; choose the smallest layout with the wanted tile count
    layouts = {}
    for n_m in range(2, 200):
        for n_mt in range(1, n_m):
            layouts.setdefault(count(n_m, n_mt), (n_m, n_mt))
    if T_min is None:
        T = _tile_count(cap, lambda T: T in layouts)
    else:
        T = min(T for T in layouts if T >= T_min)
    n_m, n_mt = layouts[T]
    live_s, live_t = (n_m - 1) * 128 + 93, (n_mt - 1) * 128 + 41
    M = n_m * 128 + 100
    g = torch.Generator(device="cuda").manual_seed(seed * 7919 + cap * 37 + HC + nproj)
    x1 = _bf16(torch.randn(M, HC, device="cuda", generator=g) * 0.5)
    zw = HC + 64
    z = _bf16(torch.randn(M, zw, device="cuda", generator=g) * 0.5)          # target operand: A2 with its own row stride
    W = _bf16(torch.randn(N, HC, device="cuda", generator=g) / 16)
    bias = _slice_vec(N, g)
    att = _slice_vec(N, g, 0.1) if nproj == 2 else None
    obs = _scales(M, g)
    nidx = torch.randperm(obs.shape[0] * NODES, device="cuda", generator=g)[:M].to(torch.int32)
    tidx = torch.randperm(obs.shape[0] * NODES, device="cuda", generator=g)[:M].to(torch.int32)
    nsrc = nproj - 1
    Ps = torch.full((M, nsrc * HC), float("nan"), dtype=torch.bfloat16, device="cuda")
    Pt = torch.full((M, HC), float("nan"), dtype=torch.bfloat16, device="cuda")
    ab = torch.full((M, nsrc * HC // 128), float("nan"), device="cuda") if att is not None else None
    dt = torch.full((M, HC // 128), float("nan"), device="cuda") if att is not None else None
    m_src = torch.tensor([live_s], dtype=torch.int32, device="cuda")
    m_tgt = torch.tensor([live_t], dtype=torch.int32, device="cuda")
    with _Cap(cap):
        _lib.check(L.mls_test_conv2_proj(x1.data_ptr(), HC, z.data_ptr(), zw, W.data_ptr(), bias.data_ptr(), obs.data_ptr(), NODES * 8,
                                         NODES, nidx.data_ptr(), tidx.data_ptr(), _lib.ptr(att), _lib.ptr(ab), _lib.ptr(dt),
                                         Ps.data_ptr(), Pt.data_ptr(), M, HC, nproj, m_src.data_ptr(), m_tgt.data_ptr(),
                                         _lib.current_stream_ptr()))
        torch.cuda.synchronize()
    tgt = slice(0, HC) if nproj == 3 else slice(HC, 2 * HC)
    src = torch.cat([torch.arange(N, device="cuda")[:tgt.start], torch.arange(N, device="cuda")[tgt.stop:]])
    flat = obs.reshape(-1, 8)[:, 7].double()
    worst = _Worst(f"GEMM {mode} cap {cap} ({T} tiles)")
    for key, A_op, idx, cols, out, dout, live in (("source", x1, nidx, src, Ps, ab, live_s),
                                                  ("target", z[:, :HC], tidx, torch.arange(N, device="cuda")[tgt], Pt, dt, live_t)):
        sc = flat[idx.long()][:, None]
        Wc = W[cols].double()
        x64 = sc * (A_op.double() @ Wc.T) + bias[cols].double()[None, :]
        S64 = sc.abs() * (A_op.double().abs() @ Wc.abs().T)
        _check_segment(worst, key, out, x64, S64, HC, live, relu=False)
        if dout is not None:
            _check_dots(worst, key + " dots", dout, x64, S64, HC, att[cols], live, dot_relu=False)
    worst.report()


@pytest.mark.parametrize("cap", CAPS)
@pytest.mark.parametrize("mode", list(SPLIT))
def test_gemm_split_modes_many_tiles_per_cta(mode, cap):
    _split_case(mode, cap)


@pytest.mark.parametrize("mode", list(SPLIT))
def test_gemm_split_modes_uncapped_two_tiles_per_sm(mode):
    _split_case(mode, 0, T_min=2 * _sms() + 5, seed=1)


@pytest.mark.parametrize("cap", [2, 5])
@pytest.mark.parametrize("nproj", [2, 3], ids=["gatv2", "transformer"])
def test_split_projection_bit_identity_at_several_tiles_per_cta(nproj, cap):
    """The existing split-vs-two-launches bit identity (M = 1000 rows), with every CTA taking several tiles on both sides."""
    with _Cap(cap):
        _split_bits(nproj, 301, True, True)


# ---------------------------------------------------------------------------------------------- fused dueling head
def _ulp_bf16(x):
    """One bf16 ulp of |x| (2^(e - 7) for |x| in [2^e, 2^(e+1))); 2^-133 at 0."""
    e = torch.floor(torch.log2(x.abs().clamp_min(2.0 ** -126)))
    return torch.pow(2.0, e - 7)


def _head_case(rows, out_mode, eps, cap):
    _lib, L = _L()
    hh, HCh, lat = 128, 512, 128 + 2 * 512
    K = lat
    M = rows + 64                                          # device-side row count below M
    g = torch.Generator(device="cuda").manual_seed(rows * 13 + out_mode * 5 + cap + len(eps))
    z = _bf16(torch.randn(M, K, device="cuda", generator=g) * 0.5)
    x1 = _bf16(torch.randn(M, HCh, device="cuda", generator=g) * 0.5)
    z[:, hh:hh + HCh] = float("nan")                       # the kernel takes these columns from x1
    A = z.clone()
    A[:, hh:hh + HCh] = x1
    w_h0 = _bf16(torch.randn(2 * hh, K, device="cuda", generator=g) / K ** 0.5)
    w1 = torch.zeros(2 * hh, 2 * hh, device="cuda")
    w1[:hh, :hh] = torch.randn(hh, hh, device="cuda", generator=g) / hh ** 0.5
    w1[hh:, hh:] = torch.randn(hh, hh, device="cuda", generator=g) / hh ** 0.5
    w_h1 = _bf16(w1)
    b_h0, b_h1 = torch.randn(2 * hh, device="cuda", generator=g) * 0.1, torch.randn(2 * hh, device="cuda", generator=g) * 0.1
    q_w2, v_w2 = torch.randn(2, hh, device="cuda", generator=g) * 0.1, torch.randn(hh, device="cuda", generator=g) * 0.1
    hv1 = torch.cat([q_w2[0], v_w2]).contiguous()
    hv2 = torch.cat([q_w2[1], torch.zeros(hh, device="cuda")]).contiguous()
    # small output biases: the greedy margin then depends on the rows' hidden activations, not on bq[1] - bq[0]
    bq, bv = torch.randn(2, device="cuda", generator=g) * 0.01, torch.randn(1, device="cuda", generator=g) * 0.01
    m_dev = torch.tensor([rows], dtype=torch.int32, device="cuda")
    graphs = rows + 5
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
    seed, offset = 0x5EED0F7E57, 31
    rand3 = torch.rand(n_out, 3, device="cuda", dtype=torch.float64, generator=g) if eps == "rand3" else None
    q = torch.full((n_out, 2), float("nan"), device="cuda")
    act = torch.full((n_out,), 77, dtype=torch.int8, device="cuda")
    with _Cap(cap):
        _lib.check(L.mls_test_head_dueling(z.data_ptr(), K, x1.data_ptr(), HCh, hh, hh + HCh, M, K, m_dev.data_ptr(), w_h0.data_ptr(),
                                           b_h0.data_ptr(), w_h1.data_ptr(), b_h1.data_ptr(), hv1.data_ptr(), hv2.data_ptr(),
                                           bq.data_ptr(), bv.data_ptr(), _lib.ptr(idx), row0 if out_mode != 2 else 0, NODES,
                                           q.data_ptr(), act.data_ptr() if out_mode != 2 else None, out_mode, eps_v, seed, offset,
                                           _lib.ptr(rand3), _lib.current_stream_ptr()))
        torch.cuda.synchronize()

    # float64 reference; the hidden layer is rounded to bf16 where the kernel rounds it
    A64 = A[:rows].double()
    pre0 = A64 @ w_h0.double().T + b_h0.double()[None, :]
    acc0 = K * U23 * (A64.abs() @ w_h0.double().abs().T)
    hid = pre0.clamp_min(0).to(torch.bfloat16).double()
    # one bf16 ulp of the hidden value, or of the pre-activation value where the kernel's fp32 value may straddle 0
    e_h = torch.where(pre0 > -acc0, _ulp_bf16(pre0.abs() + acc0) + acc0, torch.zeros_like(pre0))
    W1 = w_h1.double()
    pre1 = hid @ W1.T + b_h1.double()[None, :]
    h2 = pre1.clamp_min(0)
    e_2 = e_h @ W1.abs().T + 2 * hh * U23 * (hid.abs() @ W1.abs().T) + U23 * pre1.abs()
    v1, v2 = hv1.double(), hv2.double()
    d = [(h2[:, :hh] * v1[:hh]).sum(1), (h2[:, hh:] * v1[hh:]).sum(1), (h2[:, :hh] * v2[:hh]).sum(1)]
    e_d = [(e_2[:, sl] * vv[sl].abs()).sum(1) + 130 * 2.0 ** -24 * (h2[:, sl] * vv[sl]).abs().sum(1)
           for sl, vv in ((slice(0, hh), v1), (slice(hh, 2 * hh), v1), (slice(0, hh), v2))]
    s0, sv, s1 = d[0] + float(bq[0]), d[1] + float(bv[0]), d[2] + float(bq[1])
    mean = (s0 + s1) / 2
    o = torch.stack([(s0 - mean) + sv, (s1 - mean) + sv], 1)
    e_o = 0.5 * e_d[0] + 0.5 * e_d[2] + e_d[1] + 8 * 2.0 ** -24 * (s0.abs() + s1.abs() + sv.abs())
    t = torch.arange(rows, device="cuda")
    orow = (row0 + idx[:rows].long() if out_mode == 0 else row0 // NODES + idx[:rows].long() // NODES if out_mode == 1 else t)
    worst = _Worst(f"fused head cap {cap} rows {rows} out_mode {out_mode} {eps}")
    worst.add("q", (q[orow].double() - o).abs(), e_o[:, None] + 1e-30)
    written = torch.zeros(n_out, dtype=torch.bool, device="cuda")
    written[orow] = True
    assert torch.isnan(q[~written]).all(), "Q written outside the device row count"
    if out_mode != 2:
        assert (act[~written] == 77).all(), "action written outside the device row count"
        o_np, orow_np = o.cpu(), orow.cpu().numpy()
        want = _actions(o_np, orow_np, eps_v, seed, offset, rand3)
        swapped = _actions(o_np.flip(1), orow_np, eps_v, seed, offset, rand3)
        margin = (o[:, 1] - o[:, 0]).abs().cpu().numpy()
        explored = (want == swapped) & (margin > 0)            # the draw decided: the same action whichever Q is larger
        sure = explored | (margin > 2 * e_o.cpu().numpy())
        got = act[orow].cpu().numpy()
        assert np.array_equal(got[sure], want[sure]), f"{int((got[sure] != want[sure]).sum())} actions differ"
        qk = q[orow].cpu().numpy()                             # and greedy decisions follow the kernel's own Q-values
        np.testing.assert_array_equal(got[~explored], (qk[:, 1] > qk[:, 0]).astype(np.int8)[~explored])
    else:
        assert (act == 77).all()
    worst.report()


@pytest.mark.parametrize("cap", CAPS)
@pytest.mark.parametrize("extra", [1, 127])
@pytest.mark.parametrize("out_mode", [0, 1, 2])
@pytest.mark.parametrize("eps", ["greedy", "rand3", "philox"])
def test_fused_head_many_tiles_per_cta_against_float64(cap, extra, out_mode, eps):
    _head_case(cap * 4 * 128 + extra, out_mode, eps, cap)


@pytest.mark.parametrize("eps", ["greedy", "philox"])
def test_fused_head_uncapped_two_tiles_per_sm(eps):
    _head_case(2 * _sms() * 128 + 300, 0, eps, 0)


@pytest.mark.parametrize("cap", [2, 3])
@pytest.mark.parametrize("out_mode", [0, 2])
def test_fused_head_bit_identity_with_gemm_chain_at_several_tiles_per_cta(cap, out_mode):
    """The existing fused-head vs MODE 2 -> MODE 3 bit identity (9001 rows), with a capped grid on both sides."""
    with _Cap(cap):
        _head_chain_bits(9001, out_mode, True, "philox")


# ---------------------------------------------------------------------------------------------- forward grid invariance
def _boundary_inputs(N, B, seed):
    """Observation matrices and controlling masks that reach conv2's and conv1's item boundaries: complete graphs with every
    node controlling (several blocks of 32 targets / 256 entries; nodes past index 32 keep 33 sources), graphs with exactly 32
    and 33 controlling nodes, runs of graphs without controlling nodes longer than the two-item metadata prefetch, and (N = 20:
    three graphs per conv1 tile) a partly filled last tile."""
    from test_networks_gpu import _obs_matrix
    om = _obs_matrix(N, B, seed)
    rng = np.random.default_rng(seed)
    cm = rng.random((B, N)) < 0.3
    om[0:3, :, :2] = 0.0                                   # complete graphs
    cm[0:3] = True
    om[B - 1, :, :2] = 0.0                                  # ... also the last graph
    cm[B - 1] = True
    for gi, n_ctrl in ((4, 32), (5, 33), (9, 32), (10, 33)):
        cm[gi] = False
        cm[gi, rng.permutation(N)[:min(n_ctrl, N)]] = True
    om[9:11, :, :2] = 0.0
    cm[12:17] = False                                       # five graphs in a row without controlling nodes
    cm[B - 6:B - 2] = False
    return om, cm


FWD_MODELS = [("l_dgn", {}), ("dgn_r", {}), ("hl_dgn", {"aggregator": "max"}), ("hl_dgn", {"aggregator": "mean"})]


@pytest.mark.parametrize("kind,kw", FWD_MODELS, ids=["l_dgn", "dgn_r", "hl_dgn_max", "hl_dgn_mean"])
# conv1 tiles of 1 graph (N = 62, 60: no room for the bias rows in the weight matrix), 3 graphs (N = 20), 5 graphs (N = 12);
# N = 50 is the benchmark size (tables only up to 62 nodes, conv2 tensor cores up to 64)
@pytest.mark.parametrize("N,B", [(62, 67), (64, 45), (20, 301), (50, 203), (12, 410), (60, 77)])
def test_forward_is_bit_identical_at_every_grid(kind, kw, N, B):
    from test_networks_gpu import BF16_TOL, _module, _random_sd
    from oracle import net_oracle as no
    H = 4
    sd = _random_sd(kind, 91)
    om, cm = _boundary_inputs(N, B, 7 + N)
    m = _module(kind, N, sd, **kw).set_precision("bf16")
    args = (torch.as_tensor(om, device="cuda"), torch.as_tensor(cm, device="cuda").to(torch.uint8))
    want = no.forward_graphs(kind, sd, torch.as_tensor(om), torch.as_tensor(cm), N, **kw).numpy()
    scale = max(1.0, float(np.abs(want).max()))
    # discrete-feature tables (conv1 through attn_table: the record kernel, or the pooling kernel of HL-DGN) take N <= 62
    tables = [False, True] if N <= 62 else [False]
    for tab in tables:
        with _Cap(0):
            q0, a0 = m.forward_graphs(*args, discrete_features=tab, eps=0.25, philox_seed=5, philox_offset=3)
        for cap in (H, 2 * H, 3 * H, 7 * H):
            with _Cap(cap):
                q, a = m.forward_graphs(*args, discrete_features=tab, eps=0.25, philox_seed=5, philox_offset=3)
            assert torch.equal(q.view(torch.int32), q0.view(torch.int32)), f"Q differs at cap {cap} (tables {tab})"
            assert torch.equal(a, a0), f"actions differ at cap {cap} (tables {tab})"
        with _Cap(H):                                       # one capped run per configuration against the fp32 oracle
            qc, ac = m.forward_graphs(*args, discrete_features=tab)
        err = float(np.abs(qc.cpu().numpy() - want).max())
        assert err <= BF16_TOL * scale, (tab, err, scale)
        assert torch.equal(ac >= 0, args[1].bool())


@pytest.mark.parametrize("kind,kw", FWD_MODELS[:3], ids=["l_dgn", "dgn_r", "hl_dgn_max"])
@pytest.mark.parametrize("N", [34, 50, 62, 64])
def test_bf16_forward_on_complete_graphs_with_every_node_controlling(kind, kw, N):
    """Regression: radius_graph keeps 33 sources for a node past index 32 of a complete graph (its own hit is not among the
    first 33), and the bf16 path's CSR lists, conv2 entry lists and conv1 records were sized for 32 sources per node plus
    the self loop.  The lists of one graph ran into the next graph's and past the end of the workspace; the conv1 edge
    kernel staged only 32 bytes per node and read the rest from the row pointers behind them.  Every node of every graph
    controlling, at the default grid, through the per-node, table and topology-cache paths, against the fp32 oracle."""
    from test_networks_gpu import BF16_TOL, _module, _obs_matrix, _random_sd
    from oracle import net_oracle as no
    B = 7
    sd = _random_sd(kind, 17)
    om = _obs_matrix(N, B, 3)
    om[:, :, :2] = 0.0                                      # every pair of nodes within r
    om[B - 1, :, 0] = np.arange(N) * (0.15 / N)             # ... also on a short segment
    cm = np.ones((B, N), dtype=bool)
    want = no.forward_graphs(kind, sd, torch.as_tensor(om), torch.as_tensor(cm), N, **kw).numpy()
    scale = max(1.0, float(np.abs(want).max()))
    m = _module(kind, N, sd, **kw).set_precision("bf16")
    args = (torch.as_tensor(om, device="cuda"), torch.as_tensor(cm, device="cuda").to(torch.uint8))
    outs = [m.forward_graphs(*args)[0]]
    if N <= 62:
        outs.append(m.forward_graphs(*args, discrete_features=True)[0])
        cache = m.build_topology_cache(om[:, :, :2].copy())
        gid = torch.arange(B, dtype=torch.int32, device="cuda")
        outs.append(m.forward_graphs(*args, discrete_features=True, graph_ids=gid, graph_id_stride=1, topology_cache=cache)[0])
    for i, q in enumerate(outs):
        err = float(np.abs(q.cpu().numpy() - want).max())
        assert err <= BF16_TOL * scale, (i, err, scale)


# ---------------------------------------------------------------------------------------------- fp32 tensor-core route
@pytest.mark.parametrize("cap", [1, 2])
@pytest.mark.parametrize("kind,kw", [("l_dgn", {}), ("dgn_r", {}), ("hl_dgn", {"aggregator": "mean"})], ids=["l_dgn", "dgn_r", "hl_dgn"])
def test_fp32_tensor_core_route_meets_the_fp32_bar_at_a_capped_grid(kind, kw, cap):
    from test_networks_gpu import _assert_q, _module, _obs_matrix, _random_sd
    from oracle import net_oracle as no
    from melissa_b200 import _lib
    N, B = 50, 60
    sd = _random_sd(kind, 33)
    sd["conv1.lin_l.weight" if kind != "dgn_r" else "conv1.lin_key.weight"] *= 8.0
    om = _obs_matrix(N, B, 41)
    cm = np.random.default_rng(6).random((B, N)) < 0.3
    want = no.forward_graphs(kind, sd, torch.as_tensor(om), torch.as_tensor(cm), N, **kw).numpy()
    m = _module(kind, N, sd, **kw)
    assert _lib.get_option("fp32_tc") == 1
    with _Cap(cap):
        q, a = m.forward_graphs(torch.as_tensor(om, device="cuda"), torch.as_tensor(cm, device="cuda").to(torch.uint8))
    _assert_q(q.cpu().numpy(), want, f"{kind} fp32 tensor-core route, cap {cap}")
    margin = np.abs(want[..., 1] - want[..., 0])
    sure = cm & (margin > 1e-4)
    np.testing.assert_array_equal(a.cpu().numpy()[sure], (want[..., 1] > want[..., 0]).astype(np.int8)[sure])


def test_max_ctas_option_round_trips():
    from melissa_b200 import _lib
    assert _lib.get_option("max_ctas") == 0                 # off unless a test sets it
    with _Cap(7):
        assert _lib.get_option("max_ctas") == 7
        with _Cap(-3):
            assert _lib.get_option("max_ctas") == 0
    assert _lib.get_option("max_ctas") == 0
