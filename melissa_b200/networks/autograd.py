"""Differentiable forward of the three Q-networks for the TRAINING step (loss + backward through torch autograd).

The rollout forward is hand-written CUDA (``mls_dgn_forward``) and has no backward; a gradient step needs one.  This
module evaluates the same math with torch ops over the module's own parameters, so ``loss.backward()`` fills their
``.grad`` (SURVEY.md section 8f-2: "v1 can use autograd").  Reference math: ``networks/{l_dgn.py:92-151,
dgn_r.py:82-129, hl_dgn.py:82-119}``, ``networks/common.py:6-64`` and the PyG / tianshou ops they call (SURVEY.md
Appendix B).  It is a product module -- it never imports ``oracle`` -- and follows the structure of the CUDA path
rather than PyG's: one agent observation controls ONE node, so only the rows that node reads are evaluated

    conv2 at the controlling node c          <- sources  S1 = {c} + radius-neighbours(c)
    conv1 at the nodes of S1 (x1 rows)       <- sources  S2 = S1 + their radius-neighbours

as edge lists over (sample, target, source) triples with scatter softmax; the dense layers are plain ``F.linear``, or with
``net.set_train_precision("bf16")`` the bf16 tensor-core Function ``_LinearBF16``.
Runs wherever the parameters live (the training loop keeps them on the GPU; bf16 training precision needs CUDA tensors).
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn
import torch.nn.functional as F

R2 = float(torch.tensor(0.2, dtype=torch.float64).pow(2).to(torch.float32))     # torch_cluster: r*r narrowed to fp32
MAX_NUM_NEIGHBORS = 32


def split_rows(obs: torch.Tensor, n_agents: int, input_dim: int = 5):
    """networks/common.py:20-44,63: agent rows [bs, N*(F+3)+1] -> pos, feats, dm, ctrl."""
    if obs.ndim != 2:
        raise ValueError(f"Expected obs to be 2D, but got shape {obs.shape}")
    bs, dim = obs.shape
    d = input_dim + 3
    if dim - 1 != n_agents * d:
        raise ValueError(f"Expected {n_agents * d} feature cols for nodes, got {dim - 1}")
    node = obs[:, : dim - 1].reshape(bs, n_agents, d).float()
    return node[..., :2], node[..., 2:-1], node[..., -1:], obs[:, -1].clamp(0, n_agents - 1).long()


def radius_mask(pos: torch.Tensor) -> torch.Tensor:
    """radius_graph(pos, r=0.2, loop=False, max_num_neighbors=32) as bool [bs, target i, source j]: candidates in
    index order, kept while fma(dy, dy, dx*dx) < r^2 in fp32, the scan stops after 33 hits (self included)."""
    p = pos.to(torch.float32)
    dx = p[:, None, :, 0] - p[:, :, None, 0]
    dy = p[:, None, :, 1] - p[:, :, None, 1]
    d2 = (dy.double() * dy.double() + (dx * dx).double()).float()
    hit = d2 < R2
    hit = hit & (hit.to(torch.int16).cumsum(dim=2, dtype=torch.int16) <= MAX_NUM_NEIGHBORS + 1)
    n = p.shape[1]
    return hit & ~torch.eye(n, dtype=torch.bool, device=p.device)


def _segment_softmax(e: torch.Tensor, seg: torch.Tensor, n_seg: int) -> torch.Tensor:
    """PyG utils.softmax: exp(e - max_seg) / (sum_seg + 1e-16); e [E, H], seg [E] segment id per edge."""
    H = e.shape[1]
    idx = seg[:, None].expand(-1, H)
    mx = torch.full((n_seg, H), -torch.inf, dtype=e.dtype, device=e.device).scatter_reduce(0, idx, e.detach(), "amax", include_self=True)
    ex = (e - mx[seg]).exp()
    den = torch.zeros(n_seg, H, dtype=e.dtype, device=e.device).index_add_(0, seg, ex)
    return ex / (den[seg] + 1e-16)


def _edges(mask: torch.Tensor, targets: torch.Tensor, self_loops: bool):
    """Edge list (sample m, target i, source j) of ``mask`` [bs, i, j] restricted to target rows where ``targets``
    [bs, N] is set (+ a self loop per such target)."""
    m = mask & targets[:, :, None]
    if self_loops:
        m = m | (torch.eye(mask.shape[1], dtype=torch.bool, device=mask.device)[None] & targets[:, :, None])
    return torch.nonzero(m, as_tuple=True)


def _used_rows(n_rows, *index_lists):
    """Rows that appear in an edge list, and the map row -> position among them: the dense projections are evaluated
    on those rows only (most of a graph's nodes are neither a source nor a target of what one agent reads)."""
    used = torch.zeros(n_rows, dtype=torch.bool, device=index_lists[0].device)
    for ix in index_lists:
        used[ix] = True
    rows = torch.nonzero(used, as_tuple=True)[0]
    remap = torch.full((n_rows,), -1, dtype=torch.long, device=rows.device)
    remap[rows] = torch.arange(rows.numel(), device=rows.device)
    return rows, remap


def _gatv2(conv, x, edges, heads, N, lin):
    """PyG GATv2Conv(concat=True, negative_slope=0.2, add_self_loops=True, share_weights=False) on an edge list.
    x [bs, N, D]; returns [bs*N, H*C] with rows of non-target nodes = bias only (never read)."""
    sm, ti, sj = edges
    bs = x.shape[0]
    C = conv.att.shape[-1]
    tgt, src = sm * N + ti, sm * N + sj
    xf = x.reshape(bs * N, -1)
    rows_s, map_s = _used_rows(bs * N, src)
    rows_t, map_t = _used_rows(bs * N, tgt)
    xl = lin(conv.lin_l, xf[rows_s]).view(-1, heads, C)[map_s[src]]          # [E, H, C] source side
    xr = lin(conv.lin_r, xf[rows_t]).view(-1, heads, C)[map_t[tgt]]          # [E, H, C] target side
    s = F.leaky_relu(xl + xr, 0.2)
    e = (s * conv.att.view(1, heads, C)).sum(-1)
    a = _segment_softmax(e, tgt, bs * N)
    out = torch.zeros(bs * N, heads, C, dtype=x.dtype, device=x.device).index_add_(0, tgt, a[:, :, None] * xl)
    return out.view(bs * N, heads * C) + conv.bias


def _transformer(conv, x, edges, heads, N, lin):
    """PyG TransformerConv(root_weight=False, beta=False): no self loops, no output bias, ``lin_skip`` unused."""
    sm, ti, sj = edges
    bs = x.shape[0]
    HC = conv.lin_query.out_features
    C = HC // heads
    tgt, src = sm * N + ti, sm * N + sj
    xf = x.reshape(bs * N, -1)
    rows_s, map_s = _used_rows(bs * N, src)
    rows_t, map_t = _used_rows(bs * N, tgt)
    q = lin(conv.lin_query, xf[rows_t]).view(-1, heads, C)[map_t[tgt]]
    k = lin(conv.lin_key, xf[rows_s]).view(-1, heads, C)[map_s[src]]
    v = lin(conv.lin_value, xf[rows_s]).view(-1, heads, C)[map_s[src]]
    e = (q * k).sum(-1) / math.sqrt(C)
    a = _segment_softmax(e, tgt, bs * N)
    out = torch.zeros(bs * N, heads, C, dtype=x.dtype, device=x.device).index_add_(0, tgt, a[:, :, None] * v)
    return out.view(bs * N, HC)


def _mlp(params, x, lin):
    for m in params.model:
        x = lin(m, x) if isinstance(m, nn.Linear) else m(x)
    return x


def _dueling(net, z, lin):
    if not net.use_dueling:
        return lin(net.out_linear, z)
    q = _mlp(net.Q, z, lin)
    v = _mlp(net.V, z, lin)
    return q - q.mean(dim=1, keepdim=True) + v


def _require_f32_cuda(what, *tensors):
    """The CUDA training Functions read their operands as fp32 device memory: refuse anything else before any launch
    (under torch.autocast the dense layers would hand them bf16 tensors of half the expected size)."""
    for t in tensors:
        if t.dtype != torch.float32 or not t.is_cuda:
            from .. import _lib
            raise _lib.MelissaLibraryError(
                f"{what} takes float32 CUDA tensors, got {t.dtype} on {t.device}; there is no CPU path, and mixed-precision "
                'training is net.set_train_precision("bf16") (bf16 tensor-core GEMMs, fp32 weights), not torch.autocast')


class _LinearBF16(torch.autograd.Function):
    """nn.Linear in bf16 training precision (``mls_linear_bf16_fwd`` / ``_bwd``, ``csrc/train_linear.cu``): bf16 operands,
    fp32 accumulation on the tcgen05 GEMM, fp32 in and out.  y = bf16(x) bf16(W)^T + b, dx = bf16(dy) bf16(W),
    dW = bf16(dy)^T bf16(x), db = sum of the unrounded dy over rows; dx only when autograd asks for it."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        _require_f32_cuda("the bf16 linear layer", x, weight, *(() if bias is None else (bias,)))
        from .. import _lib
        L = _lib.lib()
        out_f, in_f = weight.shape
        x2 = x.reshape(-1, in_f)
        if x2.stride(1) != 1 or x2.stride(0) < in_f:
            x2 = x2.contiguous()
        w = weight.contiguous()
        rows = x2.shape[0]
        y = torch.empty(rows, out_f, dtype=torch.float32, device=x.device)
        if rows:
            ws = torch.empty(L.mls_linear_bf16_workspace_bytes(rows, in_f, out_f), dtype=torch.uint8, device=x.device)
            _lib.check(L.mls_linear_bf16_fwd(x2.data_ptr(), x2.stride(0), w.data_ptr(), None if bias is None else bias.data_ptr(),
                                             rows, in_f, out_f, y.data_ptr(), out_f, ws.data_ptr(), ws.numel(),
                                             _lib.current_stream_ptr()))
        ctx.save_for_backward(x2, w)
        ctx.has_bias, ctx.x_shape = bias is not None, x.shape
        return y.view(*x.shape[:-1], out_f)

    @staticmethod
    def backward(ctx, dy):
        from .. import _lib
        L = _lib.lib()
        x2, w = ctx.saved_tensors
        out_f, in_f = w.shape
        rows = x2.shape[0]
        dy2 = dy.reshape(-1, out_f)
        if dy2.stride(1) != 1 or dy2.stride(0) < out_f:
            dy2 = dy2.contiguous()
        need_dx, _, need_db = ctx.needs_input_grad
        dev = x2.device
        dx = torch.empty(rows, in_f, dtype=torch.float32, device=dev) if need_dx else None
        dw = torch.empty(out_f, in_f, dtype=torch.float32, device=dev)
        db = torch.empty(out_f, dtype=torch.float32, device=dev) if (ctx.has_bias and need_db) else None
        ws = torch.empty(max(1, L.mls_linear_bf16_workspace_bytes(rows, in_f, out_f)), dtype=torch.uint8, device=dev)
        _lib.check(L.mls_linear_bf16_bwd(x2.data_ptr(), x2.stride(0), w.data_ptr(), dy2.data_ptr(), dy2.stride(0), rows, in_f, out_f,
                                         None if dx is None else dx.data_ptr(), in_f, dw.data_ptr(),
                                         None if db is None else db.data_ptr(), ws.data_ptr(), ws.numel(), _lib.current_stream_ptr()))
        return None if dx is None else dx.view(ctx.x_shape), dw, db


def _linear_op(net):
    """How ``net``'s dense layers are evaluated in training: ``layer(x)`` (fp32) or through ``_LinearBF16``."""
    if net.train_precision == "bf16":
        return lambda layer, x: _LinearBF16.apply(x, layer.weight, layer.bias)
    return lambda layer, x: layer(x)


class _GATv2Edge(torch.autograd.Function):
    """Edge phase of GATv2Conv on fixed-capacity edge lists, forward and backward as CUDA kernels
    (``csrc/train_gatv2.cu``): out[t] = sum_e softmax_e(<att, leaky_relu(xl[src[t, e]] + xr[tgt[t]])>) xl[src[t, e]]."""

    @staticmethod
    def forward(ctx, xl, xr, att, tgt_row, src_row, src_cnt):
        _require_f32_cuda("the GATv2 edge phase", xl, xr, att)
        from .. import _lib
        L = _lib.lib()
        xl, xr, att = xl.contiguous(), xr.contiguous(), att.contiguous()
        T, heads = tgt_row.numel(), att.numel() // 128
        out = torch.empty(T, heads * 128, dtype=torch.float32, device=xl.device)
        alpha = torch.empty(T, src_row.shape[1], heads, dtype=torch.float32, device=xl.device)
        _lib.check(L.mls_gatv2_edge_fwd(xl.data_ptr(), xl.shape[1], xr.data_ptr(), xr.shape[1], att.data_ptr(), tgt_row.data_ptr(),
                                        src_row.data_ptr(), src_cnt.data_ptr(), T, heads, out.data_ptr(), alpha.data_ptr(),
                                        _lib.current_stream_ptr()))
        ctx.save_for_backward(xl, xr, att, tgt_row, src_row, src_cnt, alpha)
        return out

    @staticmethod
    def backward(ctx, dout):
        from .. import _lib
        L = _lib.lib()
        xl, xr, att, tgt_row, src_row, src_cnt, alpha = ctx.saved_tensors
        T, heads = tgt_row.numel(), att.numel() // 128
        dout = dout.contiguous()
        d_xl, d_xr = torch.zeros_like(xl), torch.zeros_like(xr)
        part = torch.empty(L.mls_gatv2_edge_bwd_blocks(T), heads * 128, dtype=torch.float32, device=xl.device)
        _lib.check(L.mls_gatv2_edge_bwd(xl.data_ptr(), xl.shape[1], xr.data_ptr(), xr.shape[1], att.data_ptr(), tgt_row.data_ptr(),
                                        src_row.data_ptr(), src_cnt.data_ptr(), T, heads, alpha.data_ptr(), dout.data_ptr(),
                                        d_xl.data_ptr(), d_xr.data_ptr(), part.data_ptr(), _lib.current_stream_ptr()))
        return d_xl, d_xr, part.sum(dim=0).view_as(att), None, None, None


class _TransformerEdge(torch.autograd.Function):
    """Edge phase of TransformerConv(root_weight=False) on the same edge lists (their first entry, the node itself, is
    skipped: no self loops): out[t] = sum_e softmax_e(<q[tgt[t]], k[src]> / sqrt(C)) v[src]."""

    @staticmethod
    def forward(ctx, q, k, v, tgt_row, src_row, src_cnt):
        _require_f32_cuda("the TransformerConv edge phase", q, k, v)
        from .. import _lib
        L = _lib.lib()
        q, k, v = q.contiguous(), k.contiguous(), v.contiguous()
        T, heads = tgt_row.numel(), q.shape[1] // 128
        out = torch.empty(T, heads * 128, dtype=torch.float32, device=q.device)
        alpha = torch.empty(T, src_row.shape[1], heads, dtype=torch.float32, device=q.device)
        _lib.check(L.mls_transformer_edge_fwd(k.data_ptr(), v.data_ptr(), k.shape[1], q.data_ptr(), q.shape[1], tgt_row.data_ptr(),
                                              src_row.data_ptr(), src_cnt.data_ptr(), T, heads, out.data_ptr(), alpha.data_ptr(),
                                              _lib.current_stream_ptr()))
        ctx.save_for_backward(q, k, v, tgt_row, src_row, src_cnt, alpha)
        return out

    @staticmethod
    def backward(ctx, dout):
        from .. import _lib
        L = _lib.lib()
        q, k, v, tgt_row, src_row, src_cnt, alpha = ctx.saved_tensors
        T, heads = tgt_row.numel(), q.shape[1] // 128
        dout = dout.contiguous()
        d_q, d_k, d_v = torch.zeros_like(q), torch.zeros_like(k), torch.zeros_like(v)
        _lib.check(L.mls_transformer_edge_bwd(k.data_ptr(), v.data_ptr(), k.shape[1], q.data_ptr(), q.shape[1], tgt_row.data_ptr(),
                                              src_row.data_ptr(), src_cnt.data_ptr(), T, heads, alpha.data_ptr(), dout.data_ptr(),
                                              d_k.data_ptr(), d_v.data_ptr(), d_q.data_ptr(), _lib.current_stream_ptr()))
        return d_q, d_k, d_v, None, None, None


def train_lists(obs_rows: torch.Tensor, n_agents: int):
    """Per-sample edge lists on the device (``mls_train_lists``): slot_base [bs], s1_cnt [bs], and for the R slots (the nodes
    the controlling nodes read, sample after sample, controlling node first) tgt_row [R], src_row [R, cap], src_cnt [R];
    rows are sample * N + node; used [bs * N] marks the node rows that are a source of some slot.  One host
    synchronisation (R)."""
    from .. import _lib
    L = _lib.lib()
    obs_rows = obs_rows.contiguous().float()
    bs, dev = obs_rows.shape[0], obs_rows.device
    cap, st = L.mls_train_list_capacity(), _lib.current_stream_ptr()
    s1_cnt = torch.empty(bs, dtype=torch.int32, device=dev)
    _lib.check(L.mls_train_lists(obs_rows.data_ptr(), obs_rows.shape[1], bs, n_agents, R2, 0, s1_cnt.data_ptr(), None, None, None, None, None, st))
    incl = torch.cumsum(s1_cnt, dim=0, dtype=torch.int64)
    slot_base = (incl - s1_cnt).contiguous()
    R = int(incl[-1].item()) if bs else 0
    tgt_row = torch.empty(R, dtype=torch.int32, device=dev)
    src_row = torch.zeros(R, cap, dtype=torch.int32, device=dev)
    src_cnt = torch.empty(R, dtype=torch.int32, device=dev)
    used = torch.zeros(bs * n_agents, dtype=torch.uint8, device=dev)
    _lib.check(L.mls_train_lists(obs_rows.data_ptr(), obs_rows.shape[1], bs, n_agents, R2, 1, None, slot_base.data_ptr(),
                                 tgt_row.data_ptr(), src_row.data_ptr(), src_cnt.data_ptr(), used.data_ptr(), st))
    return slot_base, s1_cnt, tgt_row, src_row, src_cnt, used


def q_values_l_dgn_fused(net, obs_rows: torch.Tensor) -> torch.Tensor:
    """L-DGN / DGN-R Q-values with the two attention edge phases (and their backward) on the CUDA kernels of
    ``csrc/train_gatv2.cu``; same math as ``q_values_torch`` (``l_dgn.py:92-151``, ``dgn_r.py:82-129``), dense layers through
    ``F.linear`` or ``_LinearBF16`` (training precision).  CUDA tensors only."""
    N, heads = net.agents_num, net.num_heads
    tr = net.KIND == "dgn_r"
    lin = _linear_op(net)

    def conv(c, x_src, x_tgt, tgt, src, cnt):
        if tr:
            return _TransformerEdge.apply(lin(c.lin_query, x_tgt), lin(c.lin_key, x_src), lin(c.lin_value, x_src), tgt, src, cnt)
        return _GATv2Edge.apply(lin(c.lin_l, x_src), lin(c.lin_r, x_tgt), c.att.view(-1), tgt, src, cnt) + c.bias

    pos, feats, dm, ctrl = split_rows(obs_rows, N, net.input_dim)
    bs, dev = obs_rows.shape[0], obs_rows.device
    slot_base, s1_cnt, tgt_row, src_row, src_cnt, used = train_lists(obs_rows, N)
    cap = src_row.shape[1]
    # encoder and conv1 source projection only on the node rows somebody reads (a third of them at N = 50)
    rows_u = torch.nonzero(used, as_tuple=True)[0]
    remap = torch.zeros(bs * N, dtype=torch.int32, device=dev)
    remap[rows_u] = torch.arange(rows_u.numel(), dtype=torch.int32, device=dev)
    x0 = F.relu(_mlp(net.encoder, feats.reshape(bs * N, -1)[rows_u], lin))     # [used rows, hid]
    tgt_l = tgt_row.long()
    tgt_u = remap[tgt_l].long()                                                 # a slot's node is its own first source
    # conv1 at the S1 slots: sources are (used) node rows, targets the slots' own nodes
    ar_r = torch.arange(tgt_row.numel(), dtype=torch.int32, device=dev)
    x1 = F.relu(conv(net.conv1, x0, x0[tgt_u], ar_r, remap[src_row.long()], src_cnt))                           # [R, HC]
    ctrl_slot = slot_base                                                       # slot 0 of a sample = its controlling node
    snap1 = x0[tgt_u[ctrl_slot]]
    snap2 = x1[ctrl_slot]                                                       # before the dm mask
    x1m = x1 * dm.reshape(bs * N, 1)[tgt_l]
    # conv2 at the controlling node: sources are the sample's slots (controlling node = self loop first)
    src2 = (slot_base[:, None] + torch.arange(cap, device=dev)[None, :]).to(torch.int32)
    src2 = torch.where(torch.arange(cap, device=dev)[None, :] < s1_cnt[:, None], src2, torch.zeros_like(src2)).contiguous()
    ar_b = torch.arange(bs, dtype=torch.int32, device=dev)
    x2 = F.relu(conv(net.conv2, x1m, x1m[ctrl_slot], ar_b, src2, s1_cnt))                                      # [bs, HC]
    return _dueling(net, torch.cat([snap1, snap2, x2], dim=1), lin)


def q_values_hl_dgn_fused(net, obs_rows: torch.Tensor) -> torch.Tensor:
    """HL-DGN Q-values (``hl_dgn.py:82-119``): one GATv2 layer at every node, masked, pooled over the graph; the edge
    phase and its backward on the CUDA kernels."""
    from .. import _lib
    L = _lib.lib()
    N = net.agents_num
    lin = _linear_op(net)
    pos, feats, dm, ctrl = split_rows(obs_rows, N, net.input_dim)
    obs_c = obs_rows.contiguous().float()
    bs, dev = obs_rows.shape[0], obs_rows.device
    cap = L.mls_train_list_capacity()
    tgt_row = torch.empty(bs * N, dtype=torch.int32, device=dev)
    src_row = torch.zeros(bs * N, cap, dtype=torch.int32, device=dev)
    src_cnt = torch.empty(bs * N, dtype=torch.int32, device=dev)
    _lib.check(L.mls_train_lists(obs_c.data_ptr(), obs_c.shape[1], bs, N, R2, 2, None, None, tgt_row.data_ptr(), src_row.data_ptr(),
                                 src_cnt.data_ptr(), None, _lib.current_stream_ptr()))
    x0 = F.relu(_mlp(net.encoder, feats.reshape(bs * N, -1), lin))
    out = _GATv2Edge.apply(lin(net.conv1.lin_l, x0), lin(net.conv1.lin_r, x0), net.conv1.att.view(-1), tgt_row, src_row, src_cnt)
    x1 = F.relu(out + net.conv1.bias).view(bs, N, -1) * dm
    agg = net.aggregator_name
    z = x1.amax(dim=1) if agg == "max" else (x1.mean(dim=1) if agg == "mean" else x1.sum(dim=1))
    return _dueling(net, z, lin)


def fused_training_available(net, obs_rows) -> bool:
    import os
    return (net.KIND in ("l_dgn", "hl_dgn", "dgn_r") and obs_rows.is_cuda and net.hidden_dim == 128 and net.num_heads <= 4
            and os.environ.get("MLS_TRAIN_FUSED", "1") != "0")


def q_values(net, obs_rows: torch.Tensor) -> torch.Tensor:
    """Q-values [bs, 2] of agent-observation rows [bs, 8N+1] (last column = controlling index), differentiable
    with respect to ``net``'s parameters."""
    if fused_training_available(net, obs_rows):
        return q_values_hl_dgn_fused(net, obs_rows) if net.KIND == "hl_dgn" else q_values_l_dgn_fused(net, obs_rows)
    return q_values_torch(net, obs_rows)


def q_values_torch(net, obs_rows: torch.Tensor) -> torch.Tensor:
    """The same through plain torch ops only (any device; every network kind)."""
    N, heads = net.agents_num, net.num_heads
    pos, feats, dm, ctrl = split_rows(obs_rows, N, net.input_dim)
    bs = obs_rows.shape[0]
    lin = _linear_op(net)
    mask = radius_mask(pos)
    ar = torch.arange(bs, device=obs_rows.device)
    x0 = F.relu(_mlp(net.encoder, feats, lin))                                  # [bs, N, hid]
    kind = net.KIND
    if kind == "hl_dgn":
        every = torch.ones(bs, N, dtype=torch.bool, device=obs_rows.device)
        x1 = F.relu(_gatv2(net.conv1, x0, _edges(mask, every, True), heads, N, lin)).view(bs, N, -1) * dm
        agg = net.aggregator_name
        z = x1.amax(dim=1) if agg == "max" else (x1.mean(dim=1) if agg == "mean" else x1.sum(dim=1))
        return _dueling(net, z, lin)
    tr = kind == "dgn_r"
    conv = _transformer if tr else _gatv2
    is_ctrl = torch.zeros(bs, N, dtype=torch.bool, device=obs_rows.device)
    is_ctrl[ar, ctrl] = True
    s1 = is_ctrl | mask[ar, ctrl]                                               # conv2 sources = conv1 targets
    x1 = F.relu(conv(net.conv1, x0, _edges(mask, s1, not tr), heads, N, lin)).view(bs, N, -1)
    snap1, snap2 = x0[ar, ctrl], x1[ar, ctrl]                                   # x1 snapshot is taken BEFORE the dm mask
    x1 = x1 * dm
    x2 = F.relu(conv(net.conv2, x1, _edges(mask, is_ctrl, not tr), heads, N, lin)).view(bs, N, -1)
    z = torch.cat([snap1, snap2, x2[ar, ctrl]], dim=1)
    return _dueling(net, z, lin)
