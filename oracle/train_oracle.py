"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the training-side arithmetic the reference delegates to tianshou.

PARITY UNPINNED at the tianshou boundary: tianshou 1.0.0 (requirements.txt:5) is not installable in this image and the
reference has no test or golden vector for its training step, so these functions restate the PUBLISHED algorithm of

* ``tianshou.policy.base._nstep_return`` / ``BasePolicy.compute_nstep_return`` (called by ``DQNPolicy.process_fn``
  with ``discount_factor`` and ``estimation_step``, reference l_dgn.py:69-76):
      indices = [idx, next(idx), ...] (n_step entries; next(i) = i on an episode end),
      terminal = indices[-1]; target_q = target_q_fn(terminal) * ~terminated[terminal];
      backward recursion  returns = rew[now] + gamma * returns, reset to 0 / gammas = n+1 where end_flag[now];
      result = target_q * gamma ** gammas + returns
* ``torch.optim.Adam`` (single tensor, amsgrad = False), reference l_dgn.py:66 -- this part IS pinned: torch is installed,
  tests/test_training_host.py::test_adam_restatement_is_pinned_on_torch_optim_adam runs the real optimiser beside it
* ``tianshou DQNPolicy.learn`` loss  mean((returns - Q(obs)[act])^2)  and ``DGNPolicy.learn`` (policies/dgn.py:22-71).
* the edge phases of the training kernels (csrc/train_gatv2.cu) on their fixed-capacity lists, in float64 torch with
  autograd for the backward; pinned on net_oracle's dense GATv2Conv / TransformerConv by tests/test_training_host.py.

Not product code: melissa_b200 never imports this module.
"""
from __future__ import annotations

import math

import numpy as np
import torch


def nstep_return_chain(rew: np.ndarray, terminated: np.ndarray, start: int, n_step: int, gamma: float, target_q_fn):
    """One agent's transition chain (its tianshou sub-buffer, in order): rew[t], terminated[t] (== done here: the
    environment only ever sets ``terminations``, graph.py:330-334).  Returns the n-step return of transition
    ``start`` exactly as tianshou computes it; ``target_q_fn(t)`` values the observation AFTER transition t."""
    L = len(rew)
    nxt = lambda i: i if (terminated[i] or i + 1 >= L) else i + 1
    indices = [start]
    for _ in range(n_step - 1):
        indices.append(nxt(indices[-1]))
    terminal = indices[-1]
    end_flag = terminated.copy()
    end_flag[L - 1] = True                                   # unfinished_index(): the last stored transition
    tq = 0.0 if terminated[terminal] else float(target_q_fn(terminal))
    gammas, returns = n_step, 0.0
    for n in range(n_step - 1, -1, -1):
        now = indices[n]
        if end_flag[now]:
            gammas, returns = n + 1, 0.0
        returns = float(rew[now]) + gamma * returns
    return tq * gamma ** gammas + returns


def adam_reference(p, grads, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0, state=None):
    """torch.optim.Adam over a list of gradient arrays applied in order; float64 numpy.  Without ``state`` it starts
    fresh and returns p.  With ``state = (m, v, steps_done)`` it continues from that optimiser state (the first gradient
    is step steps_done + 1) and returns (p, m, v)."""
    p = np.array(p, dtype=np.float64)
    if state is None:
        m, v, t0 = np.zeros_like(p), np.zeros_like(p), 0
    else:
        m, v, t0 = np.array(state[0], dtype=np.float64), np.array(state[1], dtype=np.float64), int(state[2])
    for t, g in enumerate(grads, start=t0 + 1):
        g = np.asarray(g, dtype=np.float64) + weight_decay * p
        m = betas[0] * m + (1 - betas[0]) * g
        v = betas[1] * v + (1 - betas[1]) * g * g
        bc1, bc2 = 1 - betas[0] ** t, 1 - betas[1] ** t
        p = p - (lr / bc1) * m / (np.sqrt(v) / np.sqrt(bc2) + eps)
    return p if state is None else (p, m, v)


def _edge_list(tgt_row, src_row, src_cnt, first):
    """(target index t, list entry e) of every edge of fixed-capacity lists: entries first .. src_cnt[t]-1 of targets
    with tgt_row[t] >= 0."""
    e = torch.arange(src_row.shape[1], device=src_row.device)
    keep = (e[None, :] >= first) & (e[None, :] < src_cnt.long()[:, None]) & (tgt_row >= 0)[:, None]
    return torch.nonzero(keep, as_tuple=True)


def _segment_softmax(logit, t, T):
    """PyG utils.softmax per target: exp(e - max) / (sum + 1e-16), max detached; logit [E, H], t [E] target index."""
    H = logit.shape[1]
    idx = t[:, None].expand(-1, H)
    mx = torch.full((T, H), -torch.inf, dtype=logit.dtype, device=logit.device).scatter_reduce(0, idx, logit.detach(), "amax")
    ex = (logit - mx[t]).exp()
    den = torch.zeros(T, H, dtype=logit.dtype, device=logit.device).index_add(0, t, ex)
    return ex / (den[t] + 1e-16)


def gatv2_edge_reference(xl, xr, att, tgt_row, src_row, src_cnt, heads):
    """Edge phase of GATv2Conv on the lists of ``mls_gatv2_edge_fwd``: out[t] = sum_e alpha[t, e] xl[src_row[t, e]] over
    e < src_cnt[t], alpha = softmax_e(<att_h, leaky_relu(xl[src] + xr[tgt_row[t]], 0.2)>); targets with tgt_row < 0
    give zeros.  xl, xr dense [rows, heads*128], att [heads*128], in the caller's dtype (float64 for a reference) and
    differentiable.  -> out [T, heads*128], alpha [T, capacity, heads] (0 outside the lists)."""
    T, cap, C = src_row.shape[0], src_row.shape[1], 128
    t, e = _edge_list(tgt_row, src_row, src_cnt, 0)
    xs = xl[src_row[t, e].long()].view(-1, heads, C)
    s = torch.nn.functional.leaky_relu(xs + xr[tgt_row[t].long()].view(-1, heads, C), 0.2)
    a = _segment_softmax((s * att.view(heads, C)).sum(-1), t, T)
    out = torch.zeros(T, heads, C, dtype=xl.dtype, device=xl.device).index_add(0, t, a[:, :, None] * xs)
    alpha = torch.zeros(T, cap, heads, dtype=xl.dtype, device=xl.device).index_put((t, e), a)
    return out.view(T, heads * C), alpha


def transformer_edge_reference(q, k, v, tgt_row, src_row, src_cnt, heads):
    """Edge phase of TransformerConv(root_weight=False, beta=False) on the same lists (``mls_transformer_edge_fwd``):
    entry 0 (the node itself) is skipped, logit = <q[tgt_row[t]], k[src]> / sqrt(128), out[t] = sum_e alpha v[src];
    a target without sources gives zeros.  -> out [T, heads*128], alpha [T, capacity, heads]."""
    T, cap, C = src_row.shape[0], src_row.shape[1], 128
    t, e = _edge_list(tgt_row, src_row, src_cnt, 1)
    src = src_row[t, e].long()
    logit = (q[tgt_row[t].long()].view(-1, heads, C) * k[src].view(-1, heads, C)).sum(-1) / math.sqrt(C)
    a = _segment_softmax(logit, t, T)
    out = torch.zeros(T, heads, C, dtype=q.dtype, device=q.device).index_add(0, t, a[:, :, None] * v[src].view(-1, heads, C))
    alpha = torch.zeros(T, cap, heads, dtype=q.dtype, device=q.device).index_put((t, e), a)
    return out.view(T, heads * C), alpha


def agent_rows(N, bs, seed, complete=(), isolated=(), ctrl=None):
    """Synthetic agent-observation rows [bs, 8N+1] float32 with the feature columns the environment writes (small
    integers and flags).  Samples in ``complete`` have every node within the radius of every other (a complete
    graph: capped lists); in samples of ``isolated`` the controlling node is far from all others.  ``ctrl``
    overrides the last column (controlling index, any float: the network clamps and truncates it)."""
    rng = np.random.default_rng(seed)
    om = np.zeros((bs, N, 8), dtype=np.float32)
    om[:, :, :2] = rng.random((bs, N, 2)) * (0.6 if N <= 20 else 1.0)
    om[:, :, 2] = rng.integers(0, 8, size=(bs, N))
    om[:, :, 3] = rng.integers(0, 5, size=(bs, N))
    om[:, :, 4:7] = rng.integers(0, 2, size=(bs, N, 3))
    om[:, :, 7] = rng.random((bs, N)) >= 0.3
    c = rng.integers(0, N, size=bs).astype(np.float32) if ctrl is None else np.asarray(ctrl, dtype=np.float32)
    for b in complete:
        om[b, :, :2] = 0.5 + rng.random((N, 2)) * 0.05
    for b in isolated:
        om[b, :, :2] = rng.random((N, 2)) * 0.4
        om[b, min(max(int(c[b]), 0), N - 1), :2] = (0.95, 0.95)
    return torch.as_tensor(np.concatenate([om.reshape(bs, -1), c[:, None]], axis=1))
