"""Shared host code of the three Q-network modules.

The modules keep the reference's constructor signature, attribute names and state_dict
keys (SURVEY.md Appendix B.6) so that checkpoints written by the reference load
unchanged, but their forward pass is one call into ``mls_dgn_forward``
(include/melissa_b200.h): obs never leaves the device, the graph is rebuilt from the node
positions inside the kernels (reference networks/common.py:47-48) and the GNN body runs
once per graph for all controlling agents.

Parameter containers only hold tensors; they have no torch compute.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Any, Dict, Optional, Tuple

import numpy as np
import torch
import torch.nn as nn

from .. import _lib

RADIUS_OF_INFLUENCE = 0.20      # reference constants.py:1


class MLPParams(nn.Module):
    """Parameter layout of tianshou ``MLP``: ``model = Sequential(Linear, ReLU, ..., Linear)``
    -> keys ``model.0.weight``, ``model.2.weight``, ..."""

    def __init__(self, input_dim: int, output_dim: int, hidden_sizes):
        super().__init__()
        dims = [input_dim, *hidden_sizes, output_dim]
        layers = []
        for k in range(len(dims) - 1):
            layers.append(nn.Linear(dims[k], dims[k + 1]))
            if k + 2 < len(dims):
                layers.append(nn.ReLU())
        self.model = nn.Sequential(*layers)

    def linears(self):
        return [m for m in self.model if isinstance(m, nn.Linear)]


def _glorot_(t: torch.Tensor):
    a = math.sqrt(6.0 / (t.size(-2) + t.size(-1)))
    with torch.no_grad():
        t.uniform_(-a, a)


class GATv2Params(nn.Module):
    """Parameter layout + default init of PyG ``GATv2Conv(in, out, heads)``."""

    def __init__(self, in_channels: int, out_channels: int, heads: int):
        super().__init__()
        self.lin_l = nn.Linear(in_channels, heads * out_channels)
        self.lin_r = nn.Linear(in_channels, heads * out_channels)
        self.att = nn.Parameter(torch.empty(1, heads, out_channels))
        self.bias = nn.Parameter(torch.zeros(heads * out_channels))
        for lin in (self.lin_l, self.lin_r):
            _glorot_(lin.weight)
            nn.init.zeros_(lin.bias)
        _glorot_(self.att)


class TransformerConvParams(nn.Module):
    """Parameter layout of PyG ``TransformerConv(in, out, heads, root_weight=False)``.
    ``lin_skip`` is constructed by PyG and saved in checkpoints but never used in forward."""

    def __init__(self, in_channels: int, out_channels: int, heads: int):
        super().__init__()
        self.lin_key = nn.Linear(in_channels, heads * out_channels)
        self.lin_query = nn.Linear(in_channels, heads * out_channels)
        self.lin_value = nn.Linear(in_channels, heads * out_channels)
        self.lin_skip = nn.Linear(in_channels, heads * out_channels)


class _Workspace:
    """Scratch memory of the forward kernels.  Once a CUDA graph has captured a forward (``pinned``), the buffer's
    address is baked into the graph (and into the TMA descriptors encoded from it), so it must never be replaced:
    a later call that needs more bytes raises instead of silently freeing memory the graph still replays into."""

    def __init__(self):
        self.buf = None
        self.pinned = False

    def get(self, nbytes: int, device):
        if self.buf is None or self.buf.numel() < nbytes or self.buf.device != device:
            if self.pinned and self.buf is not None:
                raise _lib.MelissaLibraryError(
                    f"forward workspace ({self.buf.numel()} bytes) is pinned by a captured CUDA graph but this call needs "
                    f"{nbytes} bytes: call reserve_workspace(max_graphs) before capturing")
            self.buf = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=device)
        return self.buf


class DGNBase(nn.Module):
    """Common machinery: validation, weight struct, C-ABI call."""

    KIND = ""

    def _init_common(self, input_dim, hidden_dim, output_dim, num_heads, agents_num, dueling_param, device,
                     edge_attributes):
        self.device = device
        self.input_dim = input_dim
        self.hidden_dim = hidden_dim
        self.output_dim = output_dim
        self.num_heads = num_heads
        self.agents_num = agents_num
        self.edge_attributes = edge_attributes      # accepted; no effect on results (convs get no edge_attr)
        self.use_dueling = dueling_param is not None
        self.precision = "fp32"
        self.train_precision = "fp32"
        self._ws = _Workspace()
        self._prepared = None

    def _build_heads(self, latent, dueling_param, output_dim):
        if dueling_param is None:
            # l_dgn.py:88-90 / dgn_r.py / hl_dgn.py: a single linear layer on the latent row
            if output_dim != 2:
                raise NotImplementedError("the environment's action space is Discrete(2)")
            self.head_hidden = 128                   # unused by the kernels for this head
            self.out_linear = nn.Linear(latent, output_dim)
            self.output_dim = output_dim
            return
        q_kwargs, v_kwargs = dict(dueling_param[0]), dict(dueling_param[1])
        qh, vh = list(q_kwargs.get("hidden_sizes", ())), list(v_kwargs.get("hidden_sizes", ()))
        if len(qh) != 2 or qh != vh or qh[0] != qh[1]:
            raise NotImplementedError("dueling heads must be two equal hidden layers, e.g. [128, 128]")
        self.head_hidden = qh[0]
        q_out = q_kwargs.get("output_dim", output_dim)
        if q_out != 2:
            raise NotImplementedError("the environment's action space is Discrete(2)")
        self.Q = MLPParams(latent, q_out, qh)
        self.V = MLPParams(latent, v_kwargs.get("output_dim", 1), vh)
        self.output_dim = q_out

    # ------------------------------------------------------------------ C-ABI plumbing
    def set_precision(self, precision: str):
        if precision not in _lib.PRECISIONS:
            raise ValueError(precision)
        self.precision = precision
        return self

    def set_train_precision(self, precision: str):
        """Precision of the dense layers in the differentiable training forward and its backward
        (``networks/autograd.py``): "fp32" (default) or "bf16" -- bf16 operands, fp32 accumulation on the tensor cores,
        fp32 master weights and fp32 activations between layers (``mls_linear_bf16_*``; CUDA tensors only).
        Independent of :meth:`set_precision`, which selects the rollout forward."""
        if precision not in ("fp32", "bf16"):
            raise ValueError(precision)
        self.train_precision = precision
        return self

    def _desc(self):
        return _lib.MlsNetDesc(_lib.NET_KINDS[self.KIND], self.agents_num, self.hidden_dim, self.num_heads,
                               self.input_dim, _lib.POOLS[getattr(self, "aggregator_name", "mean")],
                               _lib.PRECISIONS[self.precision], self.head_hidden)

    def _conv_tensors(self, conv):
        raise NotImplementedError

    def weights_struct(self):
        """MlsNetWeights over the live parameters (must be fp32, contiguous, on the GPU)."""
        enc = self.encoder.linears()
        q, v = (self.Q.linears(), self.V.linears()) if self.use_dueling else ([], [])
        t = {"enc_w0": enc[0].weight, "enc_b0": enc[0].bias, "enc_w1": enc[1].weight, "enc_b1": enc[1].bias}
        if not self.use_dueling:
            t["out_w"], t["out_b"] = self.out_linear.weight, self.out_linear.bias
        for name, conv in (("c1", self.conv1), ("c2", getattr(self, "conv2", None))):
            vals = self._conv_tensors(conv) if conv is not None else [None] * 8
            for k, val in zip(("wa", "ba", "wb", "bb", "wc", "bc", "att", "bias"), vals):
                t[f"{name}_{k}"] = val
        for pre, lins in (("q", q), ("v", v)):
            for k, lin in enumerate(lins):
                t[f"{pre}_w{k}"], t[f"{pre}_b{k}"] = lin.weight, lin.bias
        keep = []
        ws = _lib.MlsNetWeights()
        for k in _lib.WEIGHT_FIELDS:
            x = t.get(k)
            if x is None:
                setattr(ws, k, None)
                continue
            x = x.detach()
            if x.dtype != torch.float32 or not x.is_cuda:
                raise _lib.MelissaLibraryError(
                    f"parameter {k} must be a float32 CUDA tensor (module on {x.device}, {x.dtype}); "
                    "there is no CPU forward -- move the module to the GPU")
            x = x.contiguous()
            if x.data_ptr() % 16:
                raise _lib.MelissaLibraryError(f"parameter {k} must start on a 16-byte boundary (the kernels read it with 16-byte loads)")
            keep.append(x)
            setattr(ws, k, x.data_ptr())
        return ws, keep

    def _validate_obs(self, obs):
        if obs.ndim != 2:
            raise ValueError(f"Expected obs to be 2D, but got shape {obs.shape}")
        bs, dim = obs.shape
        expected = self.agents_num * (self.input_dim + 2 + 1)
        if dim - 1 != expected:
            raise ValueError(f"Expected {expected} feature cols for nodes, got {dim - 1}")
        return bs

    def _param_version(self):
        """Changes whenever a parameter tensor is written in place or replaced (optimizer step, load_state_dict), or
        when a kernel that writes the parameters behind torch's back says so (:meth:`mark_parameters_changed`)."""
        return (getattr(self, "_manual_version", 0),) + tuple((p.data_ptr(), p._version) for p in self.parameters())

    def mark_parameters_changed(self):
        self._manual_version = getattr(self, "_manual_version", 0) + 1

    def clone_for_target(self):
        """A detached copy for the DQN target network (tianshou: ``deepcopy(model)``) with its own, still
        unallocated, forward workspace."""
        import copy
        ws, prof = self._ws, getattr(self, "_prof", None)
        self._ws, self._prof = _Workspace(), None
        try:
            twin = copy.deepcopy(self)
        finally:
            self._ws, self._prof = ws, prof
        twin._prepared = None
        for p in twin.parameters():
            p.requires_grad_(False)
        return twin

    def prepare(self, n_graphs: int = 1, *, discrete_features: bool = True):
        """Pack the parameters into the forward workspace once (bf16 weight matrices, stacked biases and -- with
        ``discrete_features`` -- the feature tables), so that later forwards skip it (``MLS_FWD_PREPARED``).  Call
        again after the parameters change (optimizer step / load_state_dict); ``forward_graphs(prepared=True)``
        checks this with the parameters' version counters and re-packs on its own outside CUDA-graph capture."""
        if self.precision != "bf16":
            self._prepared = None
            return self
        L = _lib.lib()
        dev = next(self.parameters()).device
        desc = self._desc()
        ws, keep = self.weights_struct()
        wsp = self.reserve_workspace(max(1, int(n_graphs)), dev) if (self._ws.buf is None or self._ws.buf.device != dev) else self._ws.buf
        flags = _lib.FWD_DISCRETE_FEATURES if discrete_features else 0
        _lib.check(L.mls_dgn_prepare(C.byref(desc), C.byref(ws), flags, wsp.data_ptr(), wsp.numel(), _lib.current_stream_ptr()))
        self._prepared = (self._param_version(), flags, wsp.data_ptr())
        return self

    def build_topology_cache(self, pool_pos):
        """radius_graph lists of every graph of a STATIC pool, built once (``mls_dgn_csr_cache_build``).
        ``pool_pos``: float64/float32 [G, N, 2] node positions (what the environment writes into obs columns 0..1).
        Returns an opaque cache object for ``forward_graphs(..., graph_ids=, topology_cache=)``."""
        L = _lib.lib()
        dev = next(self.parameters()).device
        pos = torch.as_tensor(pool_pos).to(device=dev)
        G, N = int(pos.shape[0]), int(pos.shape[1])
        if N != self.agents_num:
            raise ValueError("graph pool node count does not match agents_num")
        rows = torch.zeros(G, N, 8, dtype=torch.float32, device=dev)
        rows[:, :, 0:2] = pos.to(torch.float32)          # same double -> float rounding as the environment's obs rows
        desc = self._desc()
        nbytes = L.mls_dgn_csr_cache_bytes(C.byref(desc), G)
        buf = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        _lib.check(L.mls_dgn_csr_cache_build(C.byref(desc), rows.data_ptr(), N * 8, G, buf.data_ptr(), nbytes,
                                             _lib.current_stream_ptr()))
        return {"buf": buf, "graphs": G}

    def _call(self, obs, stride, n_graphs, ctrl_mode, ctrl_mask, q, act, eps, seed, offset, rand3, offset_dev=None,
              flags=0, feature_errors=None, graph_ids=None, graph_id_stride=1, topology_cache=None, prepared=False,
              philox_row0=0):
        L = _lib.lib()
        desc = self._desc()
        ws, keep = self.weights_struct()
        nbytes = L.mls_dgn_workspace_bytes(C.byref(desc), n_graphs)
        wsp = self._ws.get(nbytes, obs.device)
        if prepared and self.precision == "bf16":
            pf = flags & _lib.FWD_DISCRETE_FEATURES
            want = (self._param_version(), pf, wsp.data_ptr())
            if getattr(self, "_prepared", None) != want:
                if torch.cuda.is_current_stream_capturing():
                    raise _lib.MelissaLibraryError("parameters changed since prepare(): call prepare() before CUDA-graph capture")
                _lib.check(L.mls_dgn_prepare(C.byref(desc), C.byref(ws), pf, wsp.data_ptr(), wsp.numel(), _lib.current_stream_ptr()))
                self._prepared = want
            flags |= _lib.FWD_PREPARED
        args = _lib.MlsForwardArgs(obs.data_ptr(), stride, n_graphs, ctrl_mode, _lib.ptr(ctrl_mask), q.data_ptr(),
                                   _lib.ptr(act), float(eps), int(flags), int(seed), int(offset), _lib.ptr(rand3),
                                   wsp.data_ptr(), wsp.numel(), None, None, 0, 0, _lib.ptr(offset_dev), _lib.ptr(feature_errors))
        args.philox_row0 = int(philox_row0)
        if topology_cache is not None and graph_ids is not None and self.precision == "bf16":
            if graph_ids.dtype != torch.int32:
                raise ValueError("graph_ids must be an int32 tensor")
            args.graph_ids = graph_ids.data_ptr()
            args.graph_id_stride = int(graph_id_stride)
            args.csr_cache_graphs = int(topology_cache["graphs"])
            args.csr_cache = topology_cache["buf"].data_ptr()
        prof = getattr(self, "_prof", None)
        if prof is not None:          # (cudaEvent start, cudaEvent stop, kernel id), see set_profile_events
            args.prof_start, args.prof_stop, args.prof_kernel = prof[0].cuda_event, prof[1].cuda_event, prof[2]
        _lib.check(L.mls_dgn_forward(C.byref(desc), C.byref(ws), C.byref(args), _lib.current_stream_ptr()))

    def reserve_workspace(self, n_graphs: int, device=None):
        """Size the forward workspace for passes of up to ``n_graphs`` graphs (call before CUDA-graph capture)."""
        device = device or next(self.parameters()).device
        desc = self._desc()
        return self._ws.get(_lib.lib().mls_dgn_workspace_bytes(C.byref(desc), int(n_graphs)), torch.device(device))

    def pin_workspace(self, pinned: bool = True):
        self._ws.pinned = bool(pinned)

    def set_profile_events(self, kernel: Optional[str], start=None, stop=None):
        """Record ``start``/``stop`` (torch.cuda.Event with timing) around one launch of the named
        kernel class in every forward call (bench.py roofline line).  ``None`` switches it off."""
        if kernel is None:
            self._prof = None
        else:
            start.record(); stop.record()      # materialise the underlying cudaEvent_t handles
            self._prof = (start, stop, _lib.PROF_KERNELS[kernel])

    # ------------------------------------------------------------------ public
    def forward(self, obs, state=None, info={}):
        """Reference signature: obs [bs, 8N+1] (ndarray or tensor; last column = controlling
        agent index) -> (q [bs, 2], state)."""
        dev = next(self.parameters()).device
        if isinstance(obs, np.ndarray):
            obs = torch.as_tensor(obs, device=dev)
        bs = self._validate_obs(obs)
        obs = obs.to(device=dev, dtype=torch.float32).contiguous()
        q = torch.empty(bs, 2, dtype=torch.float32, device=dev)
        if bs:
            self._call(obs, obs.shape[1], bs, 1, None, q, None, 0.0, 0, 0, None)
        return q, self._state_out(state)

    def _state_out(self, state):
        return state

    @torch.no_grad()
    def forward_graphs(self, obs_matrix: torch.Tensor, ctrl_mask: torch.Tensor, *, eps: float = 0.0,
                       philox_seed: int = 0, philox_offset: int = 0, rand3: Optional[torch.Tensor] = None,
                       q_out: Optional[torch.Tensor] = None, act_out: Optional[torch.Tensor] = None,
                       philox_offset_dev: Optional[torch.Tensor] = None, discrete_features: bool = False,
                       feature_errors: Optional[torch.Tensor] = None, graph_ids: Optional[torch.Tensor] = None,
                       graph_id_stride: int = 1, topology_cache=None, prepared: bool = False, philox_row0: int = 0):
        """Rollout form: obs_matrix f32 [B, N, 8] (what ``BatchedGraphEnv`` emits), ctrl_mask
        u8 [B, N] (the active set).  One GNN pass per graph; returns (q f32 [B,N,2] -- zero
        where not controlling, act i8 [B,N] -- -1 where not controlling).

        ``discrete_features=True`` (bf16 precision): the caller guarantees that the feature columns hold the
        small integers the environment writes (always true for ``BatchedGraphEnv.obs``); encoder and conv1
        projections are then evaluated once per distinct feature vector instead of once per node.
        ``feature_errors`` (int32[1] device tensor) receives the number of rows violating that promise.
        ``graph_ids`` (int32 device tensor, graph g's pool index at ``graph_ids.flatten()[g * graph_id_stride]``) +
        ``topology_cache`` (:meth:`build_topology_cache`): static graph pools skip the per-call radius_graph pass.
        ``prepared=True``: weights / feature tables are packed once per parameter version (:meth:`prepare`).
        ``philox_row0``: first batch-wide row (episode * N) of a sub-batch call, so that the exploration draws of a
        batch processed in slices equal those of one full-batch call."""
        B, N, F = obs_matrix.shape
        if N != self.agents_num or F != self.input_dim + 3:
            raise ValueError(f"Expected obs_matrix [B, {self.agents_num}, {self.input_dim + 3}], got {tuple(obs_matrix.shape)}")
        dev = obs_matrix.device
        q = q_out if q_out is not None else torch.empty(B, N, 2, dtype=torch.float32, device=dev)
        act = act_out if act_out is not None else torch.empty(B, N, dtype=torch.int8, device=dev)
        if B:
            flags = _lib.FWD_DISCRETE_FEATURES if (discrete_features and self.precision == "bf16") else 0
            self._call(obs_matrix.contiguous(), N * F, B, 0, ctrl_mask.contiguous(), q, act, eps, philox_seed,
                       philox_offset, rand3, philox_offset_dev, flags, feature_errors, graph_ids, graph_id_stride,
                       topology_cache, prepared, philox_row0)
        return q, act
