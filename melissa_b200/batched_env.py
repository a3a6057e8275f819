"""BatchedGraphEnv: B independent Melissa dissemination episodes advanced one ROUND per call
by the CUDA kernel behind ``mls_env_step`` (include/melissa_b200.h).

A "round" is what the reference's AEC environment does between two world steps: every
currently-active agent submits one action (graph_env/env/graph.py:303-321), then
``_execute_world_step`` runs (graph.py:361-389), TTL and the next active set are updated
(graph.py:330-345).  Because the shared ``obs_matrix`` only changes inside the world step,
all agents of a round decide on the same state, which is what makes the batched form
exactly equivalent (SURVEY.md section 0).

All state lives in device memory owned by torch; this class only holds tensors and calls
the C ABI.  There is no CPU path.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .topology import GraphPool

_U32 = torch.int32      # torch has no uint32 arithmetic we need; bit patterns are stored in int32 tensors


def _bits_to_i32(a: np.ndarray) -> np.ndarray:
    return np.ascontiguousarray(a.astype(np.uint32)).view(np.int32)


def pack_bits(mask: np.ndarray, W: int) -> np.ndarray:
    """bool [..., N] -> uint32 [..., W] (bit j of word j//32)."""
    n = mask.shape[-1]
    pad = W * 32 - n
    m = np.concatenate([mask.astype(bool), np.zeros(mask.shape[:-1] + (pad,), dtype=bool)], axis=-1)
    m = m.reshape(mask.shape[:-1] + (W, 32)).astype(np.uint64)
    return (m << np.arange(32, dtype=np.uint64)).sum(axis=-1).astype(np.uint32)


class ResetTuplesDevice:
    """Reset tuples (graph index, source, interested set, scripted set) resident on the device."""

    def __init__(self, graph_index, source, interested, scripted, n_nodes, device, pool_size=None):
        W = _lib.words_per_row(n_nodes)
        self.count = int(len(source))
        gi_np, src_np = np.asarray(graph_index, dtype=np.int64), np.asarray(source, dtype=np.int64)
        if self.count and (gi_np.min() < 0 or (pool_size is not None and gi_np.max() >= pool_size)):
            raise ValueError("reset tuples: graph_index outside the topology pool")
        if self.count and (src_np.min() < 0 or src_np.max() >= n_nodes):
            raise ValueError("reset tuples: source node outside the graph")
        self.max_graph = int(gi_np.max()) if self.count else -1
        self.graph_index = torch.as_tensor(np.asarray(graph_index, dtype=np.int32), device=device)
        self.source = torch.as_tensor(np.asarray(source, dtype=np.int32), device=device)
        self.interested = torch.as_tensor(_bits_to_i32(pack_bits(np.asarray(interested, dtype=bool), W)), device=device)
        self.scripted = torch.as_tensor(_bits_to_i32(pack_bits(np.asarray(scripted, dtype=bool), W)), device=device)

    def c_struct(self):
        return _lib.MlsResetTuples(_lib.ptr(self.graph_index), _lib.ptr(self.source), _lib.ptr(self.interested),
                                   _lib.ptr(self.scripted), self.count, 0)


def scripted_count(scripted_agents_ratio: float, n_nodes: int) -> int:
    """Scripted agents per episode, ``round(ratio * N)`` with Python's round (half to even), as the reference draws
    them (core.py:213)."""
    return int(round(scripted_agents_ratio * n_nodes))


class EpisodeStream:
    """Training-mode episode resets drawn on the device: a fresh tuple (graph, source, interested set, scripted set)
    for every reset, without a host-built pool.  Episode number ``r`` of global slot ``s`` is a counter-based Philox
    draw keyed by ``(seed, s, r)`` (include/melissa_b200.h, ``MlsEpisodeSampler``); the global slot of environment
    episode ``b`` is ``b + slot_offset``, so ranks that pass ``slot_offset = rank * B`` never play each other's episodes
    (:func:`melissa_b200.sharding.rank_slot_offset`).  Graphs are drawn uniformly from the first ``pool_size`` graphs
    of the environment's topology pool.

    The tuples follow the reference's training reset chain in distribution, not draw for draw; a
    :class:`ResetTuplesDevice` pool built by :func:`melissa_b200.reset_chain.episode_pool` is the draw-for-draw path."""

    def __init__(self, n_nodes: int, pool_size: int, seed: int, scripted_agents_ratio: float = 0.0, slot_offset: int = 0):
        if not (0.0 <= scripted_agents_ratio <= 1.0):
            raise ValueError("`scripted_agents_ratio` must be in [0.0, 1.0].")          # core.py:143-144
        if not 1 <= int(n_nodes) <= 256:
            raise ValueError(f"n_nodes must be in [1, 256], got {n_nodes}")
        if int(pool_size) < 1:
            raise ValueError(f"pool_size must be >= 1, got {pool_size}")
        if not 0 <= int(slot_offset) < 2 ** 31:
            raise ValueError(f"slot_offset must be in [0, 2**31), got {slot_offset}")
        self.n_nodes, self.pool_size, self.seed = int(n_nodes), int(pool_size), int(seed)
        self.scripted_agents_ratio, self.slot_offset = float(scripted_agents_ratio), int(slot_offset)
        self.n_scripted = scripted_count(self.scripted_agents_ratio, self.n_nodes)
        self.sampler = _lib.MlsEpisodeSampler(self.seed % 2 ** 64, self.pool_size, self.n_scripted,
                                              int(self.scripted_agents_ratio < 1.0), self.slot_offset)

    def sample(self, slots, episode_no, device="cuda") -> ResetTuplesDevice:
        """The tuples episode ``episode_no`` of slot ``slots`` plays (both broadcast to one shape, flattened), as a
        :class:`ResetTuplesDevice` in row order -- exactly what a stream environment draws for those restarts."""
        s, r = np.broadcast_arrays(np.asarray(slots, dtype=np.int64), np.asarray(episode_no, dtype=np.int64))
        s, r = s.ravel(), r.ravel()
        if len(s) and (s.min() < 0 or r.min() < 0 or s.max() >= 2 ** 31 or r.max() >= 2 ** 31):
            raise ValueError("slots and episode numbers must be in [0, 2**31)")
        n, W, dev = len(s), _lib.words_per_row(self.n_nodes), torch.device(device)
        out = ResetTuplesDevice.__new__(ResetTuplesDevice)
        out.count, out.max_graph = n, self.pool_size - 1
        out.graph_index = torch.empty(n, dtype=torch.int32, device=dev)
        out.source = torch.empty(n, dtype=torch.int32, device=dev)
        out.interested = torch.empty(n, W, dtype=torch.int32, device=dev)
        out.scripted = torch.empty(n, W, dtype=torch.int32, device=dev)
        if n:
            sd = torch.as_tensor(s.astype(np.int32), device=dev)
            rd = torch.as_tensor(r.astype(np.int32), device=dev)
            _lib.check(_lib.lib().mls_episode_sample(C.byref(self.sampler), self.n_nodes, sd.data_ptr(), rd.data_ptr(), n,
                                                     out.graph_index.data_ptr(), out.source.data_ptr(),
                                                     out.interested.data_ptr(), out.scripted.data_ptr(),
                                                     _lib.current_stream_ptr()))
        return out


class BatchedGraphEnv:
    """Device-resident vector of ``n_episodes`` graph environments.

    Parameters mirror ``GraphEnv.__init__`` (reference graph.py:25-42) where they affect
    the dynamics: ``number_of_agents``, ``dynamic_graph``, ``is_testing``, ``heuristic``.
    """

    def __init__(self, n_episodes: int, number_of_agents: int, pool: GraphPool, *, dynamic_graph: bool = False,
                 is_testing: bool = False, heuristic: str | None = None, device="cuda", want_obs: bool = True,
                 want_info: bool = False):
        if heuristic not in _lib.HEURISTIC_IDS:
            raise ValueError(f"Unknown heuristic policy: {heuristic}")
        if pool.n_nodes != number_of_agents:
            raise ValueError("graph pool node count does not match number_of_agents")
        self.lib = _lib.lib()                         # fails loudly when the CUDA library is missing
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.MelissaLibraryError("BatchedGraphEnv needs a CUDA device (no CPU fallback)")
        self.B, self.N = int(n_episodes), int(number_of_agents)
        self.W = _lib.words_per_row(self.N)
        self.dynamic, self.is_testing, self.heuristic = bool(dynamic_graph), bool(is_testing), heuristic
        B, N, W, dev = self.B, self.N, self.W, self.device
        self.desc = _lib.MlsEnvDesc(B, N, int(self.dynamic), int(self.is_testing), _lib.HEURISTIC_IDS[heuristic])
        # topology pool
        self.pool = pool
        adj_bits = pack_bits(pool.adj, W)
        self.pool_adj = torch.as_tensor(_bits_to_i32(adj_bits), device=dev)
        self.pool_pos = torch.as_tensor(pool.pos, dtype=torch.float64, device=dev).contiguous()
        # state
        self.node = torch.zeros(B, N, dtype=torch.int32, device=dev)
        self.recv_count = torch.zeros(B, N, dtype=torch.int16, device=dev)
        relay = heuristic in ("mpr", "probabilistic_relay")
        self.recv_from = torch.zeros(B, N, W, dtype=torch.int32, device=dev) if relay else None
        self.episode = torch.zeros(B, _lib.MLS_EP_STRIDE, dtype=torch.int32, device=dev)
        self.rewards_sum = torch.zeros(B, dtype=torch.float64, device=dev)
        self.adj = torch.zeros(B, N, W, dtype=torch.int32, device=dev) if self.dynamic else None
        self.pos = torch.zeros(B, N, 2, dtype=torch.float64, device=dev) if self.dynamic else None
        # round outputs
        self.obs = torch.zeros(B, N, 8, dtype=torch.float32, device=dev) if want_obs else None
        self.reward = torch.zeros(B, N, dtype=torch.float64, device=dev)
        self.active = torch.zeros(B, N, dtype=torch.uint8, device=dev)
        self.terminated = torch.zeros(B, N, dtype=torch.uint8, device=dev)
        self.done = torch.zeros(B, dtype=torch.uint8, device=dev)
        self.info_buf = torch.zeros(B, C.sizeof(_lib.MlsInfo) // 4, dtype=torch.int32, device=dev) if want_info else None
        self.transitions = torch.zeros(1, dtype=torch.int64, device=dev)
        self.recycle: ResetTuplesDevice | EpisodeStream | None = None
        self.philox_seed = 9
        self._state = _lib.MlsEnvState(
            _lib.ptr(self.node), _lib.ptr(self.recv_count), _lib.ptr(self.recv_from), _lib.ptr(self.episode),
            _lib.ptr(self.rewards_sum), _lib.ptr(self.adj), _lib.ptr(self.pos), _lib.ptr(self.pool_adj),
            _lib.ptr(self.pool_pos), len(pool), 0)
        self._out = _lib.MlsRoundOutputs(
            _lib.ptr(self.obs), _lib.ptr(self.reward), _lib.ptr(self.active), _lib.ptr(self.terminated),
            _lib.ptr(self.done), _lib.ptr(self.info_buf), _lib.ptr(self.transitions))

    # ------------------------------------------------------------------ helpers
    def _inputs(self, actions=None, move_offsets=None, gossip_bits=None, relay_bits=None):
        keep = []

        def dev(x, dtype):
            if x is None:
                return None
            if isinstance(x, np.ndarray):
                x = torch.as_tensor(x)
            x = x.to(device=self.device, dtype=dtype).contiguous()
            keep.append(x)
            return x

        a = dev(actions, torch.int8)
        mo = dev(move_offsets, torch.float64)
        gb = dev(gossip_bits, torch.uint8)
        rb = None
        if relay_bits is not None:
            rb_np = relay_bits.cpu().numpy() if isinstance(relay_bits, torch.Tensor) else np.asarray(relay_bits)
            rb = dev(_bits_to_i32(pack_bits(rb_np.astype(bool), self.W)), torch.int32)
        st = _lib.MlsRoundInputs(_lib.ptr(a), _lib.ptr(mo), _lib.ptr(gb), _lib.ptr(rb), self.philox_seed)
        return st, keep

    # ------------------------------------------------------------------ API
    def reset(self, tuples: ResetTuplesDevice | EpisodeStream, env_ids=None, *, move_offsets=None, gossip_bits=None,
              relay_bits=None):
        """Reset episodes ``env_ids`` (default: 0..count) from ``tuples`` -- World.reset +
        GraphEnv.reset (reference core.py:388-437, graph.py:222-248) incl. the forced
        first broadcast.  With an :class:`EpisodeStream` the episodes ``env_ids`` (default: all) draw their next
        episode on the device.  Returns (obs, active)."""
        if isinstance(tuples, EpisodeStream):
            return self._reset_sampled(tuples, env_ids, move_offsets, gossip_bits, relay_bits)
        ids = None
        if env_ids is not None:
            ids = torch.as_tensor(np.asarray(env_ids, dtype=np.int32), device=self.device)
            if len(ids) != tuples.count:
                raise ValueError("env_ids and tuples differ in length")
        elif tuples.count > self.B:
            raise ValueError("more tuples than episodes")
        self._check_tuples(tuples)
        inp, keep = self._inputs(None, move_offsets, gossip_bits, relay_bits)
        tup = tuples.c_struct()
        _lib.check(self.lib.mls_env_reset(C.byref(self.desc), C.byref(self._state), _lib.ptr(ids), C.byref(tup),
                                          C.byref(inp), C.byref(self._out), _lib.current_stream_ptr()))
        return self.obs, self.active

    def _reset_sampled(self, stream: EpisodeStream, env_ids, move_offsets, gossip_bits, relay_bits):
        self._check_stream(stream)
        ids = None
        n = self.B
        if env_ids is not None:
            ids = torch.as_tensor(np.asarray(env_ids, dtype=np.int32).ravel(), device=self.device)
            n = len(ids)
        inp, keep = self._inputs(None, move_offsets, gossip_bits, relay_bits)
        _lib.check(self.lib.mls_env_reset_sampled(C.byref(self.desc), C.byref(self._state), _lib.ptr(ids), n,
                                                  C.byref(stream.sampler), C.byref(inp), C.byref(self._out),
                                                  _lib.current_stream_ptr()))
        return self.obs, self.active

    def set_recycling(self, tuples: ResetTuplesDevice | EpisodeStream | None):
        """Episodes that finish are restarted inside the step kernel from this pool, or with a fresh episode drawn on
        the device when ``tuples`` is an :class:`EpisodeStream`."""
        if isinstance(tuples, EpisodeStream):
            self._check_stream(tuples)
        elif tuples is not None:
            self._check_tuples(tuples)
        self.recycle = tuples

    def _check_tuples(self, tuples: ResetTuplesDevice):
        if getattr(tuples, "max_graph", -1) >= len(self.pool):
            raise ValueError(f"reset tuples name graph {tuples.max_graph} but the topology pool holds {len(self.pool)} graphs")

    def _check_stream(self, stream: EpisodeStream):
        if stream.n_nodes != self.N:
            raise ValueError(f"episode stream draws {stream.n_nodes}-node episodes, the environment has {self.N} nodes")
        if stream.pool_size > len(self.pool):
            raise ValueError(f"episode stream draws from {stream.pool_size} graphs but the topology pool holds {len(self.pool)}")

    def _step(self, desc, state, inp, out):
        rec = self.recycle
        if isinstance(rec, EpisodeStream):
            rc = self.lib.mls_env_step_sampled(C.byref(desc), C.byref(state), C.byref(inp), C.byref(out), C.byref(rec.sampler),
                                               _lib.current_stream_ptr())
        else:
            t = rec.c_struct() if rec is not None else None
            rc = self.lib.mls_env_step(C.byref(desc), C.byref(state), C.byref(inp), C.byref(out),
                                       C.byref(t) if t is not None else None, _lib.current_stream_ptr())
        _lib.check(rc)

    def step(self, actions, *, move_offsets=None, gossip_bits=None, relay_bits=None):
        """One round for all episodes.  ``actions`` int8 [B, N] (device tensor or numpy):
        -1 = None, 0 = stay silent, 1 = forward; only entries of active agents are read.
        Returns (obs f32[B,N,8], reward f64[B,N], active u8[B,N], terminated u8[B,N], done u8[B])."""
        if tuple(actions.shape) != (self.B, self.N):
            raise ValueError(f"actions must have shape {(self.B, self.N)}, got {tuple(actions.shape)}")
        inp, keep = self._inputs(actions, move_offsets, gossip_bits, relay_bits)
        self._step(self.desc, self._state, inp, self._out)
        return self.obs, self.reward, self.active, self.terminated, self.done

    def step_device(self, actions_i8: torch.Tensor):
        """Hot-loop variant of :meth:`step`: ``actions_i8`` is already a contiguous int8 device tensor."""
        inp = _lib.MlsRoundInputs(actions_i8.data_ptr(), None, None, None, self.philox_seed)
        self._step(self.desc, self._state, inp, self._out)

    def step_device_slice(self, actions_i8: torch.Tensor, b0: int, b1: int):
        """One round for episodes ``[b0, b1)`` only (``actions_i8`` = the matching int8 rows).  The slices of
        a round may be stepped one after the other (pipelined with host copies); together they give exactly
        the full-batch round: recycling and the device movement stream are keyed by the batch-wide index."""
        key = (int(b0), int(b1))
        views = self.__dict__.setdefault("_slice_views", {})
        if key not in views:
            sl = lambda t: _lib.ptr(t[b0:b1]) if t is not None else None
            desc = _lib.MlsEnvDesc(b1 - b0, self.N, int(self.dynamic), int(self.is_testing), _lib.HEURISTIC_IDS[self.heuristic],
                                   b0, self.B, 0)
            state = _lib.MlsEnvState(sl(self.node), sl(self.recv_count), sl(self.recv_from), sl(self.episode), sl(self.rewards_sum),
                                     sl(self.adj), sl(self.pos), _lib.ptr(self.pool_adj), _lib.ptr(self.pool_pos), len(self.pool), 0)
            out = _lib.MlsRoundOutputs(sl(self.obs), sl(self.reward), sl(self.active), sl(self.terminated), sl(self.done),
                                       sl(self.info_buf), _lib.ptr(self.transitions))
            views[key] = (desc, state, out)
        desc, state, out = views[key]
        inp = _lib.MlsRoundInputs(actions_i8.data_ptr(), None, None, None, self.philox_seed)
        self._step(desc, state, inp, out)

    def info(self):
        """``get_info`` counters for every episode (reference graph.py:149-179) as a dict of numpy arrays."""
        buf = torch.zeros(self.B, C.sizeof(_lib.MlsInfo) // 4, dtype=torch.int32, device=self.device)
        _lib.check(self.lib.mls_env_info(C.byref(self.desc), C.byref(self._state), buf.data_ptr(), _lib.current_stream_ptr()))
        return decode_info(buf, self.N)

    def last_info(self):
        if self.info_buf is None:
            raise RuntimeError("construct with want_info=True")
        return decode_info(self.info_buf, self.N)

    # convenience views of the packed state (tests, logging)
    def flags(self):
        n = self.node.cpu().numpy().view(np.uint32)
        return dict(
            has_message=(n & _lib.F_HAS_MESSAGE) != 0, interested=(n & _lib.F_INTERESTED) != 0,
            scripted=(n & _lib.F_SCRIPTED) != 0, origin=(n & _lib.F_ORIGIN) != 0,
            has_taken_action=(n & _lib.F_HAS_TAKEN_ACTION) != 0, truncated=(n & _lib.F_TRUNCATED) != 0,
            active=(n & _lib.F_ACTIVE) != 0, steps_taken=(n >> _lib.NODE_STEPS_SHIFT) & 0xFF,
            msgs=(n >> _lib.NODE_MSGS_SHIFT) & 0xFF)


def decode_info(buf: torch.Tensor, n_nodes: int):
    raw = buf.cpu().numpy()
    out = {k: raw[:, i].copy() for i, k in enumerate(_lib.INFO_INT_FIELDS)}
    out["episode_rewards_sum"] = np.ascontiguousarray(raw[:, 12:14]).view(np.float64)[:, 0].copy()
    out["coverage"] = out["covered"] / n_nodes
    with np.errstate(divide="ignore", invalid="ignore"):
        out["coverage_interested_fraction"] = np.where(
            out["interested_agents"] > 0, out["coverage_interested_count"] / np.maximum(out["interested_agents"], 1), 0.0)
    return out
