"""Batched rollout: env round + Q-network forward + epsilon-greedy action selection for
thousands of independent episodes, all on one CUDA stream with no host synchronisation.

This is the loop the reference's collectors drive one agent at a time
(graph_env/env/utils/collectors/multi_agent_collector.py:150-308): ``policy(batch)`` ->
``exploration_noise`` -> ``env.step``.  The unit of work is the agent-transition the
reference counts at multi_agent_collector.py:274 (one live agent taking one decision).
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from .batched_env import BatchedGraphEnv, EpisodeStream, ResetTuplesDevice
from .networks.common import DGNBase
from . import reset_chain


class Rollout:
    def __init__(self, env: BatchedGraphEnv, net: DGNBase | None, *, eps: float = 0.05, seed: int = 9):
        self.env, self.net = env, net
        self.eps, self.seed = float(eps), int(seed)
        self.round_index = 0
        B, N, dev = env.B, env.N, env.device
        self.q = torch.zeros(B, N, 2, dtype=torch.float32, device=dev)
        self.act = torch.full((B, N), -1, dtype=torch.int8, device=dev)
        # device-side round counter: Philox offset of the exploration draws (so a captured CUDA
        # graph draws fresh noise on every replay)
        self.round_dev = torch.zeros(1, dtype=torch.int64, device=dev)
        # observations come from the environment kernel, whose feature columns are small integers:
        # encoder + conv1 projections are evaluated per distinct feature vector (bf16 path)
        self.discrete_features = True
        self.feature_errors = torch.zeros(1, dtype=torch.int32, device=dev)
        self.graph = None
        # host mirrors for the end-to-end (host buffer) path
        self._host = None
        # static graph pools: the radius_graph lists of every pool graph are built once and selected per episode by
        # the graph index the environment keeps on the device (episode[b][MLS_EP_GRAPH])
        self.topology_cache = None
        self.graph_ids = None
        if net is not None:
            net.reserve_workspace(B, dev)      # full-batch size up front: captured graphs bake the address in
            if not env.dynamic and net.precision == "bf16":
                self.topology_cache = net.build_topology_cache(env.pool_pos)
                self.graph_ids = env.episode.view(-1)[_lib.MLS_EP_GRAPH:]

    # ---------------------------------------------------------------- setup helpers
    @staticmethod
    def make_tuples(env: BatchedGraphEnv, count: int, base_seed: int = 9, scripted_agents_ratio: float = 0.0):
        gi, src, inter, scr, _ = reset_chain.episode_pool(base_seed, count, env.N, len(env.pool), scripted_agents_ratio)
        return ResetTuplesDevice(gi, src, inter, scr, env.N, env.device)

    def start(self, tuples: ResetTuplesDevice | EpisodeStream, recycle: bool = True):
        """Reset every episode from the first B tuples; finished episodes restart from the pool.  With an
        :class:`EpisodeStream` every episode, the first ones and every restart (also under CUDA-graph replay: the
        episode numbers live in device state), is a fresh device draw."""
        if isinstance(tuples, EpisodeStream):
            first = tuples
        else:
            if tuples.count < self.env.B:
                raise ValueError(f"need at least {self.env.B} reset tuples (one per episode), got {tuples.count}")
            first = ResetTuplesDevice.__new__(ResetTuplesDevice)
            first.count = self.env.B
            first.graph_index, first.source = tuples.graph_index[: self.env.B], tuples.source[: self.env.B]
            first.interested, first.scripted = tuples.interested[: self.env.B], tuples.scripted[: self.env.B]
        self.env.episode.zero_()            # restart counters too: the recycle pool / stream is walked from its beginning again
        self.env.reset(first)
        self.env.set_recycling(tuples if recycle else None)
        self.round_index = 0
        self.round_dev.zero_()
        self.env.transitions.zero_()

    # ---------------------------------------------------------------- device loop
    def _round_eager(self, obs, active):
        env = self.env
        if self.net is not None:
            self.net.forward_graphs(obs, active, eps=self.eps, philox_seed=self.seed, philox_offset=0,
                                    philox_offset_dev=self.round_dev, q_out=self.q, act_out=self.act,
                                    discrete_features=self.discrete_features, feature_errors=self.feature_errors,
                                    graph_ids=self.graph_ids, graph_id_stride=_lib.MLS_EP_STRIDE,
                                    topology_cache=self.topology_cache, prepared=True)
        env.step_device(self.act)
        self.round_dev.add_(1)

    def round(self):
        """forward (one GNN pass per graph for all its active agents) -> eps-greedy -> env round.
        Replays the captured CUDA graph when :meth:`capture` was called."""
        if self.graph is not None:
            self.graph.replay()
        else:
            self._round_eager(self.env.obs, self.env.active)
        self.round_index += 1

    def refresh_weights(self):
        """Re-pack the network parameters after they changed (optimizer step, load_state_dict).  Captured CUDA
        graphs keep working: they read the packed copies in the (pinned) forward workspace."""
        if self.net is not None:
            self.net.prepare(self.env.B, discrete_features=self.discrete_features)

    def capture(self, warmup_rounds: int = 2):
        """Capture one round (every kernel of forward + env step) into a CUDA graph.  All buffers
        are fixed device tensors and the exploration stream is keyed by a device-side counter,
        so a replay is exactly the eager round without the per-launch host cost."""
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(warmup_rounds):
                self._round_eager(self.env.obs, self.env.active)
                self.round_index += 1
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._round_eager(self.env.obs, self.env.active)
        self.round_index += 1
        self.graph = g
        if self.net is not None:
            self.net.pin_workspace()
        return self

    def transitions(self) -> int:
        return int(self.env.transitions.item())

    # ---------------------------------------------------------------- host-buffer loop (end to end)
    # The host wire format of an observation is the PACKED node (12 bytes: float x, y + one word holding the five
    # integer feature columns and the dm flag, ``mls_obs_pack``) instead of 8 floats (32 bytes): lossless for what the
    # environment writes, 2.7x less PCIe / host-memory traffic per round.  ``unpack_obs_host`` expands it on demand.
    def _pack(self, obs_f32: torch.Tensor, out_u8: torch.Tensor):
        rows = obs_f32.shape[0] * obs_f32.shape[1]
        _lib.check(_lib.lib().mls_obs_pack(obs_f32.data_ptr(), rows, out_u8.data_ptr(), self.pack_errors.data_ptr(),
                                           _lib.current_stream_ptr()))

    def _unpack(self, in_u8: torch.Tensor, obs_f32: torch.Tensor):
        B, N = obs_f32.shape[0], obs_f32.shape[1]
        _lib.check(_lib.lib().mls_obs_unpack(in_u8.data_ptr(), None, None, N, B, N * 8, obs_f32.data_ptr(), _lib.current_stream_ptr()))

    @staticmethod
    def unpack_obs_host(packed) -> np.ndarray:
        """Packed host observations uint8 [B, N, 12] -> float32 [B, N, 8] obs_matrix rows (graph.py:254-271)."""
        p = np.ascontiguousarray(packed.numpy() if isinstance(packed, torch.Tensor) else packed)
        B, N = p.shape[0], p.shape[1]
        xy = p[..., :8].copy().view(np.float32).reshape(B, N, 2)
        w = p[..., 8:12].copy().view(np.uint32).reshape(B, N)
        out = np.empty((B, N, 8), dtype=np.float32)
        out[..., :2] = xy
        out[..., 2] = (w >> 9) & 255
        out[..., 3] = (w >> 3) & 63
        out[..., 4] = (w >> 2) & 1
        out[..., 5] = (w >> 1) & 1
        out[..., 6] = w & 1
        out[..., 7] = w >> 31
        return out

    def _host_buffers(self):
        if self._host is None:
            env = self.env
            B, N, dev = env.B, env.N, env.device
            pin = lambda t: torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            self.pack_errors = torch.zeros(1, dtype=torch.int32, device=dev)
            pobs = torch.empty(B, N, _lib.PACKED_NODE_BYTES, dtype=torch.uint8, device=dev)
            self._host = dict(obs=pin(pobs), active=pin(env.active), reward=pin(env.reward), done=pin(env.done),
                              act=pin(self.act))
            self._dev_in = dict(pobs=torch.empty_like(pobs), obs=torch.empty_like(env.obs), active=torch.empty_like(env.active))
            self._dev_out = dict(pobs=pobs)
            self._pack(env.obs, pobs)
            self._host["obs"].copy_(pobs)
            self._host["active"].copy_(env.active)
        return self._host

    def host_drain(self):
        """Make the calling stream wait for every outstanding copy of :meth:`round_host` (``wait=False``)."""
        if getattr(self, "_pipe", None) is not None:
            torch.cuda.current_stream().wait_stream(self._pipe["d2h"])
            torch.cuda.current_stream().wait_stream(self._pipe["h2d"])

    def sync_host(self):
        """Load the pinned host mirrors with the environment's current observations / active sets."""
        h = self._host_buffers()
        self._pack(self.env.obs, self._dev_out["pobs"])
        h["obs"].copy_(self._dev_out["pobs"])
        h["active"].copy_(self.env.active)
        torch.cuda.synchronize()

    def _compute_slice(self, i: int, b0: int, b1: int):
        """unpack + forward + eps-greedy + env round + pack for episodes [b0, b1) of the host-fed observations."""
        self._unpack(self._dev_in["pobs"][b0:b1], self._dev_in["obs"][b0:b1])
        if self.net is not None:
            self.net.forward_graphs(self._dev_in["obs"][b0:b1], self._dev_in["active"][b0:b1], eps=self.eps,
                                    philox_seed=self.seed, philox_offset=0, philox_offset_dev=self.round_dev, philox_row0=b0 * self.env.N,
                                    q_out=self.q[b0:b1], act_out=self.act[b0:b1],
                                    discrete_features=self.discrete_features, feature_errors=self.feature_errors,
                                    graph_ids=None if self.graph_ids is None else self.graph_ids[b0 * _lib.MLS_EP_STRIDE:],
                                    graph_id_stride=_lib.MLS_EP_STRIDE, topology_cache=self.topology_cache, prepared=True)
        self.env.step_device_slice(self.act[b0:b1], b0, b1)
        self._pack(self.env.obs[b0:b1], self._dev_out["pobs"][b0:b1])

    def capture_host(self, sub_batches: int):
        """Capture the compute of every episode slice of :meth:`round_host` into its own CUDA graph (the slices
        are 1/sub_batches of a round: without graphs the ~24 launches per slice cost more host time than the
        kernels run).  Runs one untimed round; call before :meth:`start`."""
        self._host_buffers()
        env = self.env
        S = max(1, min(int(sub_batches), env.B))
        bounds = [(env.B * i // S, env.B * (i + 1) // S) for i in range(S)]
        self._pack(env.obs, self._dev_in["pobs"])
        self._dev_in["active"].copy_(env.active)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for i, (b0, b1) in enumerate(bounds):
                self._compute_slice(i, b0, b1)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graphs = []
        for i, (b0, b1) in enumerate(bounds):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                self._compute_slice(i, b0, b1)
            graphs.append(g)
        self._host_graphs = (S, graphs)
        if self.net is not None:
            self.net.pin_workspace()
        return self

    def feature_violations(self) -> int:
        """Node rows of the last forward whose feature columns were not the small integers the environment writes
        (always 0 for observations produced by the environment kernel; see MLS_FWD_DISCRETE_FEATURES)."""
        return int(self.feature_errors.item())

    def round_host(self, sub_batches: int = 1, wait: bool = True, trace: list | None = None):
        """The same round through host buffers, as a caller holding numpy observations would
        drive it: obs/active H2D -> forward + act -> env round -> obs/reward/active/done/act D2H.
        With ``sub_batches`` > 1 the batch is processed in that many slices of episodes: the H2D copy of
        slice i+1 and the D2H copy of slice i-1 run on their own streams while slice i computes (same
        results as one full-batch round up to the exploration draws, which are keyed per slice).
        ``wait=False`` does not make the calling stream wait for the round's last D2H copy: the slices of
        consecutive rounds then overlap too (slice i of round k+1 only waits for slice i of round k to be back
        on the host, exactly the dependency a caller feeding observations back has); call :meth:`host_drain`
        before reading the host buffers.  ``trace`` (a list) collects (tag, slice, timing event) marks of the pipeline's
        phases on their streams (diagnostics: bench.py --e2e-trace).  Returns (h2d_bytes, d2h_bytes)."""
        h = self._host_buffers()
        env = self.env
        nb = lambda t: t.numel() * t.element_size()
        nbytes = (nb(h["obs"]) + nb(h["active"]), nb(h["act"]) + nb(h["obs"]) + nb(h["reward"]) + nb(h["active"]) + nb(h["done"]))
        S = max(1, min(int(sub_batches), env.B))
        if S == 1:
            self._dev_in["pobs"].copy_(h["obs"], non_blocking=True)
            self._dev_in["active"].copy_(h["active"], non_blocking=True)
            self._unpack(self._dev_in["pobs"], self._dev_in["obs"])
            self._round_eager(self._dev_in["obs"], self._dev_in["active"])
            self._pack(env.obs, self._dev_out["pobs"])
            self.round_index += 1
            h["act"].copy_(self.act, non_blocking=True)
            h["obs"].copy_(self._dev_out["pobs"], non_blocking=True)
            h["reward"].copy_(env.reward, non_blocking=True)
            h["active"].copy_(env.active, non_blocking=True)
            h["done"].copy_(env.done, non_blocking=True)
            return nbytes
        if getattr(self, "_pipe", None) is None or self._pipe["S"] != S:
            self._pipe = dict(S=S, h2d=torch.cuda.Stream(), d2h=torch.cuda.Stream(),
                              ev_h=[torch.cuda.Event() for _ in range(S)], ev_c=[torch.cuda.Event() for _ in range(S)],
                              ev_d=[torch.cuda.Event() for _ in range(S)], rounds=0,
                              ev_start=torch.cuda.Event(), ev_end=torch.cuda.Event())
        P = self._pipe
        cur = torch.cuda.current_stream()

        def mark(stream, tag, i):
            if trace is not None:
                e = torch.cuda.Event(enable_timing=True)
                e.record(stream)
                trace.append((tag, i, e))
        bounds = [(env.B * i // S, env.B * (i + 1) // S) for i in range(S)]
        if P["rounds"] == 0 or wait:
            P["ev_start"].record(cur)               # the copies of this round start after everything queued before it
            P["h2d"].wait_event(P["ev_start"])
            P["d2h"].wait_event(P["ev_start"])
        with torch.cuda.stream(P["h2d"]):
            for i, (b0, b1) in enumerate(bounds):
                if P["rounds"] > 0:
                    P["h2d"].wait_event(P["ev_d"][i])   # slice i of the previous round is back on the host (and off _dev_in)
                mark(P["h2d"], "h2d_begin", i)
                self._dev_in["pobs"][b0:b1].copy_(h["obs"][b0:b1], non_blocking=True)
                self._dev_in["active"][b0:b1].copy_(h["active"][b0:b1], non_blocking=True)
                P["ev_h"][i].record(P["h2d"])
                mark(P["h2d"], "h2d_end", i)
        graphs = self._host_graphs[1] if getattr(self, "_host_graphs", None) and self._host_graphs[0] == S else None
        for i, (b0, b1) in enumerate(bounds):
            cur.wait_event(P["ev_h"][i])
            mark(cur, "compute_begin", i)
            if graphs is not None:
                graphs[i].replay()
            else:
                self._compute_slice(i, b0, b1)
            P["ev_c"][i].record(cur)
            mark(cur, "compute_end", i)
            with torch.cuda.stream(P["d2h"]):
                P["d2h"].wait_event(P["ev_c"][i])
                mark(P["d2h"], "d2h_begin", i)
                h["act"][b0:b1].copy_(self.act[b0:b1], non_blocking=True)
                h["obs"][b0:b1].copy_(self._dev_out["pobs"][b0:b1], non_blocking=True)
                h["reward"][b0:b1].copy_(env.reward[b0:b1], non_blocking=True)
                h["active"][b0:b1].copy_(env.active[b0:b1], non_blocking=True)
                h["done"][b0:b1].copy_(env.done[b0:b1], non_blocking=True)
                P["ev_d"][i].record(P["d2h"])
                mark(P["d2h"], "d2h_end", i)
        P["rounds"] += 1
        if wait:
            P["ev_end"].record(P["d2h"])
            cur.wait_event(P["ev_end"])             # the round is over when its last result is on the host
        self.round_dev.add_(1)
        self.round_index += 1
        return nbytes
