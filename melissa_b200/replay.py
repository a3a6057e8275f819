"""Device-resident replay of the batched rollout.

The reference keeps one tianshou sub-buffer per (env, agent) (``VectorReplayBuffer(buffer_num = envs * agents,
ignore_obs_next=True)``, l_dgn.py:170-182) and ``MultiAgentCollector`` completes an agent's transition when that
agent's next observation appears, with the reward set by the world step in between
(multi_agent_collector.py:240-308).  In the batched form all of an episode's agents decide on the same
``obs_matrix`` each round and an active agent stays active until its TTL ends (graph.py:330-345), so

    transition (round r, episode b, agent a) = (obs_matrix[r][b], a, act[r][b][a], reward[r][b][a], terminated[r][b][a])
    its successor                              = (round r+1, episode b, agent a)            (exists iff not terminated)

and the per-(env, agent) sub-buffers become ONE dense ring ``[ring round][episode][agent]``: storing a round is a
copy of what the kernels already produced, the chains are implicit, ``obs_next`` is never stored
(``ignore_obs_next``).  Frames are kept packed (12 bytes per node, ``mls_obs_pack``).  An episode only ends when
every agent that ever acted has terminated, so no chain crosses an in-place episode restart.

Everything stays on the device; sampling returns the reference's agent-observation rows ``[M, 8N+1]``.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib

F_ACTED, F_TERMINATED = 1, 2


class DeviceReplay:
    def __init__(self, n_episodes: int, n_nodes: int, ring_rounds: int, device="cuda", seed: int = 0):
        self.lib = _lib.lib()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.MelissaLibraryError("DeviceReplay needs a CUDA device (no CPU fallback)")
        self.B, self.N, self.R = int(n_episodes), int(n_nodes), int(ring_rounds)
        B, N, R, dev = self.B, self.N, self.R, self.device
        self.frames = torch.zeros(R, B, N, _lib.PACKED_NODE_BYTES, dtype=torch.uint8, device=dev)
        self.act = torch.zeros(R, B, N, dtype=torch.int8, device=dev)
        self.rew = torch.zeros(R, B, N, dtype=torch.float64, device=dev)
        self.flags = torch.zeros(R, B, N, dtype=torch.uint8, device=dev)
        self.counts = torch.zeros(R, dtype=torch.int64, device=dev)       # stored transitions per ring round
        self.cells = torch.zeros(R, B * N, dtype=torch.int32, device=dev)  # their (episode * N + agent) cells, compacted
        self._nonempty = False
        self.pack_errors = torch.zeros(1, dtype=torch.int32, device=dev)
        self.head = 0              # rounds stored so far (ring slot = head % R)
        self._pending = None       # slot whose reward / terminated are still to come
        self.gen = torch.Generator(device=dev)
        self.gen.manual_seed(int(seed))

    def __len__(self):
        """Stored transitions whose outcome is known (what tianshou calls len(buffer))."""
        return int(self.counts.sum().item())

    # ------------------------------------------------------------------ writing
    def begin_round(self, obs: torch.Tensor, active: torch.Tensor):
        """Before the policy acts: the observation every active agent of this round decides on."""
        if self._pending is not None:
            raise RuntimeError("begin_round called twice without end_round")
        slot = self.head % self.R
        _lib.check(self.lib.mls_obs_pack(obs.data_ptr(), self.B * self.N, self.frames[slot].data_ptr(),
                                         self.pack_errors.data_ptr(), _lib.current_stream_ptr()))
        acted = active.ne(0)
        self.flags[slot].copy_(acted)                                 # bit 0: acted
        self.counts[slot] = acted.sum()
        self.cells[slot].copy_(torch.nonzero_static(acted.view(-1), size=self.B * self.N, fill_value=0)[:, 0])
        self._pending = slot

    def end_round(self, act: torch.Tensor, reward: torch.Tensor, terminated: torch.Tensor):
        """After the environment round: actions taken, the reward of the world step, TTL terminations."""
        slot = self._pending
        if slot is None:
            raise RuntimeError("end_round without begin_round")
        self.act[slot].copy_(act)
        self.rew[slot].copy_(reward)
        self.flags[slot].add_(terminated.ne(0).to(torch.uint8) * F_TERMINATED * self.flags[slot])   # bit 1 only where acted
        self._pending = None
        self.head += 1

    # ------------------------------------------------------------------ sampling
    def _usable_rounds(self, n_step: int):
        """Round rho is usable when rounds rho .. rho+n_step are all in the ring (a chain still alive after n_step steps
        bootstraps from the observation of round rho+n_step, which is only packed by the next ``begin_round``).
        -> (ring slot of the oldest usable round, number of usable rounds); the newest n_step rounds are not usable."""
        if n_step >= self.R:
            raise ValueError(f"a ring of {self.R} rounds cannot hold an n-step window of {n_step} rounds plus its "
                             "bootstrap frame (needs ring_rounds > n_step)")
        filled = min(self.head, self.R)
        usable = filled - n_step                   # rounds rho .. rho+n_step must be stored; the oldest is overwritten last
        if usable <= 0:
            raise RuntimeError("not enough rounds stored for an n-step window")
        if not self._nonempty:                     # one host check, then everything stays on the device
            if int(self.counts.sum().item()) == 0:
                raise RuntimeError("replay holds no transitions yet")
            self._nonempty = True
        return (self.head - filled) % self.R, usable

    def sample_indices(self, batch_size: int, n_step: int):
        """Uniform over the stored transitions of the usable rounds (``_usable_rounds``): their n-step window AND its
        bootstrap frame are stored.  Needs ``ring_rounds > n_step``.  -> (ring round, episode, agent) int32 tensors [M]."""
        first, usable = self._usable_rounds(n_step)
        # ring slots ordered oldest -> newest
        order = (torch.arange(usable, device=self.device) + first) % self.R
        cnt = self.counts[order]
        cum = torch.cumsum(cnt, 0)
        total = cum[-1]
        u = torch.rand(batch_size, device=self.device, generator=self.gen, dtype=torch.float64)
        k = torch.minimum((u * total).long(), total - 1).clamp_(min=0)
        seg = torch.searchsorted(cum, k, right=True).clamp_(max=usable - 1)
        within = k - (cum[seg] - cnt[seg])
        rho = order[seg]
        cell = self.cells[rho, within].long()
        return rho.to(torch.int32), (cell // self.N).to(torch.int32), (cell % self.N).to(torch.int32)

    def gather(self, rho, ep, agent, n_step: int, gamma: float):
        """-> dict(obs rows [M, 8N+1] f32, act [M] i64, returns [M] f32 (n-step, without the bootstrap term),
        boot_round [M] i32 (-1: chain ended inside the window), boot_gamma [M] f32)."""
        M = int(rho.shape[0])
        dev = self.device
        rows = torch.empty(M, self.N * 8 + 1, dtype=torch.float32, device=dev)
        frame = rho.to(torch.int64) * self.B + ep.to(torch.int64)
        _lib.check(self.lib.mls_obs_unpack(self.frames.data_ptr(), frame.data_ptr(), agent.data_ptr(), self.N, M,
                                           self.N * 8 + 1, rows.data_ptr(), _lib.current_stream_ptr()))
        ret = torch.empty(M, dtype=torch.float32, device=dev)
        boot = torch.empty(M, dtype=torch.int32, device=dev)
        bg = torch.empty(M, dtype=torch.float32, device=dev)
        _lib.check(self.lib.mls_nstep_returns(self.rew.data_ptr(), self.flags.data_ptr(), self.R, self.B, self.N, rho.data_ptr(),
                                              ep.data_ptr(), agent.data_ptr(), M, int(n_step), float(gamma), ret.data_ptr(),
                                              boot.data_ptr(), bg.data_ptr(), _lib.current_stream_ptr()))
        act = self.act[rho.long(), ep.long(), agent.long()].to(torch.int64)
        return dict(obs=rows, act=act, returns=ret, boot_round=boot, boot_gamma=bg, ep=ep, agent=agent)

    def rows_at(self, ring_round, ep, agent):
        """Agent-observation rows of (ring round, episode, agent) triples (bootstrap observations)."""
        M = int(ring_round.shape[0])
        rows = torch.empty(M, self.N * 8 + 1, dtype=torch.float32, device=self.device)
        frame = ring_round.to(torch.int64) * self.B + ep.to(torch.int64)
        _lib.check(self.lib.mls_obs_unpack(self.frames.data_ptr(), frame.data_ptr(), agent.to(torch.int32).contiguous().data_ptr(),
                                           self.N, M, self.N * 8 + 1, rows.data_ptr(), _lib.current_stream_ptr()))
        return rows


class DevicePrioritizedReplay(DeviceReplay):
    """Prioritized replay over the same ring: tianshou 1.0 ``PrioritizedReplayBuffer(alpha, beta, weight_norm)``,
    restated (PARITY UNPINNED: tianshou is not a dependency; tests/per_reference.py ``PrioritizedRingReference`` is the
    float64 restatement the tests hold the kernels to).

    * one fp64 sum tree per ring slot, leaves = cells ``episode * N + agent`` holding ``p^alpha``
      (``csrc/replay_per.cu``); ``max_prio = min_prio = 1`` at construction, eps = float32 machine epsilon;
    * ``begin_round`` gives every transition of the new round ``max_prio^alpha`` and every other cell 0;
    * ``sample_indices`` draws proportionally to priority over the usable rounds of ``DeviceReplay``;
    * ``gather`` adds ``weight = (leaf / min_prio)^(-beta)`` (divided by its batch maximum with ``weight_norm``), fp32;
    * ``update_weight`` sets the sampled leaves to ``(|td| + eps)^alpha`` (last occurrence wins) and raises
      ``max_prio`` / lowers ``min_prio`` with ``|td| + eps``.

    Everything runs on the caller's stream; after the first ``sample_indices`` no method synchronises with the host.
    Differences from tianshou's numpy code: the leaf and ``|td| + eps`` are evaluated in fp64 (tianshou rounds them to
    float32 before storing them in its float64 tree), and a leaf of priority 0 is never sampled."""

    def __init__(self, n_episodes: int, n_nodes: int, ring_rounds: int, alpha: float, beta: float,
                 weight_norm: bool = True, device="cuda", seed: int = 0):
        if not alpha > 0.0:
            raise ValueError(f"alpha must be > 0 (got {alpha})")
        if not beta >= 0.0:
            raise ValueError(f"beta must be >= 0 (got {beta})")
        super().__init__(n_episodes, n_nodes, ring_rounds, device=device, seed=seed)
        self.alpha, self.beta, self.weight_norm = float(alpha), float(beta), bool(weight_norm)
        self.eps = float(np.finfo(np.float32).eps)
        size = int(self.lib.mls_per_tree_size(self.B * self.N))
        self.tree = torch.zeros(self.R, size, dtype=torch.float64, device=self.device)   # [slot][leaves .. root]
        self.prio = torch.ones(2, dtype=torch.float64, device=self.device)               # max_prio, min_prio

    def set_beta(self, beta: float) -> None:
        if not beta >= 0.0:
            raise ValueError(f"beta must be >= 0 (got {beta})")
        self.beta = float(beta)

    def begin_round(self, obs: torch.Tensor, active: torch.Tensor):
        super().begin_round(obs, active)
        slot = self._pending
        _lib.check(self.lib.mls_per_build(self.flags[slot].data_ptr(), self.B, self.N, self.prio.data_ptr(), self.alpha,
                                          self.tree[slot].data_ptr(), _lib.current_stream_ptr()))

    def sample_indices(self, batch_size: int, n_step: int):
        """Proportional to priority over the stored transitions of the usable rounds (same rule and errors as
        ``DeviceReplay.sample_indices``).  -> (ring round, episode, agent) int32 tensors [M]."""
        first, usable = self._usable_rounds(n_step)
        M = int(batch_size)
        u = torch.rand(M, device=self.device, generator=self.gen, dtype=torch.float64)
        rho, ep, agent = (torch.empty(M, dtype=torch.int32, device=self.device) for _ in range(3))
        _lib.check(self.lib.mls_per_sample(self.tree.data_ptr(), self.R, self.B, self.N, first, usable, u.data_ptr(), M,
                                           rho.data_ptr(), ep.data_ptr(), agent.data_ptr(), None, _lib.current_stream_ptr()))
        return rho, ep, agent

    def _weights(self, rho, ep, agent):
        """Importance weights of (ring round, episode, agent) triples: (leaf / min_prio)^(-beta), normalised by the
        batch maximum with ``weight_norm``.  fp32 [M]."""
        leaf = self.tree[rho.long(), ep.long() * self.N + agent.long()]
        w = (leaf / self.prio[1]).pow(-self.beta)
        if self.weight_norm:
            w = w / w.max()
        return w.to(torch.float32)

    def gather(self, rho, ep, agent, n_step: int, gamma: float):
        """``DeviceReplay.gather`` plus ``weight`` (fp32 [M], see ``_weights``)."""
        out = super().gather(rho, ep, agent, n_step, gamma)
        out["weight"] = self._weights(rho, ep, agent)
        return out

    def update_weight(self, index, new_weight: torch.Tensor):
        """tianshou ``update_weight(index, new_weight)`` with index = the (ring round, episode, agent) triple of
        ``sample_indices`` and new_weight the TD errors ``DQNPolicy.learn`` leaves in ``batch.weight``."""
        rho, ep, agent = (t.to(torch.int32).contiguous() for t in index)
        td = new_weight.detach().to(torch.float32).contiguous()
        if td.dim() != 1 or any(t.shape != td.shape for t in (rho, ep, agent)):
            raise ValueError("update_weight needs one TD error per sampled (round, episode, agent)")
        _lib.check(self.lib.mls_per_update(self.tree.data_ptr(), self.R, self.B, self.N, rho.data_ptr(), ep.data_ptr(),
                                           agent.data_ptr(), td.data_ptr(), int(td.shape[0]), self.alpha, self.eps,
                                           self.prio.data_ptr(), self.prio[1:].data_ptr(), _lib.current_stream_ptr()))
