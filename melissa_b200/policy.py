"""Policy and collector surfaces of the rollout / training path, shaped like the reference's.

Reference:
* tianshou ``DQNPolicy`` (``forward / compute_q_value / exploration_noise / set_eps / sync_weight / process_fn /
  learn / update``) as constructed in l_dgn.py:69-76 (``DQNPolicy(model, optim, discount_factor, estimation_step,
  target_update_freq, action_space)``) and ``DGNPolicy.learn`` (policies/dgn.py:22-71, the sum-of-Q loss of the "R"
  scripts);
* ``MultiAgentSharedPolicy.forward / exploration_noise / learn``
  (policies/multi_agent_managers/shared_policy.py:81-216): ``forward(batch, state) -> Batch(act, state, out,
  state_dict)`` with ``batch.obs.{agent_id, obs, mask}``;
* ``MultiAgentCollector(agents_num=, policy=, env=, buffer=, exploration_noise=)`` and
  ``collect(n_step | n_episode, random, render, no_grad)`` (collectors/multi_agent_collector.py:31-353) returning
  ``CollectStatsWithInfo`` (collectors/collector.py:15-36).

tianshou itself is not importable here, so ``Batch`` is a small attribute container with the handful of operations
those call sites use.  The Q-network forward, the action selection and the environment round are CUDA kernels; the
loss / backward of ``learn`` is torch autograd over ``networks/autograd.py``; these classes sequence them.
"""
from __future__ import annotations

import time
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _lib
from .batched_env import BatchedGraphEnv, EpisodeStream, ResetTuplesDevice
from .networks.autograd import q_values
from .networks.common import DGNBase


# ---------------------------------------------------------------------------------------------- Batch
class Batch:
    """The slice of ``tianshou.data.Batch`` the reference's policy / collector code touches: attribute and key access,
    nesting, row indexing, ``update``, ``get``, ``pop``, ``is_empty``, ``cat``."""

    def __init__(self, _dict=None, **kwargs):
        d = dict(_dict) if isinstance(_dict, (dict, Batch)) else {}
        d.update(kwargs)
        for k, v in d.items():
            self.__dict__[k] = Batch(v) if isinstance(v, dict) else v

    def keys(self):
        return self.__dict__.keys()

    def items(self):
        return self.__dict__.items()

    def __iter__(self):
        return iter(self.__dict__)

    def __contains__(self, k):
        return k in self.__dict__

    def __getitem__(self, k):
        if isinstance(k, str):
            return self.__dict__[k]
        out = Batch()
        for name, v in self.__dict__.items():
            if isinstance(v, Batch):
                out.__dict__[name] = v[k] if not v.is_empty() else Batch()
            elif isinstance(v, (np.ndarray, torch.Tensor)):
                out.__dict__[name] = v[k]
            else:
                out.__dict__[name] = v
        return out

    def __setitem__(self, k, v):
        if isinstance(k, str):
            self.__dict__[k] = v
        else:
            raise TypeError("row assignment is not supported by this Batch")

    def __len__(self):
        for v in self.__dict__.values():
            if isinstance(v, Batch):
                if not v.is_empty():
                    return len(v)
            elif isinstance(v, (np.ndarray, torch.Tensor)) and v.ndim > 0:
                return len(v)
        return 0

    def get(self, k, default=None):
        return self.__dict__.get(k, default)

    def pop(self, k, default=None):
        return self.__dict__.pop(k, default)

    def update(self, _dict=None, **kwargs):
        d = dict(_dict) if isinstance(_dict, (dict, Batch)) else {}
        d.update(kwargs)
        for k, v in d.items():
            self.__dict__[k] = Batch(v) if isinstance(v, dict) else v

    def is_empty(self):
        return len(self.__dict__) == 0

    @staticmethod
    def cat(batches):
        batches = [b if isinstance(b, Batch) else Batch(b) for b in batches]
        batches = [b for b in batches if not b.is_empty()]
        out = Batch()
        if not batches:
            return out
        for k in batches[0].keys():
            vs = [b[k] for b in batches]
            if isinstance(vs[0], Batch):
                out.__dict__[k] = Batch.cat(vs)
            elif isinstance(vs[0], torch.Tensor):
                out.__dict__[k] = torch.cat(vs)
            else:
                out.__dict__[k] = np.concatenate([np.asarray(v) for v in vs])
        return out

    def __repr__(self):
        return "Batch(" + ", ".join(f"{k}={type(v).__name__}" for k, v in self.__dict__.items()) + ")"


def to_numpy(x):
    if isinstance(x, torch.Tensor):
        return x.detach().cpu().numpy()
    return np.asarray(x)


def _obs_parts(obs):
    """batch.obs as the collectors build it: Batch(agent_id, obs, mask) (tianshou PettingZooEnv), or bare rows."""
    if isinstance(obs, (Batch, dict)):
        get = obs.get
        return get("obs"), get("mask"), get("agent_id")
    return obs, None, None


# ---------------------------------------------------------------------------------------------- DQN / DGN policy
class DQNPolicy:
    """tianshou ``DQNPolicy`` for the three DGN networks.  ``model`` is one of ``melissa_b200.networks``; ``optim`` a
    ``torch.optim.Optimizer`` or ``melissa_b200.data_parallel.FusedAdam`` (needed for ``learn`` only)."""

    def __init__(self, model: DGNBase, optim=None, discount_factor: float = 0.99, estimation_step: int = 1,
                 target_update_freq: int = 0, reward_normalization: bool = False, is_double: bool = True,
                 clip_loss_grad: bool = False, action_space=None, eps: float = 0.0, seed: int = 9, **kwargs):
        if not 0.0 <= discount_factor <= 1.0:
            raise ValueError("discount factor should be in [0, 1]")
        if estimation_step <= 0:
            raise ValueError("estimation_step should be greater than 0")
        if reward_normalization:
            raise NotImplementedError("reward_normalization is not used by any reference script")
        self.model, self.optim = model, optim
        self.eps, self.seed = float(eps), int(seed)
        self._gamma, self._n_step = float(discount_factor), int(estimation_step)
        self._target = target_update_freq > 0
        self._freq = int(target_update_freq)
        self._iter = 0
        self.is_double, self.clip_loss_grad = bool(is_double), bool(clip_loss_grad)
        self.action_space = action_space
        self.model_old = None
        if self._target:
            self.model_old = model.clone_for_target()
            self.model_old.eval()
        self.grad_sync = None          # melissa_b200.data_parallel.GradSync for multi-GPU training
        self.training = True
        self._calls = 0

    # -------------------------------------------------------------- tianshou plumbing
    def to(self, device):
        self.model.to(device)
        if self.model_old is not None:
            self.model_old.to(device)
        return self

    def train(self, mode: bool = True):
        self.training = mode
        self.model.train(mode)
        return self

    def eval(self):
        return self.train(False)

    def set_eps(self, eps: float) -> None:
        self.eps = float(eps)

    def sync_weight(self) -> None:
        """Copy the online network into the target network (DQNPolicy.sync_weight)."""
        self.model_old.load_state_dict(self.model.state_dict())

    def state_dict(self):
        # reference checkpoints are DQNPolicy.state_dict() (l_dgn.py:221): keys prefixed "model." and "model_old."
        sd = {f"model.{k}": v for k, v in self.model.state_dict().items()}
        if self.model_old is not None:
            sd.update({f"model_old.{k}": v for k, v in self.model_old.state_dict().items()})
        return sd

    def load_state_dict(self, sd):
        self.model.load_state_dict({k[len("model."):]: v for k, v in sd.items() if k.startswith("model.")})
        old = {k[len("model_old."):]: v for k, v in sd.items() if k.startswith("model_old.")}
        if self.model_old is not None and old:
            self.model_old.load_state_dict(old)

    def map_action(self, act):
        return act

    def map_action_inverse(self, act):
        return act

    # -------------------------------------------------------------- acting
    def compute_q_value(self, logits: torch.Tensor, mask):
        """logits + (1 - mask) * (min - max - 1): masked actions fall below every valid one."""
        if mask is None:
            return logits
        m = torch.as_tensor(np.asarray(mask), device=logits.device, dtype=logits.dtype)
        return logits + (1 - m) * (logits.min() - logits.max() - 1.0)

    def forward(self, batch, state=None, model: str = "model", input: str = "obs", mask=None, **kwargs):
        """``batch[input]`` holds agent-observation rows ``[bs, 8N+1]`` (bare, or under ``.obs`` next to ``.mask`` /
        ``.agent_id``) -> ``Batch(logits [bs, 2] tensor, act [bs] int64 ndarray, state)``.  The rows go through the
        CUDA forward (one launch sequence for the whole batch)."""
        net = getattr(self, model)
        obs = batch[input] if isinstance(batch, (Batch, dict)) else batch
        rows, bmask, _ = _obs_parts(obs)
        if mask is None:
            mask = bmask
        logits, hidden = net(rows, state=state, info=batch.get("info") if isinstance(batch, (Batch, dict)) else {})
        q = self.compute_q_value(logits, mask)
        act = to_numpy(q.argmax(dim=1))
        return Batch(logits=logits, act=act, state=hidden)

    __call__ = forward

    def exploration_noise(self, act, batch=None, rng: np.random.Generator | None = None):
        """tianshou: with probability eps the action becomes argmax(rand(2) + mask).  Draws from the global
        ``np.random`` stream like tianshou unless ``rng`` is given.  ``batch`` may be the collector's Batch
        (``batch.obs.mask``) or a bare mask array."""
        if not isinstance(act, np.ndarray) or np.isclose(self.eps, 0.0):
            return act
        mask = None
        if isinstance(batch, (Batch, dict)):
            _, mask, _ = _obs_parts(batch.get("obs"))
        elif batch is not None:
            mask = batch
        bsz = len(act)
        rand_mask = (rng.random(bsz) if rng is not None else np.random.rand(bsz)) < self.eps
        q = rng.random((bsz, 2)) if rng is not None else np.random.rand(bsz, 2)
        if mask is not None:
            q = q + np.asarray(mask)
        act = act.copy()
        act[rand_mask] = q.argmax(axis=1)[rand_mask]
        return act

    # -------------------------------------------------------------- learning
    def _target_q(self, rows: torch.Tensor) -> torch.Tensor:
        """DQNPolicy._target_q: double DQN -- the online net picks the action, the target net values it."""
        with torch.no_grad():
            q_online, _ = self.model(rows)
            if self._target:
                q_old, _ = self.model_old(rows)
                if self.is_double:
                    return q_old.gather(1, q_online.argmax(dim=1, keepdim=True)).squeeze(1)
                return q_old.max(dim=1)[0]
            return q_online.max(dim=1)[0]

    def process_fn(self, batch: Batch, buffer, indices=None) -> Batch:
        """n-step returns of the sampled transitions (tianshou compute_nstep_return).  ``batch`` comes from
        ``DeviceReplay.gather``: the reward sums are already there, only chains that outlive the window bootstrap."""
        boot = batch.boot_round
        ret = batch.returns
        alive = boot >= 0
        if bool(alive.any()):                 # never true with the reference defaults (TTL 4 decisions, n_step 4)
            rows = buffer.rows_at(boot[alive], batch.ep[alive], batch.agent[alive])
            ret = ret.clone()
            ret[alive] += batch.boot_gamma[alive] * self._target_q(rows)
        batch.returns = ret
        return batch

    def _backward(self, loss):
        """zero_grad -> backward -> start the gradient all-reduce (asynchronous: kernels issued next overlap it)."""
        self.optim.zero_grad()
        loss.backward()
        if self.grad_sync is not None:
            self.grad_sync.start()
        self._step_pending = True

    def finish_update(self):
        """Wait for the all-reduce, apply the optimiser step (mean over ranks).  ``learn(..., defer_step=True)`` leaves
        this to the caller so that a rollout round can be issued in between."""
        if not getattr(self, "_step_pending", False):
            return
        if self.grad_sync is not None:
            self.grad_sync.finish()
            if hasattr(self.optim, "flat"):
                self.optim.step(grad_scale=self.grad_sync.grad_scale)
            else:
                for p in self.model.parameters():
                    if p.grad is not None:
                        p.grad.mul_(self.grad_sync.grad_scale)
                self.optim.step()
        else:
            self.optim.step()
        self._step_pending = False
        self._iter += 1

    def _backward_and_step(self, loss, defer_step: bool = False):
        self._backward(loss)
        if not defer_step:
            self.finish_update()

    def learn(self, batch: Batch, **kwargs):
        """tianshou DQNPolicy.learn: q = Q(obs)[act]; loss = mean((returns - q)^2 * weight) (Huber with
        ``clip_loss_grad``); optimiser step; target sync every ``target_update_freq`` iterations."""
        if self.optim is None:
            raise RuntimeError("DQNPolicy.learn needs an optimizer")
        self.finish_update()                      # a deferred step of the previous call
        if self._target and self._iter % self._freq == 0:
            self.sync_weight()
        weight = batch.pop("weight", 1.0)
        q = q_values(self.model, batch.obs)
        q = q.gather(1, batch.act.view(-1, 1)).squeeze(1)
        returns = batch.returns.to(q.dtype).flatten()
        td = returns - q
        if self.clip_loss_grad:
            loss = torch.nn.functional.huber_loss(q.reshape(-1, 1), returns.reshape(-1, 1), reduction="mean")
        else:
            loss = (td.pow(2) * weight).mean()
        batch.weight = td.detach()
        self._backward_and_step(loss, kwargs.get("defer_step", False))
        return {"loss": loss.detach()}

    def update(self, sample_size: int, buffer, **kwargs):
        """tianshou BasePolicy.update: sample -> process_fn -> learn -> post_process_fn (a prioritized replay receives
        the TD errors as new priorities before this returns, so before the next ``begin_round`` can reuse a slot)."""
        rho, ep, agent = buffer.sample_indices(int(sample_size), self._n_step)
        batch = Batch(buffer.gather(rho, ep, agent, self._n_step, self._gamma))
        batch.rho = rho
        batch = self.process_fn(batch, buffer)
        out = self.learn(batch, buffer=buffer, **kwargs)
        if hasattr(buffer, "update_weight"):          # prioritized replay: tianshou's post_process_fn
            buffer.update_weight((rho, ep, agent), batch.weight)
        return out


class DGNPolicy(DQNPolicy):
    """policies/dgn.py:22-71: for every sampled experience the Q-values (at the taken actions) of ALL agents that were
    active in the same environment round are summed and regressed on the experience's n-step return."""

    def learn(self, batch: Batch, buffer=None, **kwargs):
        if self.optim is None:
            raise RuntimeError("DGNPolicy.learn needs an optimizer")
        if buffer is None:
            raise RuntimeError("DGNPolicy.learn needs the replay to look up the round's active observations")
        self.finish_update()
        if self._target and self._iter % self._freq == 0:
            self.sync_weight()
        weight = batch.pop("weight", 1.0)
        rho, ep = batch.rho.long(), batch.ep.long()
        acted = (buffer.flags[rho, ep] & 1).bool()                          # [M, N] active agents of the sampled rounds
        m_idx, a_idx = torch.nonzero(acted, as_tuple=True)
        rows = buffer.rows_at(rho[m_idx].to(torch.int32), ep[m_idx].to(torch.int32), a_idx.to(torch.int32))
        acts = buffer.act[rho[m_idx], ep[m_idx], a_idx].long()
        q = q_values(self.model, rows).gather(1, acts.view(-1, 1)).squeeze(1)
        batch_q = torch.zeros(len(rho), dtype=q.dtype, device=q.device).index_add_(0, m_idx, q)
        returns = batch.returns.to(q.dtype).flatten()
        td = returns - batch_q
        if self.clip_loss_grad:
            loss = torch.nn.functional.huber_loss(batch_q.reshape(-1, 1), returns.reshape(-1, 1), reduction="mean")
        else:
            loss = (td.pow(2) * weight).mean()
        batch.weight = td.detach()
        self._backward_and_step(loss, kwargs.get("defer_step", False))
        return {"loss": loss.detach()}


# ---------------------------------------------------------------------------------------------- shared-policy manager
class MultiAgentSharedPolicy:
    """Parameter sharing (shared_policy.py:14-31): every agent uses the same ``policy``.  ``env`` is anything with
    ``.agents`` (and optionally ``.agent_idx``), or the list of agent names itself."""

    def __init__(self, policy: DQNPolicy, env, **kwargs):
        self.policy = policy
        # tianshou's PettingZooEnv exposes ``agents = possible_agents``; a bare AEC env's ``agents`` is the live subset
        self.agents = list(getattr(env, "possible_agents", None) or getattr(env, "agents", env))
        self.agent_idx = getattr(env, "agent_idx", {a: i for i, a in enumerate(self.agents)})
        self.action_space = getattr(env, "action_space", None)

    def map_action(self, act):
        return act

    def map_action_inverse(self, act):
        return act

    def train(self, mode: bool = True):
        self.policy.train(mode)
        return self

    def eval(self):
        return self.train(False)

    def forward(self, batch, state=None, mask=None, **kwargs):
        """shared_policy.py:93-183.  The reference loops over agent ids and calls the network once per id group; the
        rows are independent, so ONE batched call gives the same actions.  The masked-logit shift
        ``(min - max - 1)`` is taken per id group like the reference's per-group call would."""
        if not isinstance(batch, (Batch, dict)):                              # bare rows: convenience form
            rows = batch
            ids = np.asarray(to_numpy(rows)[:, -1]).astype(np.int64).astype(str)
            batch = Batch(obs=Batch(obs=rows, mask=mask, agent_id=ids))
        rows, bmask, agent_id = _obs_parts(batch["obs"])
        if mask is None:
            mask = bmask
        if mask is not None and np.asarray(mask).ndim == 3:                   # stacked masks: last frame (shared_policy.py:147)
            mask = np.asarray(mask)[:, -1]
        if isinstance(state, Batch) and state.is_empty():
            state = None
        out = self.policy.forward(Batch(obs=rows), state=state, **kwargs)
        logits = out.logits
        act = out.act
        out_dict, state_dict = {}, {}
        if mask is not None and agent_id is not None:
            m = torch.as_tensor(np.asarray(mask), device=logits.device, dtype=logits.dtype)
            ids = np.asarray(agent_id).astype(str)
            q = logits.clone()
            for a in self.agents:
                sel = np.flatnonzero(ids == str(a))
                if len(sel) == 0:
                    out_dict[a], state_dict[a] = Batch(), Batch()
                    continue
                st = torch.as_tensor(sel, device=logits.device)
                lg = logits[st]
                q[st] = lg + (1 - m[st]) * (lg.min() - lg.max() - 1.0)
                out_dict[a] = Batch(logits=lg, act=None, state=None)
                state_dict[a] = Batch()
            act = to_numpy(q.argmax(dim=1))
            for a, o in out_dict.items():
                if not o.is_empty():
                    o.act = act[np.flatnonzero(ids == str(a))]
        holder = Batch(act=act, state=Batch(), logits=logits)
        holder["out"] = out_dict
        holder["state_dict"] = state_dict
        return holder

    __call__ = forward

    def exploration_noise(self, act, batch=None, rng=None):
        """shared_policy.py:81-91 (per agent-id group -> the sub-policy's noise; groups are independent draws)."""
        return self.policy.exploration_noise(act, batch, rng=rng)

    def process_fn(self, batch, buffer, indice=None):
        return self.policy.process_fn(batch, buffer, indice)

    def learn(self, batch, batch_size=None, repeat=None, **kwargs):
        return self.policy.learn(batch, **kwargs)

    def update(self, sample_size, buffer, **kwargs):
        return self.policy.update(sample_size, buffer, **kwargs)


class MultiAgentCollaborativeSharedPolicy(MultiAgentSharedPolicy):
    """collaborative_shared_policy.py: same forward; its process_fn gathers the round's active observations, which
    ``DGNPolicy.learn`` does here straight from the replay ring."""


# ---------------------------------------------------------------------------------------------- collector
@dataclass
class SequenceSummaryStats:
    mean: float
    std: float
    max: float
    min: float

    @classmethod
    def from_sequence(cls, seq):
        a = np.asarray(seq, dtype=np.float64)
        return cls(float(a.mean()), float(a.std()), float(a.max()), float(a.min()))


@dataclass
class CollectStatsWithInfo:
    """Field for field the reference's collect statistics (collectors/collector.py:34, multi_agent_collector.py:339-353)."""
    n_collected_episodes: int = 0
    n_collected_steps: int = 0
    collect_time: float = 0.0
    collect_speed: float = 0.0
    returns: np.ndarray = field(default_factory=lambda: np.array([]))
    returns_stat: SequenceSummaryStats | None = None
    lens: np.ndarray = field(default_factory=lambda: np.array([], dtype=int))
    lens_stat: SequenceSummaryStats | None = None
    info: dict = field(default_factory=dict)


LOGGER_KEYS = ["total_messages_transmitted", "coverage", "messages_sent", "messages_received", "n_neighbours",
               "interested_agents", "coverage_interested_fraction", "coverage_interested_count",
               "uninterested_with_message", "episode_rewards_sum"]


class BatchedCollector:
    """``MultiAgentCollector`` over a :class:`BatchedGraphEnv` (built with ``want_info=True``): same constructor
    keywords (``agents_num=, policy=, env=, buffer=, exploration_noise=``) and ``collect`` signature.  One iteration =
    forward + action selection + one environment round for every episode, on the device; finished episodes restart
    inside the step kernel from ``tuples`` (the reference's vector env resets them one by one): a
    :class:`ResetTuplesDevice` pool, or an :class:`EpisodeStream` that draws a fresh episode on the device for every
    reset.  With ``buffer`` (a
    :class:`melissa_b200.replay.DeviceReplay`) every agent transition of the round is stored, completed by the
    world step's reward exactly as multi_agent_collector.py:240-308 completes it on the agent's next observation."""

    def __init__(self, policy=None, env: BatchedGraphEnv = None, tuples: ResetTuplesDevice | EpisodeStream = None,
                 exploration_noise: bool = False, *, agents_num: int | None = None, buffer=None, **kwargs):
        if policy is None or env is None:
            raise TypeError("BatchedCollector needs policy= and env=")
        if env.info_buf is None:
            raise ValueError("BatchedCollector needs BatchedGraphEnv(..., want_info=True)")
        if agents_num is not None and agents_num != env.N:
            raise ValueError(f"agents_num={agents_num} does not match the environment's {env.N} agents")
        self.masp = policy
        self.policy = policy.policy if isinstance(policy, MultiAgentSharedPolicy) else policy
        self.env, self.buffer = env, buffer
        if tuples is None:                                       # the reference env draws its own episodes (seed 9 + env index)
            from . import reset_chain
            gi, src, inter, scr, _ = reset_chain.episode_pool(9, max(4 * env.B, 64), env.N, len(env.pool))
            tuples = ResetTuplesDevice(gi, src, inter, scr, env.N, env.device, pool_size=len(env.pool))
        self.tuples = tuples
        self.agents_num = env.N
        self.exploration_noise = exploration_noise
        self.collect_step = self.collect_episode = 0
        self.collect_time = 0.0
        self._round = 0
        B, N = env.B, env.N
        self.q = torch.zeros(B, N, 2, dtype=torch.float32, device=env.device)
        self.act = torch.full((B, N), -1, dtype=torch.int8, device=env.device)
        self.feature_errors = torch.zeros(1, dtype=torch.int32, device=env.device)
        self.reset()

    def reset(self, reset_buffer: bool = True, gym_reset_kwargs=None):
        if isinstance(self.tuples, EpisodeStream):
            first = self.tuples                  # every episode, the first ones included, is a fresh device draw
        else:
            if self.tuples.count < self.env.B:
                raise ValueError(f"need at least {self.env.B} reset tuples (one per episode), got {self.tuples.count}")
            first = ResetTuplesDevice.__new__(ResetTuplesDevice)
            first.count = self.env.B
            for k in ("graph_index", "source", "interested", "scripted"):
                setattr(first, k, getattr(self.tuples, k)[: self.env.B])
        self.env.episode.zero_()
        self.env.reset(first)
        self.env.set_recycling(self.tuples)
        self.env.transitions.zero_()

    def reset_env(self, gym_reset_kwargs=None):
        self.reset(reset_buffer=False)

    def iterate(self, eps: float = 0.0, random: bool = False):
        """One collector iteration: policy forward + action selection + environment round, all on the device."""
        env = self.env
        if self.buffer is not None:
            self.buffer.begin_round(env.obs, env.active)
        if random:
            self.act.copy_(torch.randint(0, 2, self.act.shape, device=env.device, dtype=torch.int8))
        else:
            self.policy.model.forward_graphs(env.obs, env.active, eps=eps, philox_seed=self.policy.seed,
                                             philox_offset=self._round, q_out=self.q, act_out=self.act,
                                             discrete_features=True, feature_errors=self.feature_errors, prepared=True)
        env.step_device(self.act)
        if self.buffer is not None:
            self.buffer.end_round(self.act, env.reward, env.terminated)
        self._round += 1

    def collect(self, n_step: int | None = None, n_episode: int | None = None, random: bool = False, render: bool = False,
                no_grad: bool = True, gym_render_kwargs=None) -> CollectStatsWithInfo:
        if (n_step is None) == (n_episode is None):
            raise TypeError("Please specify exactly one of n_step or n_episode")
        env = self.env
        start = time.time()
        t0 = int(env.transitions.item())
        steps = episodes = 0
        returns, lens = [], []
        stats = {k: [] for k in LOGGER_KEYS}
        eps = self.policy.eps if self.exploration_noise else 0.0
        while True:
            self.iterate(eps, random)
            done = env.done.cpu().numpy().astype(bool)
            if done.any():
                inf = env.last_info()                    # describes the round that just ended (before the restart)
                ids = np.flatnonzero(done)
                episodes += len(ids)
                returns.extend(inf["episode_rewards_sum"][ids].tolist())
                lens.extend(inf["num_moves"][ids].tolist())
                for k in LOGGER_KEYS:
                    stats[k].extend(np.asarray(inf[k])[ids].tolist())
            steps = int(env.transitions.item()) - t0
            if (n_step and steps >= n_step) or (n_episode and episodes >= n_episode):
                break
        dt = max(time.time() - start, 1e-9)
        self.collect_step += steps
        self.collect_episode += episodes
        self.collect_time += dt
        return CollectStatsWithInfo(
            n_collected_episodes=episodes, n_collected_steps=steps, collect_time=dt, collect_speed=steps / dt,
            returns=np.array(returns), returns_stat=SequenceSummaryStats.from_sequence(returns) if returns else None,
            lens=np.array(lens, dtype=int), lens_stat=SequenceSummaryStats.from_sequence(lens) if lens else None,
            info={k: SequenceSummaryStats.from_sequence(v) for k, v in stats.items() if v})


MultiAgentCollector = BatchedCollector      # the reference's class name (collectors/multi_agent_collector.py:14)
