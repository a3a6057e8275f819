"""Off-policy training loop at batched scale.

Reference: tianshou ``OffpolicyTrainer`` as configured in l_dgn.py:246-261 / hl_dgn.py (``policy, train_collector,
test_collector, max_epoch, step_per_epoch, step_per_collect, episode_per_test, batch_size, train_fn, test_fn,
update_per_step, test_in_train=False, save_best_fn, logger``).  Per epoch: until ``step_per_epoch`` agent transitions
have been collected -- ``train_fn(epoch, env_step)``, ``train_collector.collect(n_step=step_per_collect)``, then
``round(update_per_step * collected)`` calls of ``policy.update(batch_size, buffer)``; after the epoch
``test_fn(epoch, env_step)`` and ``test_collector.collect(n_episode=episode_per_test)``; the best mean test return
triggers ``save_best_fn(policy)``.

On several GPUs every rank runs this loop on its own episodes; ``policy.policy.grad_sync`` (data_parallel.GradSync)
sums the gradients with one NCCL all-reduce per update, so all ranks hold identical weights throughout.
"""
from __future__ import annotations

import time


class OffpolicyTrainer:
    def __init__(self, policy, train_collector, test_collector=None, max_epoch: int = 1, step_per_epoch: int = 1,
                 step_per_collect: int = 1, episode_per_test: int = 1, batch_size: int = 64, update_per_step: float = 1.0,
                 train_fn=None, test_fn=None, stop_fn=None, save_best_fn=None, logger=None, test_in_train: bool = False,
                 max_update_per_collect: int | None = None, verbose: bool = False, **kwargs):
        self.policy, self.train_collector, self.test_collector = policy, train_collector, test_collector
        self.max_epoch, self.step_per_epoch, self.step_per_collect = int(max_epoch), int(step_per_epoch), int(step_per_collect)
        self.episode_per_test, self.batch_size, self.update_per_step = int(episode_per_test), int(batch_size), float(update_per_step)
        self.train_fn, self.test_fn, self.stop_fn, self.save_best_fn = train_fn, test_fn, stop_fn, save_best_fn
        self.logger, self.verbose = logger, verbose
        # at batched scale one collect() returns hundreds of thousands of transitions: cap the updates per collect
        self.max_update_per_collect = max_update_per_collect
        self.env_step = self.gradient_step = 0
        self.best_reward, self.best_epoch = float("-inf"), 0
        self.last_loss = None

    def _sub_policy(self):
        return getattr(self.policy, "policy", self.policy)

    def _test(self, epoch):
        if self.test_collector is None:
            return None
        if self.test_fn:
            self.test_fn(epoch, self.env_step)
        self.test_collector.reset_env()
        res = self.test_collector.collect(n_episode=self.episode_per_test)
        rew = res.returns_stat.mean if res.returns_stat is not None else float("-inf")
        if rew > self.best_reward:
            self.best_reward, self.best_epoch = rew, epoch
            if self.save_best_fn:
                self.save_best_fn(self.policy)
        return res

    def run(self) -> dict:
        start = time.time()
        buffer = self.train_collector.buffer
        if buffer is None:
            raise ValueError("the train collector needs a replay buffer (buffer=DeviceReplay(...))")
        sub = self._sub_policy()
        test_result = self._test(0)
        for epoch in range(1, self.max_epoch + 1):
            epoch_steps = 0
            while epoch_steps < self.step_per_epoch:
                if self.train_fn:
                    self.train_fn(epoch, self.env_step)
                res = self.train_collector.collect(n_step=self.step_per_collect)
                self.env_step += res.n_collected_steps
                epoch_steps += res.n_collected_steps
                n_upd = round(self.update_per_step * res.n_collected_steps)
                if self.max_update_per_collect is not None:
                    n_upd = min(n_upd, self.max_update_per_collect)
                for _ in range(n_upd):
                    if buffer.head <= sub._n_step:
                        break
                    out = self.policy.update(self.batch_size, buffer)
                    self.last_loss = out["loss"]
                    self.gradient_step += 1
            test_result = self._test(epoch)
            if self.verbose:
                print(f"epoch {epoch}: env_step {self.env_step} gradient_step {self.gradient_step} "
                      f"loss {float(self.last_loss) if self.last_loss is not None else float('nan'):.5f} best_reward {self.best_reward:.4f}")
            if self.stop_fn and self.stop_fn(self.best_reward):
                break
        return {"duration": time.time() - start, "env_step": self.env_step, "gradient_step": self.gradient_step,
                "best_reward": self.best_reward, "best_epoch": self.best_epoch,
                "loss": float(self.last_loss) if self.last_loss is not None else None, "test_result": test_result}
