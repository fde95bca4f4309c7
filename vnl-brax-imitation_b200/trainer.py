"""`training_step` of the reference (ppo_imitation/train.py:296-349) on the GPU: rollout -> normaliser update -> SGD phase.

    (state, _), data = scan(generate_unroll, ...)                      rollout.Rollout (policy kernel + fused env step, CUDA graph)
    normalizer_params = running_statistics.update(..., pmap_axis_name)  normalizer.RunningStatistics (one pass + one all-reduce)
    for _ in range(num_updates_per_batch):                              sgd_step (train.py:270-294)
        permutation of the env axis, reshape to num_minibatches
        for each minibatch: gradient_update_fn(loss, adam, pmean)       learner.PPOLearner.update (tcgen05 TF32 GEMMs + row kernels)
    policy <- new parameters                                            policy.load_params (same device blob: captured graphs keep working)

The transition buffers stay on the device from the env kernel to the loss: a minibatch is an index list over the env axis
(`vnl_gather_rows`, which also pads traj rows 795 -> 796 floats for TMA).  One minibatch update (gathers + ~80 launches, the
gradient exchange, Adam) is captured once into CUDA graphs (collective-free: with a process group the NCCL all-reduce runs eagerly
between the gradient graph and the Adam graph) and replayed with fresh indices / noise.  torch = memory, streams,
RNG for the noise operands and `torch.distributed`; no torch math on the data path, no CPU fallback.
"""
from __future__ import annotations

from typing import Dict

from . import learner as lrn
from . import sharding
from . import train_kernels as tk


class Trainer:
    def __init__(self, env, policy, learner: "lrn.PPOLearner", rollout, stats, num_minibatches: int, num_updates_per_batch: int,
                 use_graph: bool = True, seed: int = 0, accumulate_metrics: bool = False):
        """`accumulate_metrics`: sum the loss metrics of every minibatch update on the device (`vnl_metrics_accumulate`, one 8-float
        launch per update, inside the captured gradient graph); `epoch_metrics()` returns their mean."""
        import torch

        self.torch = t = torch
        self.env, self.policy, self.learner, self.rollout, self.stats = env, policy, learner, rollout, stats
        self.B, self.T = rollout.B, rollout.T
        if self.B % num_minibatches:
            raise ValueError("num_envs must be divisible by num_minibatches")
        self.Bm = self.B // num_minibatches
        if (learner.T, learner.Bm) != (self.T, self.Bm):
            raise ValueError("learner was built for another minibatch shape")
        self.num_minibatches, self.num_updates = int(num_minibatches), int(num_updates_per_batch)
        dev = learner.device
        L = learner
        f = lambda *s: t.zeros(*s, dtype=t.float32, device=dev)
        R = self.T * self.Bm
        # static minibatch operands (graph-captured addresses)
        self.idx = t.zeros(self.Bm, dtype=t.int32, device=dev)
        self.eps = f(R * (L.L + L.nu))  # both noise operands of a minibatch in one buffer: one generator launch per minibatch
        self.mb = dict(traj=f(R, L.ld_traj), observation=f(R, L.obs), next_observation_last=f(self.Bm, L.obs), reward=f(R), discount=f(R),
                       truncation=f(R), log_prob=f(R), raw_action=f(R, L.nu), eps_z=self.eps[:R * L.L].view(R, L.L),
                       eps_ent=self.eps[R * L.L:].view(R, L.nu))
        import ctypes
        self._scalar_keys = ("reward", "discount", "truncation", "log_prob")
        self._sdst = (ctypes.c_void_p * 4)(*[self.mb[k].data_ptr() for k in self._scalar_keys])
        self.gen = t.Generator(device=dev).manual_seed(seed)
        self.use_graph, self.graph = bool(use_graph), None
        self.discount_buf = f(self.T, self.B)
        self.env_steps = 0
        self.sgd_launches = 0
        self.accumulate_metrics = bool(accumulate_metrics)
        self.metric_sum = f(8) if self.accumulate_metrics else None
        self._acc_updates0 = 0  # learner.updates when the sum was last reset

    # ---- one minibatch ----------------------------------------------------------------------------------------------------
    def _gather(self, tr):
        """`convert_data` (train.py:279-283) for one minibatch: rows of the time-major transition buffers picked by self.idx."""
        L_, st = tk.lib(), tk.stream(self.idx)
        T, B, Bm, mb = self.T, self.B, self.Bm, self.mb
        g = lambda src, width, dst, ld, T_=T: tk.check(L_.vnl_gather_rows(src.data_ptr(), T_, B, width, self.idx.data_ptr(), Bm, dst.data_ptr(), ld, st), "vnl_gather_rows")
        lr = self.learner
        g(tr["state_extras_traj_in"], lr.traj, mb["traj"], lr.ld_traj)
        g(tr["observation"], lr.obs, mb["observation"], lr.obs)
        g(tr["next_observation"][T - 1:T], lr.obs, mb["next_observation_last"], lr.obs, 1)
        g(tr["policy_extras"]["raw_action"], lr.nu, mb["raw_action"], lr.nu)
        import ctypes
        srcs = (tr["reward"], self.discount_buf, tr["state_extras"]["truncation"], tr["policy_extras"]["log_prob"])  # order of _scalar_keys
        for s_ in srcs:
            assert s_.is_contiguous() and s_.shape == (T, B) and s_.dtype == self.torch.float32
        tk.check(L_.vnl_gather_scalars(4, (ctypes.c_void_p * 4)(*[s_.data_ptr() for s_ in srcs]), self._sdst, T, B, self.idx.data_ptr(), Bm, st),
                 "vnl_gather_scalars")
        self.sgd_launches += 5

    def _accumulate(self):
        """metric_sum += this update's metrics row (enqueued right after loss_and_grads, on the same stream)."""
        m = self.learner.ws["metrics"]
        tk.check(tk.lib().vnl_metrics_accumulate(m.data_ptr(), m.numel(), self.metric_sum.data_ptr(), tk.stream(m)), "vnl_metrics_accumulate")
        self.sgd_launches += 1

    def _grads(self, tr):
        """The update up to the gradient exchange: gather, loss + gradients, and the metric accumulation when enabled."""
        n0 = self.learner.launches
        self._gather(tr)
        self.learner.loss_and_grads(self.mb)
        if self.accumulate_metrics:
            self._accumulate()
        self.sgd_launches += self.learner.launches - n0

    def _adam(self, scale: float):
        n0 = self.learner.launches
        self.learner.apply_gradients(scale)
        self.sgd_launches += self.learner.launches - n0

    def _minibatch(self, tr):
        """One eager update: gradients, their exchange over the process group (if any), Adam."""
        self._grads(tr)
        self._adam(lrn.all_reduce_gradients(self.learner.grads))

    def sgd_phase(self, tr) -> None:
        """num_updates_per_batch x num_minibatches gradient updates on the unroll `tr` (train.py:336-341).  Graph mode captures the
        update once: one graph of gradients + Adam on one rank; with a process group a graph of the gradients, the all-reduce eagerly
        (the graphs never contain a collective, see tk.capture), then a graph of Adam."""
        t = self.torch
        lr = self.learner
        dist = sharding.group()
        self.discount_buf.copy_(tr["discount"])  # `1 - done` view materialised once per unroll
        # the policy's INPUT trajectory of step t is traj[t] (acting.py:47: state.info["traj"]), i.e. rollout.traj[:T]
        tr = dict(tr, state_extras_traj_in=self.rollout.traj[:self.T])
        for _ in range(self.num_updates):
            perm = t.randperm(self.B, device=self.idx.device, generator=self.gen).to(t.int32)
            for mbi in range(self.num_minibatches):
                self.idx.copy_(perm[mbi * self.Bm:(mbi + 1) * self.Bm])
                self.eps.normal_(generator=self.gen)
                if not self.use_graph:
                    self._minibatch(tr)
                    continue
                if self.graph is None:
                    n0, l0 = lr.updates, self.sgd_launches

                    def warmup():  # a real update of this minibatch
                        self._minibatch(tr)
                        self._launches_per_update = self.sgd_launches - l0  # kernels one replay of the captured update launches
                    if dist is None:
                        fns = (lambda: (self._grads(tr), self._adam(1.0)),)
                    else:
                        fns = (lambda: self._grads(tr), lambda: self._adam(1.0 / dist.get_world_size()))
                    self.graph = tk.capture(self.idx.device, warmup, *fns)
                    # the warm-up was one update; the capture passes went through the host-side counters without executing
                    lr.updates, self.sgd_launches = n0 + 1, l0 + self._launches_per_update
                    continue  # this minibatch was the warm-up run
                self.graph[0].replay()
                if dist is not None:
                    lrn.all_reduce_gradients(lr.grads)  # lax.pmean: one 6.5 MB SUM all-reduce; its 1 / world is in the Adam graph
                    self.graph[1].replay()
                lr.updates += 1  # host-side counter (the device-side step counter advanced inside the graph)
                self.sgd_launches += self._launches_per_update

    def training_step(self) -> Dict[str, float]:
        """One `training_step`: unroll, normaliser update, SGD phase, policy refresh.  Returns the last minibatch's loss metrics."""
        ro = self.rollout
        ro.eps_z.normal_(generator=self.gen)
        ro.eps_a.normal_(generator=self.gen)
        tr = ro.generate_unroll()
        self.stats.update(tr["observation"])  # running_statistics.update with its psum (train.py:330-334)
        self.learner.set_normalizer(self.stats.mean, self.stats.std)
        self.sgd_phase(tr)
        self.policy.load_params(self.learner.policy_params())
        self.env_steps += self.B * self.T
        return self.learner.metrics_dict()

    def epoch_metrics(self, reset: bool = True) -> Dict[str, float]:
        """Mean of the loss metrics over every minibatch update since the last reset (brax `training_epoch`:
        `tree_map(jnp.mean, loss_metrics)`), named as learner.metrics_dict names them.  Needs `accumulate_metrics=True`."""
        if not self.accumulate_metrics:
            raise RuntimeError("epoch_metrics needs a Trainer built with accumulate_metrics=True")
        n = self.learner.updates - self._acc_updates0
        out = self.learner.metrics_dict(self.metric_sum / max(n, 1))
        if reset:
            self.metric_sum.zero_()
            self._acc_updates0 = self.learner.updates
        return out

    # ---- checkpoint ---------------------------------------------------------------------------------------------------------
    def state_dict(self) -> Dict[str, object]:
        """This rank's host-side training state: the noise generator and the counters (the device buffers live in the learner,
        the normaliser and the rollout)."""
        return {"gen": self.gen.get_state().numpy().copy(), "env_steps": self.env_steps, "updates": self.learner.updates}

    def load_state_dict(self, sd) -> None:
        t = self.torch
        self.gen.set_state(t.as_tensor(sd["gen"], dtype=t.uint8).cpu())
        self.env_steps = int(sd["env_steps"])
        self.learner.updates = int(sd["updates"])
        self._acc_updates0 = self.learner.updates
        if self.metric_sum is not None:
            self.metric_sum.zero_()
