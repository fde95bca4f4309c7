"""The rollout loop around the two kernels: `generate_unroll` / `actor_step` of the reference
(ppo_imitation/acting.py:30-80) for the training-wrapped env (`envs.training.wrap`: AutoResetWrapper(EpisodeWrapper(env)),
ppo_imitation/train.py:204-214).

    for t in range(unroll_length):
        action, extras = policy(state.info["traj"], state.obs, key)      # vnl_policy_forward  (1 launch)
        nstate = env.step(state, action)                                 # vnl_step_training   (1 launch)
        transition[t] = (state.obs, action, nstate.reward, 1 - nstate.done, nstate.obs,
                         extras{log_prob, raw_action, logits}, {truncation, traj} of nstate)

Both kernels write straight into the `[T(+1), B, ...]` transition buffers (each step's output pointers are slices of
them), so collecting the data costs no copies; the 2 T launches are captured once into a CUDA graph and replayed.  The
random draws are operands (`eps_z`, `eps_a`): the caller fills the static draw buffers before every unroll, as the
reference splits a fresh key per step (`acting.py:72-73`).  No CPU fallback: both kernels are required.

`autoreset="resample"` replaces brax's AutoReset (restore the cached first state) by a fresh reset of every finished episode:
new clip, start frame and reset noise, drawn on the device inside the env step (`vnl_step_training_resample`, DESIGN §3h).
"""
from __future__ import annotations

from typing import Dict, Optional

from . import train_kernels as tk


class Rollout:
    def __init__(self, env, policy, first_state, unroll_length: int, episode_length: float, use_graph: bool = True,
                 autoreset: str = "first", seed: int = 0, env_offset: int = 0):
        """`first_state`: the State returned by env.reset(...).  `autoreset="first"`: it is also the state AutoReset restores (brax
        caches `first_pipeline_state` / `first_obs` in info at reset).  `autoreset="resample"`: a finished episode restarts from a
        fresh draw of `env.resample_spec()`'s distribution, keyed by `seed`, the global env index (`env_offset` + row: this
        process's first env in a sharded run) and the env's own reset counter."""
        import torch

        self.torch = t = torch
        self.env, self.eng, self.policy = env, env.engine, policy
        self.T, self.episode_length = int(unroll_length), float(episode_length)
        dev = self.eng.device
        B = self.B = first_state.obs.shape[0]
        T = self.T
        nu, obs, traj = policy.action_size, self.eng.obs_size, self.eng.traj_size
        if (obs, traj) != (policy.obs_size, policy.traj_size):
            raise ValueError("policy and env disagree on obs / traj sizes")
        f = lambda *s: t.zeros(*s, dtype=t.float32, device=dev)
        if autoreset not in ("first", "resample"):
            raise ValueError(f"autoreset must be 'first' or 'resample', not {autoreset!r}")
        self.autoreset = autoreset
        self.first = self.first_obs = self.reset_count = None
        if autoreset == "first":
            self.first = {k: v.clone() for k, v in first_state.pipeline_state.items()}
            self.first_obs = first_state.obs.clone()
        else:
            if not hasattr(env, "resample_spec"):
                raise ValueError(f"autoreset='resample': {type(env).__name__} has no resample_spec()")
            self.start_frame_hi, self.noise_scale = env.resample_spec()
            self.seed, self.env_offset = int(seed), int(env_offset)
            # fixed addresses for the captured graph: each env's resets so far (the draw's counter) and the done list
            self.reset_count = t.zeros(B, dtype=t.int32, device=dev)
            self.scratch = t.zeros(B + 1, dtype=t.int32, device=dev)
        # env state ping-pong + episode counters of EpisodeWrapper / AutoResetWrapper
        self.state = [dict({k: v.clone() for k, v in first_state.pipeline_state.items()}, cur_frame=first_state.info["cur_frame"].clone(),
                           sub_clip_frame=first_state.info["sub_clip_frame"].clone()), self.eng.alloc_state(B)]
        if first_state.info.get("clip_idx") is not None:  # multi-clip env: every env keeps tracking its own clip
            self.state[0]["clip_id"] = first_state.info["clip_idx"].clone()
        self.cur = 0
        self.steps, self.done_prev = f(B), f(B)
        # transition buffers (time-major, like `data` after the swapaxes of intention_losses.py:133)
        self.obs, self.traj = f(T + 1, B, obs), f(T + 1, B, traj)
        self.obs[0].copy_(first_state.obs)
        self.traj[0].copy_(first_state.info["traj"])
        self.reward, self.done, self.truncation = f(T, B), f(T, B), f(T, B)
        self.metrics = f(T, B, 7)
        self.action, self.raw_action, self.logits = f(T, B, nu), f(T, B, nu), f(T, B, 2 * nu)
        self.log_prob = f(T, B)
        self.rand_log_prob = f(T, B)
        # static draw buffers: fill before every generate_unroll()
        self.eps_z, self.eps_a = f(T, B, policy.latent), f(T, B, nu)
        self.graph = None
        self.use_graph = use_graph
        self.launches = 0

    # -----------------------------------------------------------------------------------------------------------------
    def _enqueue(self):
        """The 2 T launches of one unroll on the current stream (eager or under capture)."""
        cur = self.cur
        for t in range(self.T):
            pout = {"action": self.action[t], "raw_action": self.raw_action[t], "logits": self.logits[t],
                    "log_prob": self.log_prob[t], "rand_log_prob": self.rand_log_prob[t]}
            self.policy(self.traj[t], self.obs[t], self.eps_z[t], None if self.eps_a is None else self.eps_a[t], out=pout)  # eps_a None: the mode
            out = {"obs": self.obs[t + 1], "traj": self.traj[t + 1], "reward": self.reward[t], "done": self.done[t],
                   "metrics": self.metrics[t]}
            done_in = self.done_prev if t == 0 else self.done[t - 1]
            if self.autoreset == "first":
                self.eng.step_training(self.state[cur], self.action[t], self.state[1 - cur], out, self.first, self.first_obs,
                                       self.steps, done_in, self.steps, self.truncation[t], self.episode_length)
            else:
                self.eng.step_training_resample(self.state[cur], self.action[t], self.state[1 - cur], out, self.steps, done_in, self.steps,
                                                self.truncation[t], self.episode_length, self.reset_count, self.scratch, self.seed,
                                                self.env_offset, self.start_frame_hi, self.noise_scale)
            cur = 1 - cur
        # carry: the next unroll starts from the last state / obs / traj / done
        self.done_prev.copy_(self.done[self.T - 1])
        if cur != self.cur:  # odd T: bring the state back to the buffer the (captured) launches read first
            # (its keys: without a clip index in the first state -- single-clip envs such as the humanoid -- there is no clip_id to restore)
            for k, v in self.state[self.cur].items():
                v.copy_(self.state[cur][k])

    def generate_unroll(self, eps_z=None, eps_a=None) -> Dict[str, "torch.Tensor"]:
        """One unroll; returns views of the transition buffers, named as brax's Transition (acting.py:50-57):
        observation / next_observation [T,B,obs], action [T,B,nu], reward, discount [T,B], policy extras, state extras."""
        if eps_z is not None:
            self.eps_z.copy_(eps_z)
        if eps_a is not None:
            self.eps_a.copy_(eps_a)
        if self.launches and not getattr(self, "_fresh", False):  # the previous unroll's last obs / traj are this one's first
            self.obs[0].copy_(self.obs[self.T])
            self.traj[0].copy_(self.traj[self.T])
        if not self.use_graph:
            self._enqueue()
        else:
            if self.graph is None:
                # the warm-up unroll runs on a snapshot of the carry that is restored after it (the capture executes nothing)
                snap = self._snapshot()
                self.graph, = tk.capture(self.eng.device, lambda: (self._enqueue(), self._restore(snap)), self._enqueue)
                # the graph holds the policy's operand addresses: `load_params` / `set_normalizer` copy into them from now on
                self._captured = (self.policy.blob_dev.data_ptr(), None if self.policy.obs_mean is None else self.policy.obs_mean.data_ptr(),
                                  None if self.policy.obs_std is None else self.policy.obs_std.data_ptr())
                self.policy.pin_operands()
            now = (self.policy.blob_dev.data_ptr(), None if self.policy.obs_mean is None else self.policy.obs_mean.data_ptr(),
                   None if self.policy.obs_std is None else self.policy.obs_std.data_ptr())
            if now != self._captured:  # someone swapped a tensor behind the policy's back: never replay stale addresses
                raise RuntimeError("policy operands moved after the rollout graph was captured")
            self.graph.replay()
        self.launches += 2 * self.T
        self._fresh = False
        return {"observation": self.obs[:self.T], "next_observation": self.obs[1:], "action": self.action, "reward": self.reward,
                "discount": 1.0 - self.done, "policy_extras": {"log_prob": self.log_prob, "raw_action": self.raw_action,
                                                               "logits": self.logits},
                "state_extras": {"truncation": self.truncation, "traj": self.traj[1:]}, "metrics": self.metrics}

    def reset_to(self, first_state) -> None:
        """Start over from a fresh `env.reset(...)` state WITHOUT changing any buffer address (a captured graph stays valid): the
        evaluator resets its envs before every evaluation (acting.py:111-113)."""
        for k, v in first_state.pipeline_state.items():
            if self.first is not None:
                self.first[k].copy_(v)
            self.state[self.cur][k].copy_(v)
        if self.first_obs is not None:
            self.first_obs.copy_(first_state.obs)
        self.state[self.cur]["cur_frame"].copy_(first_state.info["cur_frame"])
        self.state[self.cur]["sub_clip_frame"].copy_(first_state.info["sub_clip_frame"])
        if "clip_id" in self.state[self.cur] and first_state.info.get("clip_idx") is not None:
            self.state[self.cur]["clip_id"].copy_(first_state.info["clip_idx"])
        self.steps.zero_()
        self.done_prev.zero_()
        self.obs[0].copy_(first_state.obs)
        self.traj[0].copy_(first_state.info["traj"])
        self._fresh = True

    # ---- checkpoint --------------------------------------------------------------------------------------------------
    def state_dict(self) -> Dict[str, "np.ndarray"]:
        """The carry into the next unroll, on the host: the env state the captured launches read first ("state/<key>", clip_id only
        where the env has one), the AutoReset state ("first/<key>", "first_obs"; "reset_count" in resample mode), the obs / traj
        the next unroll starts from, the episode step counters and the last step's done flags."""
        carried = self.launches and not getattr(self, "_fresh", False)  # generate_unroll would copy obs[T] / traj[T] to row 0
        h = lambda x: x.detach().cpu().numpy().copy()
        return {k: h(v) for k, v in self._carry(carried).items()}

    def _carry(self, carried=False) -> Dict[str, "torch.Tensor"]:
        out = {"state/" + k: v for k, v in self.state[self.cur].items()}
        if self.autoreset == "first":
            out.update(("first/" + k, v) for k, v in self.first.items())
            out["first_obs"] = self.first_obs
        else:
            out["reset_count"] = self.reset_count
        out.update(obs=self.obs[self.T] if carried else self.obs[0], traj=self.traj[self.T] if carried else self.traj[0], steps=self.steps,
                   done_prev=self.done_prev)
        return out

    def load_state_dict(self, sd) -> None:
        """Copies a state_dict() into the existing buffers, as reset_to does: no address changes, so a captured unroll graph stays
        valid, and the reset kernel does not run."""
        import numpy as np
        t = self.torch
        dst = self._carry()
        if set(dst) != set(sd):
            raise ValueError(f"rollout state keys differ: missing {sorted(set(dst) - set(sd))}, unexpected {sorted(set(sd) - set(dst))}")
        for k, x in dst.items():
            a = np.asarray(sd[k])
            if tuple(a.shape) != tuple(x.shape) or a.dtype != np.dtype(str(x.dtype).replace("torch.", "")):
                raise ValueError(f"rollout state {k}: {a.dtype}{tuple(a.shape)} does not match {x.dtype}{tuple(x.shape)}")
            x.copy_(t.from_numpy(np.ascontiguousarray(a)))
        self._fresh = True  # the next unroll starts from obs[0] / traj[0]

    # -----------------------------------------------------------------------------------------------------------------
    def _snapshot(self):
        s = self.state[self.cur]
        return ({k: v.clone() for k, v in s.items()}, self.steps.clone(), self.done_prev.clone(),
                None if self.reset_count is None else self.reset_count.clone())

    def _restore(self, snap):
        st, steps, done_prev, reset_count = snap
        for k, v in st.items():
            self.state[self.cur][k].copy_(v)
        self.steps.copy_(steps)
        self.done_prev.copy_(done_prev)
        if reset_count is not None:
            self.reset_count.copy_(reset_count)

    @property
    def env_state(self) -> Dict[str, "torch.Tensor"]:
        return self.state[self.cur]
