"""Stepping an env whose consumer lives on the HOST (numpy policy, logger, another framework).

`HostStepper.step(host_action)` is the host-buffer form of `env.step`: actions come from pinned host memory, obs /
traj / reward / done land in pinned host memory, and the call returns when they are there.  The batch is cut in two at
a wave boundary of the persistent grid (`Engine.resident_envs`): the leading full waves, then the last wave; the
device-to-host copy of the first chunk runs on a second stream while the last wave computes, so only the last wave's
copy is exposed.  The episode handling is
brax's AutoResetWrapper as installed by the reference (`ppo_imitation/train.py:204-214`), fused into the launch
(`vnl_step_autoreset`); the device state ping-pongs between two preallocated buffers, nothing is allocated per step.
"""
from __future__ import annotations

from typing import Dict

from ._lib import STATE_F
from .envs.base import engine_state

HOST_FIELDS = ("obs", "traj", "reward", "done")


class HostStepper:
    """`episode_length` > 0 adds brax's EpisodeWrapper inside the AutoReset (`envs.training.wrap`: info["steps"],
    info["truncation"], done at the episode length), still one fused launch per chunk (`vnl_step_training`)."""

    def __init__(self, env, state0, autoreset: bool = True, chunk: int = 0, episode_length: float = 0.0):
        import torch

        self.torch, self.env, self.eng = torch, env, env.engine
        eng = self.eng
        ps = state0.pipeline_state
        self.B = B = ps["qpos"].shape[0]
        self.first = {k: ps[k].clone() for k in STATE_F}
        self.first_obs = state0.obs.clone()
        self.autoreset = autoreset
        self.bufs = [{k: v.clone() for k, v in engine_state(state0).items()}, eng.alloc_state(B)]
        self.out = eng.alloc_outputs(B)
        self.episode_length = float(episode_length)
        if self.episode_length > 0 and not autoreset:
            raise ValueError("the episode counter is part of the AutoReset wrapping (envs.training.wrap)")
        self.steps = torch.zeros(B, dtype=torch.float32, device=eng.device)
        self.truncation = torch.zeros(B, dtype=torch.float32, device=eng.device)
        self.prev_done = torch.zeros(B, dtype=torch.float32, device=eng.device)
        self.d_action = torch.empty(B, env.action_size, dtype=torch.float32, device=eng.device)
        self.host = {k: torch.empty_like(self.out[k], device="cpu").pin_memory() for k in HOST_FIELDS}
        self.copy_stream = torch.cuda.Stream(device=eng.device)
        if chunk > 0:
            C = int(chunk)
            self.chunks = [(a, min(a + C, B)) for a in range(0, B, C)]
        else:
            # two launches: all the full waves but the last in one (the persistent grid walks them back to back, no kernel
            # boundary in between), then the last wave -- its compute hides the first chunk's copy, only its own copy
            # (the smallest possible) is exposed
            R = max(1, eng.resident_envs)
            head = (B - 1) // R * R
            self.chunks = [(0, head), (head, B)] if head > 0 else [(0, B)]
        self.events = [torch.cuda.Event() for _ in self.chunks]
        cut = lambda d, a, b: {k: v[a:b] for k, v in d.items() if v is not None}
        # contiguous leading-dim views of every buffer, cut once
        self.views = [dict(bufs=[cut(self.bufs[0], a, b), cut(self.bufs[1], a, b)], out=cut(self.out, a, b),
                           first=cut(self.first, a, b), first_obs=self.first_obs[a:b], action=self.d_action[a:b],
                           steps=self.steps[a:b], truncation=self.truncation[a:b], prev_done=self.prev_done[a:b],
                           host={k: self.host[k][a:b] for k in HOST_FIELDS}) for a, b in self.chunks]
        self.flip = 0
        self.h2d_bytes = self.d_action.numel() * 4
        self.d2h_bytes = sum(self.host[k].numel() * 4 for k in HOST_FIELDS)

    @property
    def state(self) -> Dict:
        """The current device state (pipeline-state leaves + frame counters)."""
        return self.bufs[self.flip]

    def step(self, host_action) -> Dict:
        torch, eng = self.torch, self.eng
        main = torch.cuda.current_stream(eng.device)
        self.d_action.copy_(host_action, non_blocking=True)
        src, dst = self.flip, 1 - self.flip
        for v, ev in zip(self.views, self.events):
            if self.episode_length > 0:
                eng.step_training(v["bufs"][src], v["action"], v["bufs"][dst], v["out"], v["first"], v["first_obs"],
                                  v["steps"], v["prev_done"], v["steps"], v["truncation"], self.episode_length)
                v["prev_done"].copy_(v["out"]["done"])  # the next step's `state.done` (same stream, after the launch)
            elif self.autoreset:
                eng.step_autoreset(v["bufs"][src], v["action"], v["bufs"][dst], v["out"], v["first"], v["first_obs"])
            else:
                eng.step(v["bufs"][src], v["action"], v["bufs"][dst], v["out"])
            ev.record(main)
            with torch.cuda.stream(self.copy_stream):
                self.copy_stream.wait_event(ev)
                for k in HOST_FIELDS:
                    v["host"][k].copy_(v["out"][k], non_blocking=True)
        self.flip = dst
        self.copy_stream.synchronize()  # the host consumer needs this step's result before it can pick the next action
        return self.host
