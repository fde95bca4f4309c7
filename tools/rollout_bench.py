"""BASELINE.json configs[3] (SURVEY section 8d config 4, rows f1 / f2):

  rollout = unroll_length (20) x [ intention-network policy forward (ppo_imitation/intention_policy_network.py:20-105:
  Encoder 795->256->128->(64, 64) with ReLU + LayerNorm, reparameterise, Decoder 296->128->256->60, tanh-normal sample,
  obs normalised by the running statistics) + the fused env step (vnl_step_autoreset) ], 8192 envs per GPU,
  random-init weights (there is no checkpoint).

  POLICY=kernel (default): the repo's tcgen05 policy kernel (vnl_policy_forward, one launch, row f1), normal draws
  pre-generated for the whole unroll (the caller owns the RNG stream, like the reference's key argument);
  POLICY=torch: the same network through torch / cuBLAS (library kernels, ~25 launches) -- the comparison line.
  GRAPH=1: the packaged loop (rollout.Rollout); there AUTORESET=first|resample (first) selects how finished episodes restart
  (brax's first-state restore, or a fresh draw of clip, start frame and noise on the device: DESIGN §3h).

Also times the PPO gradient all-reduce message (policy 341 k + value 1.289 M fp32 parameters = 6.5 MB,
ppo_imitation/train.py:251-253) over NCCL when launched under torchrun.

    python tools/rollout_bench.py                                  # 1 GPU
    python -m torch.distributed.run --nproc-per-node N tools/rollout_bench.py"""
import importlib
import json
import os
import sys

import numpy as np
import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (workload builders)


class MLP(nn.Module):
    def __init__(self, sizes, final_act):
        super().__init__()
        layers = []
        for i in range(len(sizes) - 1):
            layers.append(nn.Linear(sizes[i], sizes[i + 1]))
            if i < len(sizes) - 2 or final_act:
                layers += [nn.ReLU(), nn.LayerNorm(sizes[i + 1])]
        self.net = nn.Sequential(*layers)

    def forward(self, x):
        return self.net(x)


class IntentionPolicy(nn.Module):
    """Encoder(traj) -> (mean, logvar) -> z; Decoder([z, obs]) -> 2 * action_size logits (configs/train_config.yaml:15-17)."""

    def __init__(self, traj_size, obs_size, nu, latents=64, enc=(256, 128), dec=(128, 256)):
        super().__init__()
        self.enc = MLP([traj_size, *enc], True)
        self.mean = nn.Linear(enc[-1], latents)
        self.logvar = nn.Linear(enc[-1], latents)
        self.dec = MLP([latents + obs_size, *dec, 2 * nu], False)

    def forward(self, traj, obs):
        h = self.enc(traj)
        mean, logvar = self.mean(h), self.logvar(h)
        z = mean + torch.randn_like(mean) * torch.exp(0.5 * logvar)
        logits = self.dec(torch.cat([z, obs], dim=-1))
        loc, scale = logits.chunk(2, dim=-1)
        scale = torch.nn.functional.softplus(scale) + 1e-3
        return torch.tanh(loc + scale * torch.randn_like(loc))  # NormalTanhDistribution sample (ppo_networks.py:45-83)


def main():
    sh = importlib.import_module("vnl-brax-imitation_b200.sharding")
    rank, local_rank, world = sh.env_info()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        sh.init_process_group("nccl")
    B, unroll, reps = int(os.environ.get("ENVS", 8192)), 20, int(os.environ.get("REPS", 3))
    env = bench.make_env("rodent", str(dev))
    eng = env.engine
    qpos, qvel, start = bench.workload_draws("rodent", env, B * world, *sh.shard_range(B * world, rank, world))
    s0 = env.reset_from(qpos, qvel, start)
    first, first_obs = dict(s0.pipeline_state), s0.obs
    torch.manual_seed(rank)
    which = os.environ.get("POLICY", "kernel")
    autoreset = os.environ.get("AUTORESET", "first")  # GRAPH=1 only: "resample" restarts finished episodes from fresh draws
    if which == "torch":
        policy = IntentionPolicy(eng.traj_size, eng.obs_size, env.action_size).to(dev).eval()
    else:
        pol = importlib.import_module("vnl-brax-imitation_b200.policy")
        params = pol.init_params(np.random.default_rng(rank), pol.param_shapes(eng.traj_size, eng.obs_size, env.action_size))
        kpol = pol.IntentionPolicy(params, str(dev), torch.zeros(eng.obs_size), torch.ones(eng.obs_size))
        pout = kpol.alloc_outputs(B)
        gen = torch.Generator(device=dev).manual_seed(rank)
        eps_z = torch.randn(unroll, B, kpol.latent, device=dev, generator=gen)
        eps_a = torch.randn(unroll, B, env.action_size, device=dev, generator=gen)
    if os.environ.get("GRAPH") == "1" and which != "torch":
        # the packaged loop: rollout.Rollout = generate_unroll over vnl_policy_forward + vnl_step_training (Episode + AutoReset
        # wrappers fused, episode_length 150), 2 x 20 launches replayed as one CUDA graph, draws refilled per unroll
        ro = importlib.import_module("vnl-brax-imitation_b200.rollout").Rollout(env, kpol, s0, unroll, 150.0, use_graph=True,
                                                                                  autoreset=autoreset, env_offset=B * rank)
        stats = importlib.import_module("vnl-brax-imitation_b200.normalizer").RunningStatistics(eng.obs_size, str(dev))
        kpol.set_normalizer(stats.mean, stats.std)  # shared tensors: every update is seen by the next policy launch
        stats.update(ro.generate_unroll(eps_z, eps_a)["observation"])
        torch.cuda.synchronize()
        sh.barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(reps):
            ro.eps_z.normal_(generator=gen)
            ro.eps_a.normal_(generator=gen)
            stats.update(ro.generate_unroll()["observation"])  # running_statistics.update + its psum (train.py:330-334)
        g1.record()
        torch.cuda.synchronize()
        ms = sh.reduce_scalars(dict(ms=g0.elapsed_time(g1)), op="max", device=dev)["ms"]
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
            dist.destroy_process_group()
        if rank == 0:
            print(json.dumps({"config": "rodent PPO rollout (rollout.Rollout, CUDA graph of 2 x %d launches; draws generated and the obs normaliser updated + all-reduced inside the timed region): %d envs/GPU" % (unroll, B),
                              "autoreset": autoreset, "n_gpus": world, "rollout_env_steps_per_s": world * B * unroll * reps / (ms * 1e-3), "ms_per_unroll": ms / reps}), flush=True)
        return
    a_st = {k: v.clone() for k, v in first.items()}
    a_st["cur_frame"], a_st["sub_clip_frame"] = s0.info["cur_frame"].clone(), s0.info["sub_clip_frame"].clone()
    b_st, out = eng.alloc_state(B), eng.alloc_outputs(B)
    out["obs"].copy_(s0.obs); out["traj"].copy_(s0.info["traj"])
    mean_o, std_o = torch.zeros(eng.obs_size, device=dev), torch.ones(eng.obs_size, device=dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    t_pol = t_env = 0.0

    def unroll_once(timed):
        nonlocal a_st, b_st, t_pol, t_env
        for t in range(unroll):
            e0, e1, e2 = ev(), ev(), ev()
            e0.record()
            if which == "torch":
                with torch.no_grad():
                    act = policy(out["traj"], (out["obs"] - mean_o) / std_o).contiguous()  # obs only is normalised
            else:
                act, _ = kpol(out["traj"], out["obs"], eps_z[t], eps_a[t], out=pout)
            e1.record()
            eng.step_autoreset(a_st, act, b_st, out, first, first_obs)
            e2.record()
            a_st, b_st = b_st, a_st
            if timed:
                marks.append((e0, e1, e2))

    marks = []
    unroll_once(False)
    torch.cuda.synchronize()
    sh.barrier()
    w0, w1 = ev(), ev()
    w0.record()
    for _ in range(reps):
        unroll_once(True)
    w1.record()
    torch.cuda.synchronize()
    ms = sh.reduce_scalars(dict(ms=w0.elapsed_time(w1)), op="max", device=dev)["ms"]
    t_pol = float(np.mean([a.elapsed_time(b) for a, b, _ in marks]))
    t_env = float(np.mean([b.elapsed_time(c) for _, b, c in marks]))
    res = {"config": "rodent PPO rollout: %d envs/GPU x unroll %d, intention network forward (%s, random init) + fused env step" % (
               B, unroll, "torch/cuBLAS" if which == "torch" else "vnl_policy_forward tcgen05 kernel"), "policy": which,
           "n_gpus": world, "rollout_env_steps_per_s": world * B * unroll * reps / (ms * 1e-3), "ms_per_unroll": ms / reps,
           "policy_forward_ms": t_pol, "env_step_ms": t_env, "policy_share": t_pol / (t_pol + t_env)}
    # gradient all-reduce message of one minibatch update (6.5 MB fp32)
    n_grad = 341_000 + 1_289_000
    g = torch.randn(n_grad, device=dev)
    if world > 1:
        import torch.distributed as dist
        for _ in range(5):
            dist.all_reduce(g)
        torch.cuda.synchronize()
        a0, a1 = ev(), ev()
        a0.record()
        for _ in range(50):
            dist.all_reduce(g)
        a1.record()
        torch.cuda.synchronize()
        res["grad_allreduce_us"] = sh.reduce_scalars(dict(us=a0.elapsed_time(a1) / 50 * 1e3), op="max", device=dev)["us"]
        res["grad_allreduce_bytes"] = n_grad * 4
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
