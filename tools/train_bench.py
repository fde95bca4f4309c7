"""BASELINE.json configs[3] as a whole: the reference's `training_step` (ppo_imitation/train.py:296-349) -- rollout of ENVS envs x
unroll 20 (policy kernel + fused env step), normaliser update, SGD phase of UPDATES x MINIBATCHES minibatch updates (tcgen05 TF32
GEMMs, Adam) with the gradient all-reduce over NCCL at N > 1 -- timed phase by phase with CUDA events, max over ranks.

    python tools/train_bench.py                                             # 1 GPU
    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/train_bench.py
  env: ENVS (8192) MINIBATCHES (32) UPDATES (16) STEPS (2) GRAPH (1) X3 (0)
       ENV=rodent|humanoid (rodent) -- the tracking env; CLIP=standing|moving (standing) -- the humanoid's packaged stand-in clip
       (`envs.humanoid.packaged_humanoid(moving=...)`; the rodent always tracks its packaged clip)
  AUTORESET=first|resample (first) -- how finished training episodes restart: brax's first-state restore, or a fresh draw (DESIGN §3h)
  PROFILE=1 (with GRAPH=0): after the warm-up step, ONE eager minibatch update between cudaProfilerStart / Stop and exit -- the region
  `ncu --profile-from-start off --metrics gpu__time_duration.sum` lists (tools/make_profiles.py summarises the csv)."""
import importlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def build(dev, rank, world, B, unroll, nmb, nup, graph=True, x3=False, env_name="rodent", clip="standing"):
    P = lambda n: importlib.import_module("vnl-brax-imitation_b200." + n)
    sh, trn = P("sharding"), P("train")
    if env_name not in ("rodent", "humanoid") or clip not in ("standing", "moving"):
        raise ValueError("ENV must be rodent or humanoid, CLIP standing or moving")
    if env_name == "humanoid":
        model, ref = P("envs.humanoid").packaged_humanoid(moving=clip == "moving")
        env = P("envs").HumanoidTracking(model=model, reference_clip=ref, device=str(dev))
    else:
        env = bench.make_env("rodent", str(dev))
    qpos, qvel, start = bench.workload_draws(env_name, env, B * world, *sh.shard_range(B * world, rank, world))
    s0 = env.reset_from(qpos, qvel, start)
    # train()'s assembly (the same seeds: identical initial networks on every rank, the trainer's noise seeded by its rank)
    cfg = dict(trn.DEFAULTS, num_envs=B * world, batch_size=B * world // nmb, unroll_length=unroll, num_minibatches=nmb, num_updates_per_batch=nup,
               policy="bf16" if os.environ.get("POLICY") == "bf16" else "3xtf32", autoreset=os.environ.get("AUTORESET", "first"))
    tr = trn.Run(env, cfg, rank=rank, world_size=world, first_state=s0, use_graph=graph, learner_x3=x3, accumulate_metrics=False, evaluate=False).trainer
    return tr


def main():
    sh = importlib.import_module("vnl-brax-imitation_b200.sharding")
    rank, local_rank, world = sh.env_info()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        sh.init_process_group("nccl")
    B, unroll = int(os.environ.get("ENVS", 8192)), 20
    nmb, nup, steps = int(os.environ.get("MINIBATCHES", 32)), int(os.environ.get("UPDATES", 16)), int(os.environ.get("STEPS", 2))
    graph, x3 = os.environ.get("GRAPH", "1") == "1", os.environ.get("X3", "0") == "1"
    env_name, clip = os.environ.get("ENV", "rodent"), os.environ.get("CLIP", "standing")
    tr = build(dev, rank, world, B, unroll, nmb, nup, graph, x3, env_name, clip)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    m = tr.training_step()  # warm-up: graph captures
    torch.cuda.synchronize()
    if os.environ.get("PROFILE") == "1":
        data = tr.rollout.generate_unroll()
        data = dict(data, state_extras_traj_in=tr.rollout.traj[:unroll])
        tr.discount_buf.copy_(data["discount"])
        tr.idx.copy_(torch.randperm(B, device=dev)[:tr.Bm].to(torch.int32))
        tr.eps.normal_(generator=tr.gen)
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        tr._minibatch(data)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        print(json.dumps({"profiled": "one eager minibatch update", "rows": unroll * tr.Bm}), flush=True)
        return
    sh.barrier()
    t_ro = t_sgd = 0.0
    w0, w1 = ev(), ev()
    w0.record()
    for _ in range(steps):
        a, b, c = ev(), ev(), ev()
        a.record()
        tr.rollout.eps_z.normal_(generator=tr.gen); tr.rollout.eps_a.normal_(generator=tr.gen)
        data = tr.rollout.generate_unroll()
        tr.stats.update(data["observation"])
        tr.learner.set_normalizer(tr.stats.mean, tr.stats.std)
        b.record()
        tr.sgd_phase(data)
        tr.policy.load_params(tr.learner.policy_params())
        c.record()
        torch.cuda.synchronize()
        t_ro += a.elapsed_time(b); t_sgd += b.elapsed_time(c)
    w1.record()
    torch.cuda.synchronize()
    m = tr.learner.metrics_dict()
    red = sh.reduce_scalars(dict(ms=w0.elapsed_time(w1), ro=t_ro, sgd=t_sgd), op="max", device=dev)
    what = env_name if env_name == "rodent" else "%s (%s clip)" % (env_name, clip)
    res = {"config": "%s PPO training_step: %d envs/GPU x unroll %d; SGD phase %d updates x %d minibatches of %d rows (%s, %s)" % (
               what, B, unroll, nup, nmb, unroll * B // nmb, "3xTF32" if x3 else "TF32", "CUDA graph per minibatch update" if graph else "eager"),
           "n_gpus": world, "training_env_steps_per_s": world * B * unroll * steps / (red["ms"] * 1e-3), "ms_per_training_step": red["ms"] / steps,
           "rollout_ms": red["ro"] / steps, "sgd_phase_ms": red["sgd"] / steps, "ms_per_minibatch_update": red["sgd"] / steps / (nup * nmb),
           "minibatch_updates_per_training_step": nup * nmb, "last_metrics": m}
    nparams = sum(int(np.prod(s)) for s in tr.learner.shapes.values())  # 1630397 for the rodent
    flops = 6.0 * nparams * (unroll * B // nmb)  # fwd + bwd of both networks per minibatch update
    res["sgd_tflops_dense"] = flops * nup * nmb / (red["sgd"] / steps * 1e-3) / 1e12
    if world > 1:  # the one whole-buffer gradient all-reduce the trainer issues per update, on its own
        import torch.distributed as dist
        lrn = importlib.import_module("vnl-brax-imitation_b200.learner")
        g = tr.learner.grads
        for _ in range(5):
            lrn.all_reduce_gradients(g)
        torch.cuda.synchronize()
        a0, a1 = ev(), ev()
        a0.record()
        for _ in range(50):
            lrn.all_reduce_gradients(g)
        a1.record()
        torch.cuda.synchronize()
        us = sh.reduce_scalars(dict(us=a0.elapsed_time(a1) / 50 * 1e3), op="max", device=dev)["us"]
        res["grad_allreduce_us_standalone"] = us
        res["grad_allreduce_bytes"] = int(g.numel() * 4)
        res["allreduce_share_of_sgd_phase_if_exposed"] = us * 1e-3 / res["ms_per_minibatch_update"]
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
