"""Run `train()` (vnl-brax-imitation_b200/train.py) on the rodent or the humanoid and print one JSON line per evaluation, then a
summary: training env-steps/s, eval time per evaluation, checkpoint write time and size, and the GPU's name and power limit.

    python tools/train.py                                                   # 1 GPU
    python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 tools/train.py
  env: ENV=rodent|humanoid (rodent)  CLIP=standing|moving (standing; the humanoid's packaged clip)  ENVS (8192, global)
       NUM_TIMESTEPS (2 training steps per epoch)  NUM_EVALS (3)  MINIBATCHES (32)  UPDATES (16)  EVAL_ENVS (128)
       CKPT_DIR (none: no checkpoints)  RESUME (a step_<n> directory, or "latest" for the newest one in CKPT_DIR)"""
import importlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_identity(index: int) -> dict:
    """Name and power limit of the card the run used, read in the same run."""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": limit}
    except Exception as e:  # the numbers above stay valid; say that the card was not identified
        return {"gpu": "unknown (%s)" % type(e).__name__, "power_limit": "unknown"}


def main():
    import torch
    P = lambda n: importlib.import_module("vnl-brax-imitation_b200." + n)
    sh, trn, ckpt = P("sharding"), P("train"), P("checkpoint")
    rank, local_rank, world = sh.env_info()
    torch.cuda.set_device(local_rank)
    dev = "cuda:%d" % local_rank
    if world > 1:
        sh.init_process_group("nccl")
    env_name, clip = os.environ.get("ENV", "rodent"), os.environ.get("CLIP", "standing")
    if env_name == "humanoid":
        model, ref = P("envs.humanoid").packaged_humanoid(moving=clip == "moving")
        env = P("envs").HumanoidTracking(model=model, reference_clip=ref, device=dev)
    elif env_name == "rodent":
        rod = P("envs.rodent")
        model, ref = rod.packaged_rodent()
        env = P("envs").RodentTracking(reference_clip=ref, model=model, device=dev, **rod.RODENT_ENV_ARGS)
    else:
        raise ValueError("ENV must be rodent or humanoid")
    B, nmb = int(os.environ.get("ENVS", 8192)), int(os.environ.get("MINIBATCHES", 32))
    num_evals = int(os.environ.get("NUM_EVALS", 3))
    cfg = dict(num_envs=B, batch_size=B // nmb, num_minibatches=nmb, num_updates_per_batch=int(os.environ.get("UPDATES", 16)),
               num_evals=num_evals, num_eval_envs=int(os.environ.get("EVAL_ENVS", 128)))
    per_step = B * 20
    num_timesteps = int(os.environ.get("NUM_TIMESTEPS", 2 * max(num_evals - 1, 1) * per_step))
    ckpt_dir, resume = os.environ.get("CKPT_DIR") or None, os.environ.get("RESUME") or None
    if resume == "latest":
        resume = ckpt.latest(ckpt_dir)
        if resume is None:
            raise SystemExit("RESUME=latest: no checkpoint in %s" % ckpt_dir)
    evals = []

    def progress(step, metrics):
        evals.append(metrics)
        line = {"step": step, **{k: v for k, v in metrics.items() if isinstance(v, float)}}
        print(json.dumps(line), flush=True)

    full = dict(trn.DEFAULTS, **cfg)
    trn.check_config(env, full, world)
    run = trn.Run(env, full, rank=rank, world_size=world)
    t0 = time.perf_counter()
    run.fit(num_timesteps, progress_fn=progress, checkpoint_dir=ckpt_dir, restore_checkpoint_path=resume)
    wall = time.perf_counter() - t0
    if rank == 0:
        trained = [m for m in evals if "training/sps" in m]
        train_s = (trained[-1]["training/walltime"] - (float(ckpt.read_meta(resume)["training_walltime"]) if resume else 0.0)) if trained else 0.0
        steps = len(trained) * run_steps_per_epoch(trn, num_timesteps, full)
        summary = {"summary": "%s%s train(): %d envs x unroll 20, %d x %d minibatch updates per training step, %d evals%s" % (
                       env_name, "" if env_name == "rodent" else " (%s clip)" % clip, B, full["num_updates_per_batch"], nmb, num_evals,
                       ", resumed from %s" % resume if resume else ""),
                   "n_gpus": world, "training_env_steps_per_s": steps / train_s if train_s else None, "epochs_run": len(trained),
                   "training_sps_per_epoch": [m["training/sps"] for m in trained],
                   "eval_s_per_evaluation": [m["eval/epoch_eval_time"] for m in evals], "wall_s": wall, "final_env_steps": run.env_steps,
                   "checkpoints": [{k: c[k] for k in ("step", "seconds", "bytes")} for c in run.checkpoint_log],
                   "last_training_metrics": {k: v for k, v in (trained[-1] if trained else {}).items() if k.startswith("training/")}}
        summary.update(gpu_identity(local_rank))
        print(json.dumps(summary), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


def run_steps_per_epoch(trn, num_timesteps, cfg):
    s = trn.schedule(num_timesteps, cfg["num_evals"], cfg["batch_size"], cfg["num_minibatches"], cfg["unroll_length"])
    return s["training_steps_per_epoch"] * s["env_steps_per_training_step"]


if __name__ == "__main__":
    main()
