"""The cost of per-clip evaluation (DESIGN §3i) on a rodent clip library: Evaluator.run_evaluation with per_clip off and on,
alternated in one process, and the time of the two per-clip kernels and of the result copy.

  env:      RodentMultiClipTracking over CLIPS (64) SYNTHETIC variants of the packaged clip (clip i: the clip time-reversed for odd i,
            rolled by 17 i frames for even i), EVAL_ENVS = CLIPS x WINDOWS (24) envs, episode length 150, CUDA graph, fp32-class
            policy (PrecisePolicy, 3xTF32) with freshly initialised parameters;
  timing:   a warm-up evaluation per setting (graph capture), then REPS (5) alternations of one evaluation per setting;
            eval/epoch_eval_time of each (reset + unroll + reductions + synchronise; the result copy to the host comes after it);
  profile:  one more evaluation with per_clip on under torch.profiler: mean device time of vnl_eval_metrics, vnl_eval_clip_stats
            and vnl_eval_frame_profile, and, in a profiler run of its own, the two device-to-host copies of the per-clip results.

    CLIPS=842 python tools/eval_bench.py [out.json]      (default out: profiles/eval_per_clip.json; results are kept per clip count)"""
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

P = lambda n: importlib.import_module("vnl-brax-imitation_b200." + n)


def synthetic_clips(clip, n):
    """n clips of the packaged clip's length: clip i is the clip time-reversed (odd i) or rolled by 17 i frames (even i)."""
    T = clip.position.shape[0]
    out = []
    for i in range(n):
        idx = np.arange(T)[::-1] if i % 2 else np.roll(np.arange(T), 17 * i)
        out.append(clip.replace(**{k: np.asarray(getattr(clip, k))[idx] for k in ("position", "quaternion", "joints", "body_positions", "velocity",
                                                                                  "angular_velocity", "joints_velocity", "body_quaternions")
                                   if getattr(clip, k) is not None}))
    return out


def cuda_times(prof, patterns):
    """{key: [device us]} of the profiler's CUDA events whose name contains the key's pattern."""
    out = {k: [] for k in patterns}
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        for k, pat in patterns.items():
            if pat in ev.name:
                out[k].append(ev.device_time if hasattr(ev, "device_time") else ev.cuda_time)
    return out


def main():
    dev = "cuda:0"
    nclips, windows, reps, T = int(os.environ.get("CLIPS", 64)), int(os.environ.get("WINDOWS", 24)), int(os.environ.get("REPS", 5)), 150
    B = nclips * windows
    rod, ev, pol = P("envs.rodent"), P("evaluator"), P("policy")
    model, clip = rod.packaged_rodent()
    t0 = time.perf_counter()
    env = P("envs").RodentMultiClipTracking(reference_clips=synthetic_clips(clip, nclips), model=model, device=dev, **rod.RODENT_ENV_ARGS)
    build_s = time.perf_counter() - t0
    eng = env.engine
    params = pol.init_params(np.random.default_rng(0), pol.param_shapes(eng.traj_size, eng.obs_size, env.action_size))
    policy = pol.PrecisePolicy(params, dev)
    evals = {flag: ev.Evaluator(env, policy, num_eval_envs=B, episode_length=T, seed=0, per_clip=flag) for flag in (False, True)}
    times = {False: [], True: []}
    for e in evals.values():
        e.run_evaluation({})  # capture + warm-up
    for _ in range(reps):
        for flag, e in evals.items():
            times[flag].append(e.run_evaluation({})["eval/epoch_eval_time"])
    e = evals[True]
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        e._unroll()
        torch.cuda.synchronize()
    k = cuda_times(prof, {"eval_metrics": "eval_metrics_kernel", "clip_stats": "eval_clip_stats_kernel", "frame_profile": "eval_frame_profile_kernel"})
    cols = [(n, rod.METRIC_KEYS.index(n)) for n in env.metric_keys] + [("reward", len(rod.METRIC_KEYS))]
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        e._per_clip_metrics(cols)
    copies = cuda_times(prof, {"d2h": "Memcpy DtoH"})["d2h"]
    off, on = np.median(times[False]), np.median(times[True])
    run = {"config": "RodentMultiClipTracking, %d SYNTHETIC clips (time-reversed / rolled variants of the packaged clip), %d eval envs "
                     "(%d windows per clip), episode length %d, PrecisePolicy (3xtf32), CUDA graph; per_clip off / on alternated, %d "
                     "evaluations each after a warm-up" % (nclips, B, windows, T, reps),
           "task_blob_bytes": int(env.task_blob.nbytes), "env_build_s": build_s,
           "eval_s": {"per_clip_off": times[False], "per_clip_on": times[True]},
           "median_eval_s": {"per_clip_off": off, "per_clip_on": on}, "median_overhead_s": on - off,
           "kernel_us": {n: float(np.mean(v)) if v else None for n, v in k.items()},
           "result_copy_us": copies, "result_bytes": int(e.clip_out.nbytes + e.clip_count.nbytes)}
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    run["gpu"] = q
    print(json.dumps(run), flush=True)
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "eval_per_clip.json")
    res = {}
    if os.path.exists(path):
        with open(path) as f:
            res = json.load(f)
    res[str(nclips)] = run
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
