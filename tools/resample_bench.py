"""The cost of the resampling AutoReset (DESIGN §3h) on the rodent: rollout.Rollout env-steps/s with autoreset="first" and
autoreset="resample", alternated in one process, and the kernels of one `vnl_step_training_resample` call at 0 %, the measured and
100 % done.

  rollout: ENVS (8192) envs x unroll 20, CUDA graph, fp32-class policy (PrecisePolicy, 3xTF32), obs normaliser updated per unroll;
           REPS (5) alternations of one timed unroll per mode after a warm-up; the done fraction per step of each mode.
  reset:   one env step of ENVS envs from the workload's reset states with a chosen fraction of the envs truncated
           (steps_in = episode_length - 1), 20 calls under torch.profiler: mean time of the step kernel (mode 0), the done-list
           compaction and the list reset (mode 5).

    python tools/resample_bench.py [out.json]"""
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (workload builders)

P = lambda n: importlib.import_module("vnl-brax-imitation_b200." + n)


def main():
    dev = torch.device("cuda", 0)
    B, unroll, reps, EP = int(os.environ.get("ENVS", 8192)), 20, int(os.environ.get("REPS", 5)), 150.0
    env = bench.make_env("rodent", str(dev))
    eng = env.engine
    qpos, qvel, start = bench.workload_draws("rodent", env, B, 0, B)
    s0 = env.reset_from(qpos, qvel, start)
    pol, nz, ro_m = P("policy"), P("normalizer"), P("rollout")
    params = pol.init_params(np.random.default_rng(0), pol.param_shapes(eng.traj_size, eng.obs_size, env.action_size))
    gen = torch.Generator(device=dev).manual_seed(0)
    modes = {}
    for mode in ("first", "resample"):
        stats = nz.RunningStatistics(eng.obs_size, str(dev))
        policy = pol.PrecisePolicy(params, str(dev), stats.mean, stats.std)
        ro = ro_m.Rollout(env, policy, s0, unroll, EP, use_graph=True, autoreset=mode, seed=0)
        modes[mode] = dict(ro=ro, stats=stats, ms=[], done=[])

    def one(m, timed):
        ro, stats = m["ro"], m["stats"]
        ro.eps_z.normal_(generator=gen)
        ro.eps_a.normal_(generator=gen)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        tr = ro.generate_unroll()
        stats.update(tr["observation"])
        e1.record()
        torch.cuda.synchronize()
        if timed:
            m["ms"].append(e0.elapsed_time(e1))
            m["done"].append(float((1 - tr["discount"]).mean()))
    for m in modes.values():  # capture + two warm-up unrolls per mode
        one(m, False)
        one(m, False)
    for _ in range(reps):
        for m in modes.values():
            one(m, True)
    res = {"config": "rodent rollout.Rollout, %d envs x unroll %d, CUDA graph, PrecisePolicy (3xtf32), normaliser update per unroll; "
                     "modes alternated, one timed unroll each, %d repetitions" % (B, unroll, reps), "rollout": {}}
    for k, m in modes.items():
        ms = np.array(m["ms"])
        res["rollout"][k] = dict(env_steps_per_s=[B * unroll / (x * 1e-3) for x in ms], ms_per_unroll=ms.tolist(),
                                 median_env_steps_per_s=float(B * unroll / (np.median(ms) * 1e-3)), done_fraction_per_step=m["done"])
    # where an unroll's time goes: one more unroll per mode under torch.profiler, kernel time summed by kind
    kinds = (("env_step", "vnl_env_kernel<0>"), ("env_reset", "vnl_env_kernel<5>"), ("done_list", "done_list"))
    for k, m in modes.items():
        m["ro"].eps_z.normal_(generator=gen)
        m["ro"].eps_a.normal_(generator=gen)
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            m["ro"].generate_unroll()
            torch.cuda.synchronize()
        per = {}
        for ev in prof.events():
            if ev.device_type != torch.autograd.DeviceType.CUDA:
                continue
            kind = next((n for n, pat in kinds if pat in ev.name), "other")
            per[kind] = per.get(kind, 0.0) + (ev.device_time if hasattr(ev, "device_time") else ev.cuda_time) / 1e3
        res["rollout"][k]["profiled_unroll_kernel_ms"] = per
    r = res["rollout"]
    res["resample_over_first"] = r["resample"]["median_env_steps_per_s"] / r["first"]["median_env_steps_per_s"]
    measured = float(np.mean(r["resample"]["done_fraction_per_step"]))

    # ---- the kernels of one call at a given done fraction ----------------------------------------------------------------------
    st = dict({k: v.clone() for k, v in s0.pipeline_state.items()}, cur_frame=s0.info["cur_frame"].clone(),
              sub_clip_frame=s0.info["sub_clip_frame"].clone(), clip_id=s0.info["clip_idx"].clone())
    act = torch.rand(B, env.action_size, device=dev, generator=gen) * 2 - 1
    out, o = eng.alloc_state(B), eng.alloc_outputs(B)
    cnt, scratch = torch.zeros(B, dtype=torch.int32, device=dev), torch.zeros(B + 1, dtype=torch.int32, device=dev)
    res["reset_launch"] = {}
    for label, frac in (("0", 0.0), ("measured", measured), ("100", 1.0)):
        steps = torch.zeros(B, device=dev)
        n = int(round(frac * B))
        steps[torch.randperm(B, generator=torch.Generator().manual_seed(1))[:n].to(dev)] = EP - 1
        call = lambda: eng.step_training_resample(st, act, out, o, steps, torch.zeros(B, device=dev), steps.clone(), torch.zeros(B, device=dev),
                                                  EP, cnt, scratch, 0, 0, *env.resample_spec())
        for _ in range(3):
            call()
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(20):
                call()
            torch.cuda.synchronize()
        times = {}
        for ev in prof.events():
            name = ev.name
            key = "step" if "vnl_env_kernel<0>" in name else "reset" if "vnl_env_kernel<5>" in name else "done_list" if "done_list" in name else None
            if key and ev.device_type == torch.autograd.DeviceType.CUDA:
                times.setdefault(key, []).append(ev.device_time if hasattr(ev, "device_time") else ev.cuda_time)
        done_n = int((o["done"] > 0).sum())
        res["reset_launch"][label] = dict(done_fraction=done_n / B, **{k + "_us": float(np.mean(v)) for k, v in times.items()})
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    res["gpu"] = q
    line = json.dumps(res)
    print(line, flush=True)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
