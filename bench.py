#!/usr/bin/env python
"""Benchmark of the hot path: rodent imitation env-steps/s (BASELINE.json `metric`).

    python bench.py --gpus N --steps K --warmup W            our arm (one process per GPU under torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  the reference arm: the CPU implementation of the same path

A "step" is one pass of the hot path over one batch: ONE fused launch that advances every env of the rank's shard by
one env step (5 MJX-style physics substeps + reward / obs / trajectory window / termination) and applies brax's
AutoReset (restore the cached first state where done; `info` keeps running -- SURVEY quirk Q7).
Workload (BASELINE.json configs[1]): rodent.xml (0.9 rescale, torque actuators, CG 6x6, pyramidal, eulerdamp),
clip transform_snips_groom.p, 4096 envs per GPU, iid U(-1, 1) actions, weak scaling (env shards are independent,
no data-path collective).

`value`      whole-job env-steps/s with state and pre-generated actions resident in HBM (CUDA events, max over ranks).
`e2e`        the same metric through the public host-buffer API (`hostio.HostStepper.step`, the host form of `env.step` +
             AutoReset): every step copies the step's actions from pinned host memory and returns once obs, traj, reward
             and done are in pinned host memory (two launches cut at the last wave boundary; the first chunk's copy
             overlaps the last wave's compute).
`roofline`   HBM view of the fused kernel (algorithmic bytes at the step boundary / launch time) against the measured copy
             bandwidth; `roofline_fp32` is the binding one (SURVEY 8d): algorithmic FLOPs / launch time against an FFMA
             microkernel measured in the same run.
`cpu_baseline` the CPU oracle (fp32 build, OpenMP over envs, all host cores) on a bounded sample, rank 0, N = 1 only.

`--dump-outputs DIR` writes what the timed path returned in its last timed step (rank 0's shard) as DIR/<name>.npy, so that
two builds run with the same arguments, and therefore the same seeded inputs, can be compared output for output.
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ENVS_PER_GPU = 4096
ENV_ARG_KEYS = ("end_eff_names", "appendage_names", "walker_body_names", "joint_names", "center_of_mass", "clip_length",
                "sub_clip_length", "ref_traj_length", "termination_threshold")


def pkg(name=""):
    return importlib.import_module("vnl-brax-imitation_b200" + (("." + name) if name else ""))


# ------------------------------------------------------------------------------------------------------------------
# work model (SURVEY 8d)
# ------------------------------------------------------------------------------------------------------------------
def algorithmic_bytes(dims, obs_size, traj_size, ntrack):
    """Compulsory HBM words at the step boundary, recomputed from the fields the kernel really moves."""
    nq, nv, na, nu, nb = dims["nq"], dims["nv"], dims["na"], dims["nu"], dims["nbody"]
    rd = nq + nv + na + nv + 3 * ntrack + nu + 2 + 1  # state, old xpos of the tracked bodies, action, 2 frame ints, done flag
    wr = nq + nv + na + nv + 3 * nb + 4 * nb + 3 + nv + obs_size + traj_size + 1 + 1 + 7 + 2 + 4
    return 4 * (rd + wr)


def algorithmic_flops(dims, depth, n_frames, I, L):
    """Work-optimal FLOPs per env step (SURVEY 8d formula), with the executed solver iterations I per substep and
    line-search iterations L per solver iteration."""
    nb, nv, nu, ncon, nefc, nlim, P = (dims[k] for k in ("nbody", "nv", "nu", "ncon", "nefc", "nlimit", "nM"))
    ed = 1 if dims["eulerdamp"] else 0
    ldl = float(np.sum(depth * (depth - 1.0)))
    Jp = 12 * nv + 6 * nb + 45 * ncon + nlim
    nsolve, nmul = 2 + I + ed, 3 + I
    f = 350 * nb + 60 * nv + 10 * nb + 70 * nv + 12 * P + (1 + ed) * ldl + 250 * nb + 40 * nv + 4 * nu + 80 * ncon
    f += Jp + 40 * nefc + nsolve * 4 * P + nmul * 4 * P + 3 * (2 * Jp + 6 * nefc)
    f += I * (2 * Jp + 12 * nefc + (2 + 3 * L) * 8 * nefc + 12 * nv) + 6 * nv + 40
    return n_frames * f


# ------------------------------------------------------------------------------------------------------------------
# output dump
# ------------------------------------------------------------------------------------------------------------------
DUMP_BYTES = 64 << 20


def host_copy(arrays, prefix=""):
    """Flat {name: numpy array} copy of a (nested) dict of tensors / arrays; '/' in names becomes '.'."""
    out = {}
    for k, v in arrays.items():
        name = prefix + k.replace("/", ".")
        if isinstance(v, dict):
            out.update(host_copy(v, name + "."))
        else:
            out[name] = v.detach().cpu().numpy() if hasattr(v, "detach") else np.asarray(v)
    return out


def dump_outputs(path, arrays, seed=0):
    """Writes `arrays` (from `host_copy`) as <path>/<name>.npy: float32 stays float32, everything else becomes float64 (exact
    for the integer outputs).  At most DUMP_BYTES in all: arrays are visited smallest first and each may use an equal share of
    the budget left; those within their share are written whole, larger ones as a fixed, seeded sample of their elements
    (flattened, in index order) that depends only on the seed and the array's size."""
    flat = {k: v.astype(np.float32 if v.dtype == np.float32 else np.float64) for k, v in arrays.items()}
    os.makedirs(path, exist_ok=True)
    left = DUMP_BYTES
    order = sorted(flat, key=lambda k: (flat[k].nbytes, k))
    for i, k in enumerate(order):
        v = flat[k]
        share = left // (len(order) - i)
        if v.nbytes > share:
            keep = max(1, share // v.itemsize)
            v = v.reshape(-1)[np.unique(np.random.default_rng(seed).integers(0, v.size, size=keep))]
        left -= v.nbytes
        np.save(os.path.join(path, k + ".npy"), v)


# ------------------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index, period=0.2):
        super().__init__(daemon=True)
        self.index, self.period, self.samples, self.reasons, self.stop_flag = index, period, [], set(), threading.Event()
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self.stop_flag.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            self.stop_flag.wait(self.period)

    def finish(self):
        self.stop_flag.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------------------------
def build_workload():
    rod, mb = pkg("envs.rodent"), pkg("model_blob")
    model, clip = rod.packaged_rodent()
    return rod, mb, model, clip


WORKLOADS = {
    # BASELINE.json configs[1] (the config the metric is quoted on) and configs[2]
    "rodent": dict(envs=4096, nu=30, text="rodent imitation env step+reward/obs (envs/rodent.py, rodent.xml, transform_snips_groom.p)"),
    "humanoid": dict(envs=8192, nu=21, text="CMU humanoid imitation env step+reward/obs (envs/humanoid.py, humanoid.xml, synthetic "
                                            "standing clip: qpos0 tiled x256 -- the reference clip humanoid_traj_stand.p is absent)"),
    # BASELINE.json configs[3]: the PPO rollout / the whole training_step, and configs[4]: the two-agent physics sweep point
    "rollout": dict(envs=8192, nu=30, text="rodent PPO rollout (ppo_imitation/acting.py:30-80: intention-network policy + fused env step with the "
                                           "Episode / AutoReset wrappers, one CUDA graph per unroll, normaliser updated per unroll)"),
    "train": dict(envs=8192, nu=30, text="rodent PPO training_step (ppo_imitation/train.py:296-349: rollout + normaliser + 16 x 32 minibatch "
                                         "updates of 5120 rows: loss fwd / bwd on tcgen05 TF32 GEMMs, Adam, gradient all-reduce)"),
    "rodent_pair": dict(envs=16384, nu=60, text="rodent_pair.xml two-agent physics env step (5 substeps, U(-1,1) controls, no task logic: the "
                                                "reference has no env class for this model)"),
    # BASELINE.json configs[0]: the reference's own CPU-runnable plumbing case (a parity case; benched only on request)
    "ant": dict(envs=256, nu=8, text="ant imitation env step+reward/obs (envs/ant.py, ant.xml brax-style fused, Newton 1x4, still clip: "
                                     "init_qpos tiled -- the reference clip ant_traj_still.p is absent)"),
}


def make_env(workload, device):
    """(env, qpos, qvel, start) builder for the rank-local shard."""
    envs = pkg("envs")
    if workload == "humanoid":
        hum = pkg("envs.humanoid")
        model, clip = hum.packaged_humanoid()
        return envs.HumanoidTracking(model=model, reference_clip=clip, device=device)
    if workload == "ant":
        antm = pkg("envs.ant")
        model, clip = antm.packaged_ant()
        return envs.AntTracking(model=model, reference_clip=clip, device=device)
    rod = pkg("envs.rodent")
    model, clip = rod.packaged_rodent()
    return envs.RodentTracking(reference_clip=clip, model=model, device=device, **rod.RODENT_ENV_ARGS)


def workload_draws(workload, env, total, lo, hi):
    if workload == "humanoid":  # HumanoidTracking.reset (humanoid.py:78-102): frame ~ randint(0, 250 - 150 - 5), no noise
        rng = np.random.default_rng(0)
        start = rng.integers(0, 95, size=total).astype(np.int32)[lo:hi]
        rt = env._ref_traj
        qpos = np.hstack([rt.position[start], rt.quaternion[start], rt.joints[start]]).astype(np.float32)
        qvel = np.hstack([rt.velocity[start], rt.angular_velocity[start], rt.joints_velocity[start]]).astype(np.float32)
        return qpos, qvel, start
    if workload == "ant":  # AntTracking.reset (ant.py:76-103): start_frame = 0, no noise
        start = np.zeros(total, dtype=np.int32)[lo:hi]
        rt = env._ref_traj
        qpos = np.hstack([rt.position[start], rt.quaternion[start], rt.joints[start]]).astype(np.float32)
        qvel = np.hstack([rt.velocity[start], rt.angular_velocity[start], rt.joints_velocity[start]]).astype(np.float32)
        return qpos, qvel, start
    return initial_draws(env._ref_traj, total, lo, hi)


def initial_draws(fclip, total, lo, hi, seed=0):
    """RodentTracking.reset draws (envs/rodent.py:123-132) for global env ids [lo, hi) out of `total`."""
    rng = np.random.default_rng(seed)
    start = rng.integers(0, 235, size=total).astype(np.int32)
    noise = (1e-3 * rng.standard_normal((total, 74))).astype(np.float32)
    s = start[lo:hi]
    qpos = np.hstack([fclip.position[s], fclip.quaternion[s], fclip.joints[s]]).astype(np.float32) + noise[lo:hi]
    qvel = np.hstack([fclip.velocity[s], fclip.angular_velocity[s], fclip.joints_velocity[s]]).astype(np.float32)
    return qpos, qvel, s


def cpu_oracle_rate(seconds_target=12.0, nthreads=0, steps=None, sample_envs=None, warmup=1):
    """env-steps/s of the CPU oracle (fp32, OpenMP over envs) on a bounded sample of the same workload."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle  # the reference arm / cpu_baseline leg is the one place bench.py may execute oracle/
    rod, mb, model, clip = build_workload()
    task, fclip, idx, obs_size, traj_size = rod.rodent_task_tables(model, clip, **{k: rod.RODENT_ENV_ARGS[k] for k in ENV_ARG_KEYS})
    blob = mb.build_model_blob(model)
    dims = mb.read_dims(blob)
    # torchrun exports OMP_NUM_THREADS=1 to its workers: size the pool from the cores this process may run on
    nt = nthreads or len(os.sched_getaffinity(0))
    kw = dict(precision=32, dims=dims, obs_size=obs_size, traj_size=traj_size, nthreads=nt)
    rng = np.random.default_rng(0)

    def run(B, nsteps, nwarm):
        qpos, qvel, start = initial_draws(fclip, ENVS_PER_GPU, 0, B)
        s, _ = oracle.reset(blob, task, qpos, qvel, start, **kw)
        first = {k: v.copy() for k, v in s.items()}
        per_step = []
        for it in range(nwarm + nsteps):
            a = rng.uniform(-1, 1, size=(B, 30))
            t0 = time.perf_counter()
            s, o = oracle.step(blob, task, s, a, **kw)
            d = o["done"] > 0  # AutoReset: restore the first pipeline state where done (info keeps running, Q7)
            for k in ("qpos", "qvel", "act", "qacc_warmstart", "xpos", "xquat", "subtree_com", "qfrc_actuator"):
                s[k][d] = first[k][d]
            if it >= nwarm:
                per_step.append(time.perf_counter() - t0)
        return float(np.sum(per_step)), float(np.mean(per_step))

    if sample_envs is None:
        t_pilot, _ = run(8 * nt, 1, 1)
        rate = 8 * nt / max(t_pilot, 1e-6)
        nsteps = steps or 4
        sample_envs = int(min(ENVS_PER_GPU, max(8 * nt, rate * seconds_target / nsteps)))
    nsteps = steps or 4
    total, mean = run(sample_envs, nsteps, warmup)
    return dict(value=sample_envs * nsteps / total, ms_per_step=1e3 * mean, cores=nt, envs=sample_envs, steps=nsteps,
                sample="%d envs x %d env steps of the bench workload (fp32 oracle, OpenMP over envs)" % (sample_envs, nsteps))


def workload_config(workload, B, world):
    """`config` keys shared verbatim by both arms (the driver compares them)."""
    wl = WORKLOADS[workload]
    return {"workload": "%s, %d envs per GPU, 5 physics substeps per env step, U(-1,1) actions, AutoReset with the "
                        "reference's info-not-reset quirk" % (wl["text"], B),
            "envs_per_gpu": B, "global_envs": B * world, "parallelism": "env shards, dp%d, no data-path collective" % world}


def run_reference(args):
    """Reference arm: the CPU implementation of the same path on the box's host cores.  The reference's own arithmetic
    (mujoco-mjx / brax on JAX-CPU) is not installable here (SURVEY 8c), so this times the repo's CPU restatement of it
    (`kind: "port"`): the same workload, the same K timed + W warm-up steps as our arm, each step over a bounded sample of
    the 4096-env batch sized so that the run ends within a few minutes (the whole batch when the cores allow)."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    K, W = args.steps, args.warmup
    B = args.envs_per_gpu or WORKLOADS["rodent"]["envs"]
    nt = len(os.sched_getaffinity(0))
    pilot = cpu_oracle_rate(steps=1, sample_envs=8 * nt, warmup=1)
    budget_s = 90.0
    sample = int(min(B, max(8 * nt, pilot["value"] * budget_s / (K + W))))
    r = cpu_oracle_rate(steps=K, sample_envs=sample, warmup=W)
    cfg = workload_config("rodent", B, 1)
    cfg["reference_sample"] = "each step advances %d of the %d envs (bounded sample); CPU port of the path on %d host cores" % (sample, B, r["cores"])
    line = {"impl": "reference", "metric": "rodent imitation env-steps/s", "value": r["value"], "unit": "env-steps/s",
            "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": r["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": r["value"], "unit": "env-steps/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
            "e2e": {"value": r["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "CPU PORT, not the reference's JAX-CPU path: mujoco-mjx / brax / jax are not installable in this image "
                    "(SURVEY 8c), so this arm times the repo's C++ restatement of the path (oracle/, fp32, OpenMP over envs)"}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist

    sh = pkg("sharding")
    rank, local_rank, world = sh.env_info()
    if world != args.gpus and world > 1:
        raise SystemExit("--gpus must equal WORLD_SIZE under torchrun")
    if world == 1 and args.gpus > 1:
        raise SystemExit("launch with: python -m torch.distributed.run --nproc-per-node %d bench.py --gpus %d ..." % (args.gpus, args.gpus))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        sh.init_process_group("nccl")
    mb = pkg("model_blob")
    wl = WORKLOADS[args.workload]
    env = make_env(args.workload, str(dev))
    eng = env.engine
    B = args.envs_per_gpu or wl["envs"]
    total = B * world
    lo, hi = sh.shard_range(total, rank, world)
    qpos, qvel, start = workload_draws(args.workload, env, total, lo, hi)
    K, W = args.steps, args.warmup

    s0 = env.reset_from(qpos, qvel, start)
    first = dict(s0.pipeline_state)
    first_obs = s0.obs
    gen = torch.Generator(device=dev)
    gen.manual_seed(1234 + rank)  # Philox counter RNG on the device, pre-generated so RNG cost is outside the timed region
    actions = torch.rand(W + K, B, env.action_size, generator=gen, device=dev) * 2 - 1

    def fresh_state():
        st = {k: v.clone() for k, v in first.items()}
        st["cur_frame"] = s0.info["cur_frame"].clone()
        st["sub_clip_frame"] = s0.info["sub_clip_frame"].clone()
        return st

    # ---- device-resident loop -----------------------------------------------------------------------------------
    a_st, b_st, out = fresh_state(), eng.alloc_state(B), eng.alloc_outputs(B)
    stats_acc = torch.zeros(4, dtype=torch.float64, device=dev)

    def one_step(i):
        nonlocal a_st, b_st
        eng.step_autoreset(a_st, actions[i], b_st, out, first, first_obs)
        a_st, b_st = b_st, a_st

    for i in range(W):
        one_step(i)
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = eng.launches
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(W, W + K):
        one_step(i)
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.finish()
    launches = eng.launches - launches0
    done_frac = float(out["done"].mean())
    # the next state and outputs of the last timed step, before the roofline loop below steps on
    last = host_copy({**{k: a_st[k] for k in pkg("_lib").STATE_F + ("cur_frame", "sub_clip_frame")}, **out}) if args.dump_outputs and rank == 0 else None

    # ---- per-launch duration of the fused kernel for the roofline (events bracket every launch on its stream; the
    # clock sampler is off), and the solver counters of the executed-FLOP model ---------------------------------------
    nk = min(K, 20)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(nk)]
    for j, i in enumerate(range(W, W + nk)):
        evs[j][0].record()
        one_step(i)
        evs[j][1].record()
        stats_acc += out["stats"].sum(0)
    torch.cuda.synchronize()
    kernel_ms = float(np.mean([a.elapsed_time(b) for a, b in evs]))
    stats_steps = nk

    # ---- end to end through the public API with host buffers ------------------------------------------------------
    host_actions = torch.empty(K, B, env.action_size, dtype=torch.float32).pin_memory()
    host_actions.copy_(actions[W:W + K].cpu())
    stepper = pkg("hostio").HostStepper(env, s0, autoreset=True)  # the public host-buffer form of env.step (+ AutoReset)
    launches_e2e0 = eng.launches
    for i in range(min(W, 3)):
        stepper.step(host_actions[i])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(K):
        stepper.step(host_actions[i])  # returns once obs / traj / reward / done of this step are in pinned host memory
    t1.record()
    torch.cuda.synchronize()
    e2e_ms_total = t0.elapsed_time(t1)
    h2d, d2h = stepper.h2d_bytes, stepper.d2h_bytes
    e2e_chunks = len(stepper.chunks)

    # ---- FP32 probe ---------------------------------------------------------------------------------------------------
    blocks, iters = 148 * 16, 20000
    scratch = torch.empty(blocks * 256, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    eng.lib.vnl_ffma_probe(blocks, 200, scratch.data_ptr(), stream)
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    eng.lib.vnl_ffma_probe(blocks, iters, scratch.data_ptr(), stream)
    p1.record()
    torch.cuda.synchronize()
    ffma_tflops = blocks * 256 * iters * 32 / (p0.elapsed_time(p1) * 1e-3) / 1e12

    # ---- max over ranks ---------------------------------------------------------------------------------------------
    red = sh.reduce_scalars(dict(ms=ms_total, e2e=e2e_ms_total, kern=kernel_ms), op="max", device=dev)
    sums = sh.reduce_scalars(dict(launches=float(launches)), op="sum", device=dev)
    rank_ms = [ms_total / K]
    if world > 1:
        gathered = [torch.zeros(1, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(gathered, torch.tensor([ms_total / K], dtype=torch.float64, device=dev))
        rank_ms = [float(g.item()) for g in gathered]
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    if last is not None:
        dump_outputs(args.dump_outputs, last)
    ms_total, e2e_ms_total, kernel_ms = red["ms"], red["e2e"], red["kern"]
    value = total * K / (ms_total * 1e-3)
    e2e_value = total * K / (e2e_ms_total * 1e-3)

    dims = eng.dims
    depth = mb.read_field(env.model_blob, "VNL_F_DOF_DEPTH", np.int32).astype(np.float64)
    st = (stats_acc / (stats_steps * B)).cpu().numpy()  # per env step: solver iters, ls iters, active contacts, active limits
    nfr = eng.n_frames
    I = st[0] / nfr
    L = st[1] / max(st[0], 1e-9)
    flops = algorithmic_flops(dims, depth, nfr, I, L)
    flops_static = algorithmic_flops(dims, depth, nfr, dims["iterations"], dims["ls_iterations"])
    ntrack = len(env._body_idxs) if hasattr(env, "_body_idxs") else dims["nbody"]
    nbytes = algorithmic_bytes(dims, eng.obs_size, eng.traj_size, ntrack)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    hbm_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    traffic = None
    try:  # dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed ncu --set full capture
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        if int(tj.get("envs", 0)) == B and args.workload == "rodent":
            traffic = float(tj["dram_bytes_per_launch"])
    except Exception:
        pass
    ach_gbs = B * nbytes / (kernel_ms * 1e-3) / 1e9
    ach_tf = B * flops / (kernel_ms * 1e-3) / 1e12
    line = {
        "metric": "%s imitation env-steps/s" % args.workload, "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": ms_total / K, "rank_ms_per_step": rank_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {**workload_config(args.workload, B, world),
                   "l2": "not flushed: the whole batch state (%.0f MB) is L2-resident; numbers are L2-warm as in the rollout loop"
                         % (B * nbytes / 1e6), "done_fraction": done_frac},
        "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms_total / K, "launches_per_step": e2e_chunks,
                "api": "hostio.HostStepper.step (vnl_step_autoreset in two launches cut at a wave boundary, D2H of the first overlaps compute of the last wave)"},
        "gpu_launches": int(sums["launches"]),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gbs / hbm_peak,
                     "traffic": traffic, "peak_source": hbm_src, "bytes_per_env_step": nbytes, "kernel_ms": kernel_ms,
                     "note": "this path is FP32-latency bound, not HBM bound (intensity ~%d flop/B); see roofline_fp32" % (flops / nbytes)},
        "roofline_fp32": {"bound": "fp32", "achieved": ach_tf, "peak": ffma_tflops, "unit": "TFLOP/s", "frac": ach_tf / ffma_tflops,
                          "peak_source": "FFMA microkernel measured in this run (nominal 74.4)", "flops_per_env_step": flops,
                          "flops_per_env_step_static_max": flops_static,
                          "flops_note": "SURVEY 8(d) count of the REFERENCE algorithm; it includes one M.search mat-vec per CG iteration "
                                        "(%.0f flop per env step, %.1f %% of the count) that this kernel replaces by an exact recursion "
                                        "(DESIGN section 3)" % (nfr * I * 4 * dims["nM"] * (1 if dims.get("solver", 1) != 2 else 0),
                                                               100.0 * nfr * I * 4 * dims["nM"] * (1 if dims.get("solver", 1) != 2 else 0) / flops),
                          "executed": {"solver_iters_per_substep": I, "ls_iters_per_solver_iter": L,
                                       "active_contacts_per_substep": st[2] / nfr, "active_limits_per_substep": st[3] / nfr}},
    }
    if world == 1 and not args.no_cpu_baseline and args.workload == "rodent":
        r = cpu_oracle_rate(seconds_target=12.0)
        line["cpu_baseline"] = {"value": r["value"], "unit": "env-steps/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]}
    else:
        line["cpu_baseline"] = None
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# BASELINE.json configs[3] / configs[4] as driver-runnable workloads
# ------------------------------------------------------------------------------------------------------------------
def _finish_extra(args, line_fn, ms_total, e2e_ms_total, K, dev, sampler, launches):
    """max over ranks, clocks, one JSON line from rank 0."""
    import torch.distributed as dist
    sh = pkg("sharding")
    rank, _, world = sh.env_info()
    clocks = sampler.finish()
    red = sh.reduce_scalars(dict(ms=ms_total, e2e=e2e_ms_total), op="max", device=dev)
    sums = sh.reduce_scalars(dict(launches=float(launches)), op="sum", device=dev)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank == 0:
        line = line_fn(red["ms"], red["e2e"], int(sums["launches"]))
        line.update({"n_gpus": world, "steps": K, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                     "dtype": "f32", "data": "synthetic", "clocks": clocks, "cpu_baseline": None})
        print(json.dumps(line), flush=True)


def run_pair(args):
    """configs[4]: rodent_pair.xml physics env steps (5 substeps, no task logic: the reference has no env class for this model)."""
    import torch
    sh, mjcf, mb, lib = pkg("sharding"), pkg("mjcf"), pkg("model_blob"), pkg("_lib")
    rank, local_rank, world = sh.env_info()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        sh.init_process_group("nccl")
    model = mjcf.load_model(os.path.join(ROOT, "vnl-brax-imitation_b200", "data", "rodent_pair_model.npz"))
    eng = lib.Engine(mb.build_model_blob(model), None, device=str(dev))
    B = args.envs_per_gpu or WORKLOADS["rodent_pair"]["envs"]
    K, W = args.steps, args.warmup
    rng = np.random.default_rng(rank)
    qpos = np.tile(model.arrays["qpos0"], (B, 1)).astype(np.float32) + (1e-3 * rng.standard_normal((B, model.nq))).astype(np.float32)
    a, b = eng.alloc_state(B), eng.alloc_state(B)
    a["qpos"].copy_(torch.tensor(qpos, device=dev))
    gen = torch.Generator(device=dev)
    gen.manual_seed(67280421310721)  # torch's default CUDA seed: the controls this workload has always drawn, on every rank
    ctrl = torch.rand(W + K, B, model.nu, generator=gen, device=dev) * 2 - 1
    stats = torch.zeros(B, 4, dtype=torch.int32, device=dev)
    host_ctrl = torch.empty(K, B, model.nu).pin_memory()
    host_ctrl.copy_(ctrl[W:].cpu())
    host_q = torch.empty(B, model.nq).pin_memory()

    def step(c):
        nonlocal a, b
        eng.pipeline_step(a, c, b, 5, stats)
        a, b = b, a
    for i in range(W):
        step(ctrl[i])
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = eng.launches
    sh.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        step(ctrl[W + i])
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, host_copy({**{k: a[k] for k in lib.STATE_F}, "stats": stats}))
    dctrl = torch.empty(B, model.nu, device=dev)
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(K):  # host-buffer form: controls from pinned memory in, qpos back to pinned memory, every step
        dctrl.copy_(host_ctrl[i], non_blocking=True)
        step(dctrl)
        host_q.copy_(a["qpos"], non_blocking=True)
        torch.cuda.current_stream().synchronize()
    t1.record()
    torch.cuda.synchronize()
    total = B * world

    def line(ms_t, e2e_t, launches):
        return {"metric": "rodent_pair physics env-steps/s", "value": total * K / (ms_t * 1e-3), "unit": "env-steps/s", "ms_per_step": ms_t / K,
                "config": {"workload": WORKLOADS["rodent_pair"]["text"] + ", %d envs per GPU" % B, "envs_per_gpu": B, "global_envs": total,
                           "parallelism": "env shards, dp%d, no data-path collective" % world, "envs_per_cta": eng.envs_per_cta},
                "e2e": {"value": total * K / (e2e_t * 1e-3), "unit": "env-steps/s", "h2d_bytes_per_step": B * model.nu * 4, "d2h_bytes_per_step": B * model.nq * 4},
                "gpu_launches": launches, "roofline": None}
    _finish_extra(args, line, ms, t0.elapsed_time(t1), K, dev, sampler, eng.launches - l0)


def run_train(args, sgd: bool):
    """configs[3]: rollout of 8192 envs/GPU x unroll 20 (policy + fused env step); with `sgd` the whole training_step of the
    reference (ppo_imitation/train.py:296-349): + normaliser update + SGD phase (16 x 32 minibatch updates, gradient all-reduce)."""
    import torch
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import train_bench
    sh = pkg("sharding")
    rank, local_rank, world = sh.env_info()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        sh.init_process_group("nccl")
    name = "train" if sgd else "rollout"
    B, unroll = args.envs_per_gpu or WORKLOADS[name]["envs"], 20
    nmb, nup = 32, (16 if sgd else 0)
    tr = train_bench.build(dev, rank, world, B, unroll, nmb, max(nup, 1), True, False)
    K, W = args.steps, args.warmup
    host_metric = torch.empty(8).pin_memory()

    def one(read_back):
        tr.rollout.eps_z.normal_(generator=tr.gen); tr.rollout.eps_a.normal_(generator=tr.gen)
        data = tr.rollout.generate_unroll()
        tr.stats.update(data["observation"])
        if sgd:
            tr.learner.set_normalizer(tr.stats.mean, tr.stats.std)
            tr.sgd_phase(data)
            tr.policy.load_params(tr.learner.policy_params())
        if read_back:  # the step's result on the host: loss metrics (train) / mean reward of the unroll (rollout)
            host_metric[:1].copy_(data["reward"].mean().reshape(1), non_blocking=True)
            if sgd:
                host_metric.copy_(tr.learner.ws["metrics"], non_blocking=True)
            torch.cuda.current_stream().synchronize()
        return data
    for _ in range(min(W, 3)):
        one(False)
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = tr.rollout.launches + tr.sgd_launches
    sh.barrier()
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    e0.record()
    for _ in range(K):
        one(False)
    e1.record()
    for _ in range(K):
        data = one(True)
    e2.record()
    torch.cuda.synchronize()
    if args.dump_outputs and rank == 0:
        # next_observation[:-1] is observation[1:] (one buffer): only its last row is new
        last = {"rollout": dict(data, next_observation=data["next_observation"][-1:])}
        if sgd:
            last.update(policy=tr.learner.policy_params(), value=tr.learner.value_params(), loss_metrics=tr.learner.ws["metrics"])
        dump_outputs(args.dump_outputs, host_copy(last))
    total = B * world * unroll
    launches = tr.rollout.launches + tr.sgd_launches - l0  # the captured update's kernels are counted per replay

    def line(ms_t, e2e_t, launches_):
        return {"metric": ("rodent PPO training env-steps/s" if sgd else "rodent PPO rollout env-steps/s"), "value": total * K / (ms_t * 1e-3),
                "unit": "env-steps/s", "ms_per_step": ms_t / K,
                "config": {"workload": WORKLOADS[name]["text"] + ", %d envs per GPU" % B, "envs_per_gpu": B, "global_envs": B * world, "unroll_length": unroll,
                           "parallelism": "env shards, dp%d; collectives: normaliser all-reduce (1.9 KB)%s" % (world, ", gradient all-reduce 6.5 MB per minibatch update (2 buckets)" if sgd else ""),
                           "step": "one training_step" if sgd else "one unroll of 20 env steps", "minibatch_updates_per_step": nup * nmb,
                           "policy": "PrecisePolicy (3xTF32)", "learner": "TF32 (one tensor-core pass)"},
                "e2e": {"value": total * K / (e2e_t * 1e-3), "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 32,
                        "note": "the rollout loop has no host input; the step's result (loss metrics / mean reward) is read back every step"},
                "gpu_launches": launches_ // 2, "roofline": None}
    _finish_extra(args, line, e0.elapsed_time(e1), e1.elapsed_time(e2), K, dev, sampler, launches)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=12)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=0, help="default: the workload's BASELINE.json size")
    ap.add_argument("--workload", default="rodent", choices=sorted(WORKLOADS), help="rodent = the config the metric is quoted on")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3)
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "rodent_pair":
        run_pair(args)
    elif args.workload in ("rollout", "train"):
        run_train(args, args.workload == "train")
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
