"""Shared fixtures.  `-m "not gpu"` runs on a CPU-only host (oracle vs golden vectors, host logic,
C-ABI symbols); `-m gpu` are the kernel-vs-oracle parity tests and call through the C ABI."""
import importlib
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

# a checkout of the original VNL-Brax-Imitation project (its MJCF assets): optional, the tests that read it skip without it
REFERENCE = os.environ.get("VNL_REFERENCE")


def reference_asset(name):
    """Path of assets/<name> in the VNL_REFERENCE checkout, or None."""
    path = os.path.join(REFERENCE, "assets", name) if REFERENCE else None
    return path if path and os.path.exists(path) else None


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu on the GPU box")


def pkg(name=""):
    return importlib.import_module("vnl-brax-imitation_b200" + (("." + name) if name else ""))


@pytest.fixture(scope="session")
def rodent():
    """(model, clip, model_blob, task_blob, dims, sizes) from the packaged fixtures."""
    rod = pkg("envs.rodent")
    mb = pkg("model_blob")
    model, clip = rod.packaged_rodent()
    args = {k: rod.RODENT_ENV_ARGS[k] for k in ("end_eff_names", "appendage_names", "walker_body_names", "joint_names",
                                                "center_of_mass", "clip_length", "sub_clip_length", "ref_traj_length",
                                                "termination_threshold")}
    task_blob, fclip, idx, obs_size, traj_size = rod.rodent_task_tables(model, clip, **args)
    model_blob = mb.build_model_blob(model)
    return dict(model=model, clip=clip, fclip=fclip, model_blob=model_blob, task_blob=task_blob, idx=idx,
                dims=mb.read_dims(model_blob), obs_size=obs_size, traj_size=traj_size)


@pytest.fixture(scope="session")
def golden():
    return np.load(os.path.join(ROOT, "tests", "golden", "rodent_clip_golden.npz"))


@pytest.fixture(scope="session")
def oracle_mod():
    import oracle
    oracle.build()
    return oracle


def start_states(rodent, B, seed=0, noise=1e-3):
    """Reset draws of `RodentTracking.reset` (envs/rodent.py:123-132) with numpy's default_rng."""
    rng = np.random.default_rng(seed)
    rt = rodent["fclip"]
    start = rng.integers(0, 235, size=B).astype(np.int32)
    qpos = np.hstack([rt.position[start], rt.quaternion[start], rt.joints[start]]).astype(np.float32)
    qpos = qpos + (noise * rng.standard_normal(qpos.shape)).astype(np.float32)
    qvel = np.hstack([rt.velocity[start], rt.angular_velocity[start], rt.joints_velocity[start]]).astype(np.float32)
    return qpos, qvel, start


@pytest.fixture(scope="session")
def gpu_env(rodent):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    envs = pkg("envs")
    rod = pkg("envs.rodent")
    return envs.RodentTracking(reference_clip=rodent["clip"], model=rodent["model"], device="cuda:0", **rod.RODENT_ENV_ARGS)
