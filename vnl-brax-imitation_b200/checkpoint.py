"""Checkpoints of a training run (train.train): one directory per evaluation, written atomically, restored in place.

    checkpoint_dir/step_<env_steps>/
        meta.json         format version, env class and sizes, network shapes, hyperparameters, world size, schedule position
        learner.npz       flat params / Adam m / v (padding included), step_dev, bc_dev          (PPOLearner.state_dict)
        normalizer.npz    count, mean, summed_variance, std                                      (RunningStatistics.state_dict)
        policy.npz        the flax-named policy tree + normalizer/mean, normalizer/std: the deployable artefact (INTEGRATION.md)
        rank<r>.npz       rank r's rollout carry (rollout/...), trainer generator and counters (trainer/...); on rank 0 also the
                          evaluator's random streams (evaluator/...)

Every rank writes into step_<n>.tmp/; after a barrier rank 0 renames it to step_<n>.  A failure part-way leaves at most a .tmp
directory, which `latest` ignores, and never touches earlier checkpoints.  Plain file I/O of host arrays: the device side is
PPOLearner / RunningStatistics / Rollout / Trainer / Evaluator `state_dict` / `load_state_dict` (copies into the existing buffers).
"""
from __future__ import annotations

import json
import os
import re
import shutil
from typing import Dict, Optional

import numpy as np

FORMAT_VERSION = 1
_STEP = re.compile(r"^step_(\d+)$")


def step_dir(checkpoint_dir: str, env_steps: int) -> str:
    return os.path.join(checkpoint_dir, "step_%d" % int(env_steps))


def latest(checkpoint_dir: str) -> Optional[str]:
    """Path of the complete checkpoint with the most env steps (step_<n>; .tmp directories are skipped), or None."""
    if not os.path.isdir(checkpoint_dir):
        return None
    steps = [(int(m.group(1)), n) for n in os.listdir(checkpoint_dir)
             if (m := _STEP.match(n)) and os.path.isfile(os.path.join(checkpoint_dir, n, "meta.json"))]
    return os.path.join(checkpoint_dir, max(steps)[1]) if steps else None


def flatten(prefix: str, d: Dict[str, object]) -> Dict[str, np.ndarray]:
    return {prefix + "/" + k: np.asarray(v) for k, v in d.items()}


def unflatten(d, prefix: str) -> Dict[str, np.ndarray]:
    p = prefix + "/"
    return {k[len(p):]: d[k] for k in d if k.startswith(p)}


def write_npz(path: str, arrays: Dict[str, np.ndarray]) -> None:
    with open(path, "wb") as f:
        np.savez(f, **arrays)


def read_npz(path: str) -> Dict[str, np.ndarray]:
    with np.load(path, allow_pickle=False) as z:
        return {k: z[k] for k in z.files}


def save(checkpoint_dir: str, env_steps: int, rank: int, rank_arrays: Dict[str, np.ndarray], meta: Optional[dict] = None,
         shared: Optional[Dict[str, Dict[str, np.ndarray]]] = None, barrier=None) -> str:
    """Collective over the ranks: each passes its rank<r>.npz arrays; rank 0 also `meta` and the shared files
    ({"learner": ..., "normalizer": ..., "policy": ...}).  `barrier` synchronises the ranks (None: a single process).
    Returns the final directory."""
    sync = barrier or (lambda: None)
    final = step_dir(checkpoint_dir, env_steps)
    tmp = final + ".tmp"
    if rank == 0:
        shutil.rmtree(tmp, ignore_errors=True)  # the leftover of an interrupted write of this step
        os.makedirs(tmp)
    sync()
    try:
        write_npz(os.path.join(tmp, "rank%d.npz" % rank), rank_arrays)
        if rank == 0:
            for name, arrays in (shared or {}).items():
                write_npz(os.path.join(tmp, name + ".npz"), arrays)
            with open(os.path.join(tmp, "meta.json"), "w") as f:
                json.dump(meta, f, indent=1, sort_keys=True)
    except BaseException:
        if rank == 0:
            shutil.rmtree(tmp, ignore_errors=True)
        raise
    sync()
    if rank == 0:
        if os.path.isdir(final):  # the same step written again (a run repeated from an earlier checkpoint)
            shutil.rmtree(final)
        os.rename(tmp, final)
    sync()
    return final


def read_meta(path: str) -> dict:
    with open(os.path.join(path, "meta.json")) as f:
        return json.load(f)


def load(path: str, rank: int) -> Dict[str, Dict[str, np.ndarray]]:
    """{"meta", "learner", "normalizer", "rank"} of a checkpoint directory, as host arrays."""
    out = {"meta": read_meta(path)}
    for name in ("learner", "normalizer"):
        out[name] = read_npz(os.path.join(path, name + ".npz"))
    rank_file = os.path.join(path, "rank%d.npz" % rank)
    if not os.path.isfile(rank_file):
        raise ValueError("world_size: checkpoint %s has no state for rank %d" % (path, rank))
    out["rank"] = read_npz(rank_file)
    return out


def _first_difference(saved, current, path: str) -> Optional[str]:
    if isinstance(saved, dict) and isinstance(current, dict):
        for k in sorted(set(saved) | set(current)):
            d = _first_difference(saved.get(k), current.get(k), "%s[%s]" % (path, k) if path else k)
            if d:
                return d
        return None
    return None if saved == current else path


def check_meta(saved: dict, current: dict, fields) -> None:
    """Refuses a checkpoint whose `fields` differ from the run's, naming the first field (and entry) that differs."""
    current = json.loads(json.dumps(current))  # tuples -> lists, as the saved side
    for k in fields:
        d = _first_difference(saved.get(k), current.get(k), k)
        if d:
            raise ValueError("checkpoint does not match this run: %s is %r in the checkpoint, %r here"
                             % (d, _lookup(saved, d), _lookup(current, d)))


def _lookup(meta: dict, path: str):
    keys = re.findall(r"[^\[\]]+", path)
    for k in keys:
        meta = meta.get(k) if isinstance(meta, dict) else None
    return meta


def policy_arrays(policy_params: Dict[str, np.ndarray], mean, std) -> Dict[str, np.ndarray]:
    """policy.npz: the flax tree (names of policy.param_shapes) + the normaliser's mean / std."""
    out = {k: np.asarray(v, dtype=np.float32) for k, v in policy_params.items()}
    out["normalizer/mean"], out["normalizer/std"] = np.asarray(mean, dtype=np.float32), np.asarray(std, dtype=np.float32)
    return out


def load_policy(path: str):
    """(policy_params, {"mean", "std"}) of a policy.npz (or of the checkpoint directory holding one)."""
    if os.path.isdir(path):
        path = os.path.join(path, "policy.npz")
    a = read_npz(path)
    norm = unflatten(a, "normalizer")
    return {k: v for k, v in a.items() if not k.startswith("normalizer/")}, norm
