"""ctypes binding of libvnl_b200.so (the C ABI of include/vnl_b200.h) over torch CUDA tensors.

torch is plumbing only: device memory, streams.  There is NO CPU fallback: if the CUDA library
is missing or no GPU is visible, construction raises.
"""
from __future__ import annotations

import ctypes
import os
from typing import Dict, Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VNL_B200_LIB") or os.path.join(_HERE, "libvnl_b200.so")  # override: developer A/B builds

STATE_F = ("qpos", "qvel", "act", "qacc_warmstart", "xpos", "xquat", "subtree_com", "qfrc_actuator")
STATE_I = ("cur_frame", "sub_clip_frame", "clip_id")
OUT_F = ("obs", "traj", "reward", "done", "metrics")
VNL_TABLE_OFF, VNL_MAX_FIELDS = 64, 96  # include/vnl_b200.h
VNL_DATA_OFF = VNL_TABLE_OFF + 2 * VNL_MAX_FIELDS
VNL_XLA_STEP_NBUF = 32


class VnlState(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in STATE_F + STATE_I]


class VnlEpisode(ctypes.Structure):
    _fields_ = [("steps_in", ctypes.c_void_p), ("done_in", ctypes.c_void_p), ("steps_out", ctypes.c_void_p),
                ("truncation_out", ctypes.c_void_p), ("episode_length", ctypes.c_float)]


class VnlResample(ctypes.Structure):
    _fields_ = [("seed", ctypes.c_uint64), ("env_offset", ctypes.c_int32), ("start_frame_hi", ctypes.c_int32),
                ("noise_scale", ctypes.c_float), ("reset_count", ctypes.c_void_p), ("scratch", ctypes.c_void_p)]


class VnlOutputs(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in OUT_F + ("stats",)]


class VnlContext(ctypes.Structure):
    """Host-side call context (include/vnl_b200.h): header copies + the caller-owned workspace.  Read-only for the library."""
    _fields_ = [("model_hdr", ctypes.c_uint32 * VNL_DATA_OFF), ("task_hdr", ctypes.c_uint32 * VNL_TABLE_OFF),
                ("workspace", ctypes.c_void_p), ("workspace_bytes", ctypes.c_uint64)]


class VnlXlaOpaque(ctypes.Structure):
    """`opaque` of the XLA custom calls: batch size + the same header copies (stateless boundary)."""
    _fields_ = [("B", ctypes.c_int32), ("version", ctypes.c_int32), ("model_hdr", ctypes.c_uint32 * VNL_DATA_OFF),
                ("task_hdr", ctypes.c_uint32 * VNL_TABLE_OFF), ("workspace_bytes", ctypes.c_uint64)]


EXPORTS = ("vnl_step", "vnl_reset", "vnl_pipeline_step", "vnl_forward_dump", "vnl_dump_size", "vnl_check_model",
           "vnl_check_task", "vnl_context_init", "vnl_step_smem_bytes", "vnl_xla_step", "vnl_xla_reset", "vnl_xla_step_rc",
           "vnl_xla_reset_rc", "vnl_xla_make_opaque", "vnl_version", "vnl_ffma_probe", "vnl_step_profiled",
           "vnl_step_autoreset", "vnl_envs_per_cta", "vnl_resident_envs", "vnl_workspace_bytes", "vnl_step_training",
           "vnl_debug_layout", "vnl_process_clip", "vnl_step_training_resample")


IEEE_LIB_PATH = os.path.join(_HERE, "libvnl_b200_ieee.so")  # A/B twin: IEEE div / sqrt in the physics kernels (tests only)


def load_library(path: Optional[str] = None) -> ctypes.CDLL:
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: build it with __graft_entry__.build() (nvcc, sm_100a). "
                           "There is no CPU fallback for the product path.")
    lib = ctypes.CDLL(path)
    CTX, ST, OUT = ctypes.POINTER(VnlContext), ctypes.POINTER(VnlState), ctypes.POINTER(VnlOutputs)
    v, i, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_size_t
    lib.vnl_version.restype = ctypes.c_char_p
    lib.vnl_dump_size.restype = sz
    lib.vnl_dump_size.argtypes = [v]
    lib.vnl_step_smem_bytes.argtypes = [v]
    lib.vnl_envs_per_cta.argtypes = [v]
    lib.vnl_resident_envs.argtypes = [v]
    lib.vnl_workspace_bytes.restype = sz
    lib.vnl_workspace_bytes.argtypes = [v]
    lib.vnl_check_model.argtypes = [v, sz]
    lib.vnl_check_task.argtypes = [v, sz]
    lib.vnl_context_init.argtypes = [CTX, v, sz, v, sz]
    lib.vnl_step.argtypes = [CTX, v, v, i, ST, v, ST, OUT, v]
    lib.vnl_step_autoreset.argtypes = [CTX, v, v, i, ST, v, ST, OUT, ST, v, v]
    lib.vnl_step_training.argtypes = [CTX, v, v, i, ST, v, ST, OUT, ST, v, ctypes.POINTER(VnlEpisode), v]
    lib.vnl_step_training_resample.argtypes = [CTX, v, v, i, ST, v, ST, OUT, ctypes.POINTER(VnlEpisode), ctypes.POINTER(VnlResample), v]
    lib.vnl_reset.argtypes = [CTX, v, v, i, ST, ST, OUT, v]
    lib.vnl_pipeline_step.argtypes = [CTX, v, i, i, ST, v, ST, v, v]
    lib.vnl_forward_dump.argtypes = [CTX, v, i, ST, v, v, v]
    lib.vnl_step_profiled.argtypes = [CTX, v, v, i, ST, v, ST, OUT, v, v, i]
    lib.vnl_ffma_probe.argtypes = [i, i, v, v]
    for name in ("vnl_xla_step", "vnl_xla_reset"):
        getattr(lib, name).argtypes = [v, ctypes.POINTER(v), ctypes.c_char_p, sz, v]
        getattr(lib, name).restype = None
        getattr(lib, name + "_rc").argtypes = [v, ctypes.POINTER(v), ctypes.c_char_p, sz]
    lib.vnl_xla_make_opaque.argtypes = [CTX, i, ctypes.POINTER(VnlXlaOpaque)]
    # clip preprocessing on the GPU (SURVEY 8 row f4): qpos [n, T, nq] -> the ReferenceClip tables
    lib.vnl_process_clip.argtypes = [CTX, v, i, i, v, ctypes.c_float, ctypes.c_float, v, v, v, v, v]
    return lib


def _ptr(t) -> Optional[int]:
    return None if t is None else t.data_ptr()


class Engine:
    """Device-resident model / task blobs + typed wrappers of the C entry points.

    All tensors are torch CUDA tensors (fp32 / int32, contiguous, batch-major)."""

    def __init__(self, model_blob: np.ndarray, task_blob: Optional[np.ndarray] = None, device: str = "cuda:0",
                 lib_path: Optional[str] = None):
        import torch

        if not torch.cuda.is_available():
            raise RuntimeError("vnl_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        self.torch = torch
        self.lib = load_library(lib_path)
        self.device = torch.device(device)
        self.model_host = np.ascontiguousarray(model_blob, dtype=np.uint32)
        rc = self.lib.vnl_check_model(self.model_host.ctypes.data, self.model_host.nbytes)
        if rc:
            raise ValueError(f"bad model blob ({rc})")
        self.model_dev = torch.from_numpy(self.model_host.view(np.int32)).to(self.device)
        self.task_host = self.task_dev = None
        if task_blob is not None:
            self.task_host = np.ascontiguousarray(task_blob, dtype=np.uint32)
            rc = self.lib.vnl_check_task(self.task_host.ctypes.data, self.task_host.nbytes)
            if rc:
                raise ValueError(f"bad task blob ({rc})")
            self.task_dev = torch.from_numpy(self.task_host.view(np.int32)).to(self.device)
        # the call context: header copies + this engine's workspace.  Nothing is registered with the library.
        self.ctx = VnlContext()
        rc = self.lib.vnl_context_init(ctypes.byref(self.ctx), self.model_host.ctypes.data, self.model_host.nbytes,
                                       None if self.task_host is None else self.task_host.ctypes.data,
                                       0 if self.task_host is None else self.task_host.nbytes)
        if rc:
            raise ValueError(f"vnl_context_init failed ({rc})")
        from . import model_blob as mb
        self.dims = mb.read_dims(self.model_host)
        self.dump_size = int(self.lib.vnl_dump_size(self.model_host.ctypes.data))
        self.smem_bytes = int(self.lib.vnl_step_smem_bytes(self.model_host.ctypes.data))
        self.envs_per_cta = int(self.lib.vnl_envs_per_cta(self.model_host.ctypes.data))
        with torch.cuda.device(self.device):
            self.resident_envs = int(self.lib.vnl_resident_envs(self.model_host.ctypes.data))
            nbytes = int(self.lib.vnl_workspace_bytes(self.model_host.ctypes.data))
        # inertia workspace of the resident envs (L2-resident scratch the kernels address by CTA / env slot)
        self.workspace = torch.empty(max(nbytes, 4) // 4, dtype=torch.float32, device=self.device)
        self.ctx.workspace, self.ctx.workspace_bytes = self.workspace.data_ptr(), nbytes
        self._cref = ctypes.byref(self.ctx)
        if self.task_host is not None:
            self.obs_size = int(self.task_host[mb.C["VNL_TH_OBS_SIZE"]])
            self.traj_size = int(self.task_host[mb.C["VNL_TH_TRAJ_SIZE"]])
            self.n_frames = int(self.task_host[mb.C["VNL_TH_NFRAMES"]])
        self.launches = 0

    def close(self):
        """Nothing to release in the library (it keeps no state); kept for callers of the round-1 API."""

    def context_for_stream(self):
        """A second context with its OWN workspace: one workspace serves one stream at a time, so a caller that steps
        the same model from several streams / host threads takes one context per stream."""
        t = self.torch
        ctx = VnlContext()
        ctypes.memmove(ctypes.byref(ctx), ctypes.byref(self.ctx), ctypes.sizeof(VnlContext))
        work = t.empty_like(self.workspace)
        ctx.workspace = work.data_ptr()
        return ctx, work

    def xla_opaque(self, B: int, ctx: Optional[VnlContext] = None) -> bytes:
        """The `opaque` bytes of vnl_xla_step / vnl_xla_reset for a batch of B envs."""
        op = VnlXlaOpaque()
        rc = self.lib.vnl_xla_make_opaque(ctypes.byref(ctx or self.ctx), int(B), ctypes.byref(op))
        if rc:
            raise ValueError(f"vnl_xla_make_opaque failed ({rc})")
        return bytes(op)

    # ---- allocation helpers ---------------------------------------------------------------
    def alloc_state(self, B: int) -> Dict[str, "torch.Tensor"]:
        t, d, dev = self.torch, self.dims, self.device
        z = lambda *s: t.zeros(*s, dtype=t.float32, device=dev)
        return dict(qpos=z(B, d["nq"]), qvel=z(B, d["nv"]), act=z(B, d["na"]), qacc_warmstart=z(B, d["nv"]),
                    xpos=z(B, d["nbody"], 3), xquat=z(B, d["nbody"], 4), subtree_com=z(B, 3), qfrc_actuator=z(B, d["nv"]),
                    cur_frame=t.zeros(B, dtype=t.int32, device=dev), sub_clip_frame=t.zeros(B, dtype=t.int32, device=dev),
                    clip_id=t.zeros(B, dtype=t.int32, device=dev))

    def alloc_outputs(self, B: int) -> Dict[str, "torch.Tensor"]:
        t, dev = self.torch, self.device
        z = lambda *s: t.zeros(*s, dtype=t.float32, device=dev)
        return dict(obs=z(B, self.obs_size), traj=z(B, self.traj_size), reward=z(B), done=z(B), metrics=z(B, 7),
                    stats=t.zeros(B, 4, dtype=t.int32, device=dev))

    @staticmethod
    def _state(s: Dict) -> VnlState:
        st = VnlState()
        for k in STATE_F:
            v = s.get(k)
            if v is not None:
                assert v.is_contiguous() and v.dtype.is_floating_point and v.element_size() == 4, k
            setattr(st, k, _ptr(v))
        for k in STATE_I:
            v = s.get(k)
            if v is not None:
                assert v.is_contiguous() and v.element_size() == 4, k
            setattr(st, k, _ptr(v))
        return st

    @staticmethod
    def _outputs(o: Dict) -> VnlOutputs:
        out = VnlOutputs()
        for k in OUT_F:
            assert o[k].is_contiguous()
            setattr(out, k, _ptr(o[k]))
        out.stats = _ptr(o.get("stats"))
        return out

    def _stream(self) -> int:
        return self.torch.cuda.current_stream(self.device).cuda_stream

    def _check(self, rc: int, what: str):
        if rc:
            raise RuntimeError(f"{what} failed with code {rc}")
        self.launches += 1

    # ---- entry points -----------------------------------------------------------------------
    def step(self, state: Dict, action, out_state: Dict, outputs: Dict):
        B = state["qpos"].shape[0]
        a, b, o = self._state(state), self._state(out_state), self._outputs(outputs)
        assert action.is_contiguous() and action.shape == (B, self.dims["nu"])
        self._check(self.lib.vnl_step(self._cref, self.model_dev.data_ptr(), self.task_dev.data_ptr(), B, ctypes.byref(a),
                                      action.data_ptr(), ctypes.byref(b), ctypes.byref(o), self._stream()), "vnl_step")

    def step_autoreset(self, state: Dict, action, out_state: Dict, outputs: Dict, first: Dict, first_obs):
        """`vnl_step` + brax AutoResetWrapper in the same launch (restore `first` / `first_obs` where done)."""
        B = state["qpos"].shape[0]
        a, b, o, f = self._state(state), self._state(out_state), self._outputs(outputs), self._state(first)
        assert action.is_contiguous() and action.shape == (B, self.dims["nu"]) and first_obs.is_contiguous()
        self._check(self.lib.vnl_step_autoreset(self._cref, self.model_dev.data_ptr(), self.task_dev.data_ptr(), B, ctypes.byref(a),
                                                action.data_ptr(), ctypes.byref(b), ctypes.byref(o), ctypes.byref(f),
                                                first_obs.data_ptr(), self._stream()), "vnl_step_autoreset")

    def step_training(self, state: Dict, action, out_state: Dict, outputs: Dict, first: Dict, first_obs, steps, done_in,
                      steps_out, truncation, episode_length: float):
        """`vnl_step_training`: AutoResetWrapper(EpisodeWrapper(env)).step in one launch (action_repeat 1)."""
        B = state["qpos"].shape[0]
        a, b, o, f = self._state(state), self._state(out_state), self._outputs(outputs), self._state(first)
        assert action.is_contiguous() and action.shape == (B, self.dims["nu"]) and first_obs.is_contiguous()
        for t in (steps, done_in, steps_out, truncation):
            assert t.is_contiguous() and t.shape == (B,) and t.element_size() == 4 and t.dtype.is_floating_point
        ep = VnlEpisode(steps.data_ptr(), done_in.data_ptr(), steps_out.data_ptr(), truncation.data_ptr(), float(episode_length))
        self._check(self.lib.vnl_step_training(self._cref, self.model_dev.data_ptr(), self.task_dev.data_ptr(), B, ctypes.byref(a),
                                               action.data_ptr(), ctypes.byref(b), ctypes.byref(o), ctypes.byref(f),
                                               first_obs.data_ptr(), ctypes.byref(ep), self._stream()), "vnl_step_training")

    def step_training_resample(self, state: Dict, action, out_state: Dict, outputs: Dict, steps, done_in, steps_out, truncation,
                               episode_length: float, reset_count, scratch, seed: int, env_offset: int, start_frame_hi: int,
                               noise_scale: float):
        """`vnl_step_training_resample`: the training step without the first-state restore; done envs are reset in place to a
        fresh draw (clip, start frame in [0, start_frame_hi), qpos noise), keyed by `seed`, the global env index
        (`env_offset` + row) and `reset_count` (int32 [B], incremented per reset).  `scratch`: int32 [B + 1] for the done list."""
        t = self.torch
        B = state["qpos"].shape[0]
        a, b, o = self._state(state), self._state(out_state), self._outputs(outputs)
        assert action.is_contiguous() and action.shape == (B, self.dims["nu"])
        for x in (steps, done_in, steps_out, truncation):
            assert x.is_contiguous() and x.shape == (B,) and x.element_size() == 4 and x.dtype.is_floating_point
        assert reset_count.is_contiguous() and reset_count.shape == (B,) and reset_count.dtype == t.int32
        assert scratch.is_contiguous() and scratch.numel() >= B + 1 and scratch.dtype == t.int32
        ep = VnlEpisode(steps.data_ptr(), done_in.data_ptr(), steps_out.data_ptr(), truncation.data_ptr(), float(episode_length))
        rs = VnlResample(int(seed) & 0xFFFFFFFFFFFFFFFF, int(env_offset), int(start_frame_hi), float(noise_scale), reset_count.data_ptr(),
                         scratch.data_ptr())
        self._check(self.lib.vnl_step_training_resample(self._cref, self.model_dev.data_ptr(), self.task_dev.data_ptr(), B, ctypes.byref(a),
                                                        action.data_ptr(), ctypes.byref(b), ctypes.byref(o), ctypes.byref(ep),
                                                        ctypes.byref(rs), self._stream()), "vnl_step_training_resample")

    def reset(self, state: Dict, out_state: Dict, outputs: Dict):
        B = state["qpos"].shape[0]
        a, b, o = self._state(state), self._state(out_state), self._outputs(outputs)
        self._check(self.lib.vnl_reset(self._cref, self.model_dev.data_ptr(), self.task_dev.data_ptr(), B, ctypes.byref(a),
                                       ctypes.byref(b), ctypes.byref(o), self._stream()), "vnl_reset")

    def pipeline_step(self, state: Dict, ctrl, out_state: Dict, nsteps: int, stats=None):
        B = state["qpos"].shape[0]
        a, b = self._state(state), self._state(out_state)
        self._check(self.lib.vnl_pipeline_step(self._cref, self.model_dev.data_ptr(), B, int(nsteps), ctypes.byref(a), _ptr(ctrl),
                                               ctypes.byref(b), _ptr(stats), self._stream()), "vnl_pipeline_step")

    def forward_dump(self, state: Dict, ctrl=None):
        t = self.torch
        B = state["qpos"].shape[0]
        dump = t.empty(B, self.dump_size, dtype=t.float32, device=self.device)
        a = self._state(state)
        self._check(self.lib.vnl_forward_dump(self._cref, self.model_dev.data_ptr(), B, ctypes.byref(a), _ptr(ctrl), dump.data_ptr(),
                                              self._stream()), "vnl_forward_dump")
        return dump
