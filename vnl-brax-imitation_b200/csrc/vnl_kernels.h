// vnl_kernels.h -- shared declarations between the kernels and the C ABI layer.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/vnl_b200.h"

namespace vnl {


struct Dims {
  int nq, nv, nu, na, nbody, njnt, ngeom, npair, ncon, nlimit, nefc, nM, nlevel, maxdepth, nroot;
  int solver, iterations, ls_iterations, eulerdamp;
  float timestep, gx, gy, gz, tolerance, ls_tolerance, impratio, meaninertia;
  int ktab_words;  // size of VNL_F_KTAB
  int ndslot;      // partial-sum slots of the descendant mat-vec program (VNL_KS_NDSLOT)
  int TA, TD;      // steps of the mat-vec lane programs (VNL_MH_TA / VNL_MH_TD)
  int stream;      // 1: M and K live in the global workspace (large models: buys residency); 0: resident in shared memory
                   // (small models whose residency is bound by the register file anyway).  Set by decide_stream().
  int naslot;      // partial-sum slots of the ancestor mat-vec program (VNL_MH_NASLOT)
  int env_warps;   // warps cooperating on one env (VNL_MH_ENV_WARPS): lane count of the mat-vec programs / 32
  // stage-dump offsets (layout of oracle.dump_layout)
  int dump_xpos, dump_xipos, dump_xanchor, dump_subtree_com, dump_cinert, dump_qM, dump_cvel, dump_passive, dump_con,
      dump_efc, dump_qacc, dump_total;
};

// Per-env shared-memory layout (float offsets); see make_layout for the regions and who lives in them when.
struct Lay {
  int qpos, qvel, act, ctrl, warm, cdof, Mdiag, Kdiag, rcom, qfrc_smooth, qacc_smooth, act_dot, ints;  // whole substep
  int Mn, H, jr;                                                          // Newton solver only (dense Hessian)
  int xpos, xquat, cvel;                                                  // region R0, kinematics .. constraint rows
  int Jaref, qacc, Ma, grad, Mgrad, search, Mv, qfrc_con;                 // region R0, solver .. integrator
  int xipos, xanchor, xaxis, cacc, t16;                                   // region R1, kinematic passes
  int part, tmpv, lim_dof, limrow_of_dof, cbody, crel, cframe, cmu, efcD, Jv;  // region R1, solves / constraint rows
  int K;                                                                  // region R1, factorisation workspace
  int Ms, Ks;                                                             // resident copies of M and K (stream == 0 only)
  int total;
};

struct Params {
  const uint32_t* model;
  const uint32_t* task;
  Dims dims;
  int B, nsteps;
  VnlState in, out;
  VnlState first;         // optional cached first state (AutoReset), first.qpos == nullptr when unused
  const float* first_obs;
  VnlEpisode episode;     // optional EpisodeWrapper bookkeeping, episode.steps_out == nullptr when unused
  const float* ctrl;
  VnlOutputs outputs;
  int32_t* stats;
  float* dump;
  long long* prof;  // optional [32] per-phase clock64 accumulators of one env (developer hook)
  int prof_env;
  float* work;      // inertia workspace (vnl_set_workspace), work_stride floats per resident env
  int work_stride;
  int lsgroups;     // lockstep groups per CTA (1 = the whole CTA)
  int lockstep;     // 0 = warps free-run, 1 = CTA barrier at every substep start, 2 = also before the integrator, 3 = at every phase boundary (default)
  VnlResample rs;   // mode 5 (reset over a list): the draw's key and counters, the list of envs to reset in rs.scratch (last: the
                    // parameter offsets of the other modes stay as they were)
};

struct LaunchInfo { int smem_bytes, warps_per_cta, ctas; };  // warps_per_cta = env groups per CTA

// floats of workspace per resident env: the A-order and the D-order copy of the off-diagonal entries of the inertia M,
// then the same two copies of its inverse factor K
inline int work_stride(const Dims& d) { return d.stream ? (2 * (d.TA + d.TD) * 32 * d.env_warps + 31) & ~31 : 0; }

// vnl_kernels.cu is compiled once per (env-group width -DVNL_EW=1, 2; inertia home -DVNL_STREAM=0, 1) into its own namespace.
// decide_stream() fills Dims::stream: resident inertia unless that would cost a resident env.
struct LayoutEntry { const char* name; int offset, size; };  // floats; for the layout / liveness test
#define VNL_DECL(ns) namespace ns { int layout_table(const Dims& d, LayoutEntry* out, int cap); void decide_stream(Dims& d); LaunchInfo launch_info(const Dims& d, int B); cudaError_t launch(int mode, const Params& p, cudaStream_t stream); }
VNL_DECL(ew1s0) VNL_DECL(ew1s1) VNL_DECL(ew2s0) VNL_DECL(ew2s1)
#undef VNL_DECL

inline void any_decide_stream(Dims& d) { if (d.env_warps == 2) ew2s1::decide_stream(d); else ew1s1::decide_stream(d); }
inline LaunchInfo any_launch_info(const Dims& d, int B) {
  if (d.env_warps == 2) return d.stream ? ew2s1::launch_info(d, B) : ew2s0::launch_info(d, B);
  return d.stream ? ew1s1::launch_info(d, B) : ew1s0::launch_info(d, B);
}
inline cudaError_t any_launch(int mode, const Params& p, cudaStream_t stream) {
  const bool st = p.dims.stream != 0;
  if (p.dims.env_warps == 2) return st ? ew2s1::launch(mode, p, stream) : ew2s0::launch(mode, p, stream);
  if (p.dims.env_warps == 1) return st ? ew1s1::launch(mode, p, stream) : ew1s0::launch(mode, p, stream);
  return cudaErrorInvalidValue;
}

}  // namespace vnl
