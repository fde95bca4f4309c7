// vnl_kernels.cu -- fused MJX-style physics + imitation reward/obs/termination step for sm_100a.
//
// ONE WARP PER ENVIRONMENT (optionally two: -DVNL_EW=2, a second instantiation in the same library).  The whole env
// step -- n_frames x (forward dynamics, constraint solve, semi-implicit Euler) and the clip-indexed reward /
// observation / trajectory window / termination -- runs in one launch with the env's working set (~20 KB for the
// rodent) resident in shared memory; the joint-space inertia alone lives in an L2-resident global workspace, laid out
// in the order the mat-vec lane programs consume it.  HBM is touched only for the state in and the state +
// observations out (~8.7 KB per env step).  A CTA holds as many envs as shared memory allows (10 rodents) plus one
// copy of the packed index tables (VNL_F_KTAB); the grid is persistent (one CTA per SM, envs dealt slot-major).
// Inside an env the lanes cooperate through shuffles and __syncwarp only; the CTA-wide barriers are NOT data
// dependencies: they keep the co-resident warps at the same phase of the substep so that they share instruction
// fetches (the substep's ~200 KB of SASS dwarfs the instruction caches) -- see `lockstep`.
//
// Formulation (differs from the dense one XLA executes for the reference, same mathematics):
//   * joint-space inertia kept tree-sparse (MuJoCo qM layout), factorised as L^T D L without fill-in; the
//     unit-triangular factor is inverted once per factorisation (the inverse has the same ancestor sparsity), so every
//     later M^-1 x is two parallel sparse mat-vecs instead of two serial triangular sweeps;
//   * the constraint Jacobian is never materialised: limit rows are one-hot, contact rows are frame . (v_lin + w x r)
//     of the contact's body, so J x and J^T f are sums over the ancestor chain of a handful of bodies; only ACTIVE
//     rows (pos < 0) are kept -- inactive rows contribute exactly zero to every solver quantity in the reference;
//   * kinematics composes per-body local joint transforms level by level; velocities / accelerations go down the
//     tree in one pass, composite inertias and RNE forces come back up in one pass (16 floats per body).
//
// Reference semantics restated: mjx.forward / mjx.step as reached from envs/rodent.py:148,181 and
// RodentTracking.step / reset (envs/rodent.py:119-470) -- see oracle/vnl_oracle.cpp, the CPU restatement these
// kernels are tested against.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>


#include "../../include/vnl_blob.h"
#include "vnl_device.cuh"
#include "vnl_kernels.h"

#ifndef VNL_EW
#define VNL_EW 1
#endif
#ifndef VNL_STREAM
#define VNL_STREAM 1
#endif
#ifdef VNL_IEEE  // A/B build (Makefile: libvnl_b200_ieee.so): exact reciprocal square root instead of the 2-ulp intrinsic
#define VNL_RSQRT(x) (1.0f / sqrtf(x))
#else
#define VNL_RSQRT(x) rsqrtf(x)
#endif
#define VNL_CAT2(a, b) a##b
#define VNL_CAT(a, b) VNL_CAT2(a, b)

namespace vnl {
namespace VNL_CAT(VNL_CAT(ew, VNL_EW), VNL_CAT(s, VNL_STREAM)) {  // one instantiation of everything below per (env-group width, inertia home): see Makefile

constexpr bool kStream = VNL_STREAM != 0;  // M and K streamed from the global workspace (1) or resident in shared memory (0): Dims::stream
constexpr int kEnvWarps = VNL_EW;          // warps cooperating on one env
constexpr int kEnvThreads = 32 * VNL_EW;   // = lanes of the mat-vec programs (VNL_MH_ENV_WARPS of the blob must agree)
// envs per CTA upper bound: one-warp groups are bounded by shared memory (10 rodents) or by the register file (16 warps x 128
// registers: humanoid, ant), two-warp groups by the register
// file (16 warps x 128 registers) and by the named barriers (1 .. 8 for the groups)
constexpr int kMaxEnvs = VNL_EW == 1 ? 16 : 8;
// floats per body of t16 (cinert / crb 10 + rne force 6): an ODD stride, so that lane-per-body accesses (cinert build,
// local rne, inert_mul / dot6 by dof_body) hit 32 different banks instead of 2 (stride 16 = 16-way conflicts)
#ifndef VNL_TS
#define VNL_TS 17
#endif
constexpr int kTS = VNL_TS;

#define LANE ((int)(threadIdx.x & 31))
#define FULLMASK 0xffffffffu
// kEnvWarps warps (kEnvThreads threads) cooperate on one env.  ETID = thread index inside the env's group.  Wide loops
// stride over kEnvThreads; reductions are done redundantly by every warp over all elements (identical results in each
// warp, fixed order, no exchange); level-serial passes simply leave the extra lanes idle.
#define ETID ((int)(threadIdx.x % kEnvThreads))
#define EWARP ((int)((threadIdx.x >> 5) % kEnvWarps))
#define ESLOT ((int)(threadIdx.x / kEnvThreads))

// barrier over the threads of one env (named barrier 1 + slot; barrier 0 stays the CTA-wide lockstep barrier)
__device__ __forceinline__ void env_sync() {
  if (kEnvWarps == 1) __syncwarp();
  else asm volatile("bar.sync %0, %1;" ::"r"(1 + ESLOT), "n"(kEnvThreads) : "memory");
}

// Lockstep barrier over one GROUP of env slots (named barriers 9..15; `groups` <= 7).  The env slots of a CTA are split
// into `groups` contiguous groups that each walk the substep in lockstep (shared instruction fetches) while the groups
// drift against each other, so that one group's shared-memory-bound phases overlap another's latency-bound ones.
__device__ __forceinline__ void group_sync(int groups) {
  if (groups <= 1) { __syncthreads(); return; }
  const int W = blockDim.x / kEnvThreads, g = ESLOT * groups / W;
  const int first = (g * W + groups - 1) / groups, last = ((g + 1) * W + groups - 1) / groups;
  asm volatile("bar.sync %0, %1;" ::"r"(9 + g), "r"((last - first) * kEnvThreads) : "memory");
}

__host__ __device__ inline int align4(int x) { return (x + 3) & ~3; }

// Per-env shared-memory layout.  Three parts: arrays that live through the whole substep, and two recycled regions whose
// tenants change with the phase of the substep (P1 kinematics, P2 com / cdof, P3 velocity + rne passes, P4 smooth forces,
// P5 inertia build, P6 factorise + invert, P7 smooth solve, P8 constraint rows, P9 solver, P10 integrator):
//   R0  P1-P8: xpos, xquat, cvel (P8 is their last reader; the caller's copies went to the output state in P1)
//       P9-P10: Jaref and the solver vectors qacc .. qfrc_con
//   R1  P1-P2: xipos, xanchor, xaxis | P3-P5: cacc, then crb * cdof ("fd") in the same place
//       P2-P5: t16 = cinert / crb (10) + rne force (6) per body, behind them
//       P5-P6, P10: F, the factorisation workspace (M, then L^T D L, then K), from behind fd / part+tmpv on (over t16)
//       P7-P10: part, tmpv (mat-vec scratch) at the very start (fd is dead by then)
//       P8-P9: the constraint rows (limit list, contacts, efcD, Jv) behind part / tmpv (F is dead: K went to the workspace)
// Only M_diag, K_diag survive of the inertia; M and K themselves are streamed from the global workspace.
__host__ __device__ inline void make_layout(const Dims& d, Lay& L) {
  int o = 0;
#define A(name, n) L.name = o; o += align4(n)
  A(qpos, d.nq); A(qvel, d.nv); A(act, d.na); A(ctrl, d.nu); A(warm, d.nv);
  A(cdof, d.nv * 6); A(Mdiag, d.nv); A(Kdiag, d.nv); A(rcom, d.nroot * 3);
  A(qfrc_smooth, d.nv); A(qacc_smooth, d.nv); A(act_dot, d.na); A(ints, 16);
  L.Ms = L.Ks = 0;
  if (!d.stream) { A(Ms, d.nM + 1); A(Ks, d.nM + 1); }
  L.Mn = L.H = L.jr = 0;
  if (d.solver == 2) { A(Mn, d.nM); A(H, d.nv * d.nv); A(jr, 3 * d.nv); }  // Newton: natural-order M, dense Hessian, row scratch
  const int r0 = o;
  A(xpos, d.nbody * 3); A(xquat, d.nbody * 4); A(cvel, d.nbody * 6);
  const int r0a = o;
  o = r0;
  A(Jaref, d.nefc); A(qacc, d.nv); A(Ma, d.nv); A(grad, d.nv); A(Mgrad, d.nv); A(search, d.nv); A(Mv, d.nv); A(qfrc_con, d.nv);
  if (r0a > o) o = r0a;
  const int r1 = o;
  A(xipos, d.nbody * 3); A(xanchor, d.njnt * 3); A(xaxis, d.njnt * 3);
  const int cacc_n = align4((d.nbody > d.nv ? d.nbody : d.nv) * 6);
  if (o - r1 < cacc_n) o = r1 + cacc_n;
  L.cacc = r1;
  A(t16, d.nbody * kTS);
  int r1end = o;
  o = r1;
  A(part, d.naslot + d.ndslot); A(tmpv, d.nv);
  const int scratch_end = o;
  A(lim_dof, d.nlimit); A(limrow_of_dof, d.nv); A(cbody, d.ncon); A(crel, d.ncon * 3); A(cframe, d.ncon * 6); A(cmu, d.ncon);
  A(efcD, d.nefc); A(Jv, d.nefc > 6 * d.ncon ? d.nefc : 6 * d.ncon);
  if (o > r1end) r1end = o;
  o = r1 + (cacc_n > scratch_end - r1 ? cacc_n : scratch_end - r1);  // F clears fd (P5) and part / tmpv (P10)
  A(K, d.nM + 40);  // + the zero slots the padded program terms and descendant lists point at
  if (o > r1end) r1end = o;
  o = r1end;
#undef A
  L.total = o;
}

// CTA-shared context (start of dynamic shared memory): dimensions, layout, field offsets and the BYTE offsets (from the
// start of shared memory) of the staged index tables.  Everything in shared memory is addressed as smem + offset so
// that the compiler emits 32-bit LDS / STS (a pointer stored in memory would come back generic).
struct __align__(16) Cta {
  Dims d;
  Lay L;
  const uint32_t* mb;
  uint32_t foff[VNL_F_MODEL_COUNT];
  uint32_t o_lvl_start, o_lvl_bp, o_parent, o_child_adr, o_child_list, o_body_dofadr, o_body_dofnum, o_body_tree, o_lastdof, o_sub_end,
      o_roots, o_mrow, o_mcol, o_dof_body, o_dpart_adr, o_apart_adr, o_madr, o_erow, o_elvl, o_desc_adr, o_desc_src, o_desc_k, o_ddof, o_dlvl, o_anc_start, o_kitem, o_klvl, o_prog_a, o_prog_d;
  int TA, TD, ndslot, nheight, lockstep, work_stride;
  float* work;
  long long* prof;
  int prof_env;
  __device__ __forceinline__ const int* fi(int f) const { return (const int*)(mb + foff[f]); }
  __device__ __forceinline__ const float* ff(int f) const { return (const float*)(mb + foff[f]); }
};
constexpr int kCtaFloats = (int)((sizeof(Cta) + 15) / 16 * 4);

// Every device function re-derives its view of shared memory from the `smem` symbol: c = CTA context, s = this warp's
// env slice (float offset `so`).
#define VNL_SMEM                                                  \
  extern __shared__ __align__(16) float smem[];                    \
  const Cta& c = *reinterpret_cast<const Cta*>(smem);              \
  float* const s = smem + so;
#define TB8(name) (reinterpret_cast<const uint8_t*>(smem) + c.o_##name)
#define TB16(name) reinterpret_cast<const uint16_t*>(reinterpret_cast<const uint8_t*>(smem) + c.o_##name)
#define TB32(name) reinterpret_cast<const uint32_t*>(reinterpret_cast<const uint8_t*>(smem) + c.o_##name)

// Phase clocks of tools/gpu_prof.py.  The object is passed BY VALUE through the (noinline) phase functions: by reference it had an
// address, lived in local memory, and every mark() of a production launch paid a local load for its null test (1.1 % of the stall
// samples, long_scoreboard, 116 of the kernel's 195 local-memory instructions).  The running time stamp sits in the env's `ints` slots.
struct Prof {
  long long* p;
  int t0o;  // float offset (in shared memory) of the 8-byte time stamp
  __device__ __forceinline__ void mark(int i) const {
    if (p) {
      extern __shared__ __align__(16) float smem[];
      env_sync();
      if (ETID == 0) { long long* t0 = reinterpret_cast<long long*>(smem + t0o); const long long t = clock64(); p[i] += t - *t0; *t0 = t; }
    }
  }
};

// ---------------------------------------------------------------------------------------------------------------------
// sparse-inertia helpers (one env group).  Vector arguments are float offsets into the env slice.
// ---------------------------------------------------------------------------------------------------------------------
// One section of a lane program: part[slot] = sum over the lane's terms of V[entry] * x[index] (see VnlKtab).
// A program is stored as [T / 4][lanes][4] words: the four consecutive steps of a lane sit in one 16-byte word, so a
// lane fetches them (and, from the workspace copies, their four V operands) with one 128-bit load.  T is a multiple
// of 8 (host pads).  All loads of a batch are issued before any partial sum is flushed.
#define VNL_LDV(w) (*reinterpret_cast<const float*>(Vb + ((w) & 0x3ffcu)))
#define VNL_LDX(w) (*reinterpret_cast<const float*>(xb + (((w) >> 14) & 0x3fcu)))
#define VNL_FLUSHTO(pt, w) if ((w) < 0xff000000u) { (pt)[(w) >> 24] = acc; acc = 0.0f; }
__device__ __forceinline__ void spmv_section(const uint32_t* __restrict__ prog, int T, const float* __restrict__ V,
                                             const float* __restrict__ x, float* __restrict__ part) {
  const char* Vb = reinterpret_cast<const char*>(V);
  const char* xb = reinterpret_cast<const char*>(x);
  const uint4* pp = reinterpret_cast<const uint4*>(prog) + ETID;
  float acc = 0.0f;
  for (int t = 0; t < T; t += 4, pp += kEnvThreads) {
    const uint4 w = *pp;
    const float v0 = VNL_LDV(w.x), x0 = VNL_LDX(w.x), v1 = VNL_LDV(w.y), x1 = VNL_LDX(w.y);
    const float v2 = VNL_LDV(w.z), x2 = VNL_LDX(w.z), v3 = VNL_LDV(w.w), x3 = VNL_LDX(w.w);
    acc += v0 * x0; VNL_FLUSHTO(part, w.x)
    acc += v1 * x1; VNL_FLUSHTO(part, w.y)
    acc += v2 * x2; VNL_FLUSHTO(part, w.z)
    acc += v3 * x3; VNL_FLUSHTO(part, w.w)
  }
}

// The joint-space inertia M lives in GLOBAL memory (L2), one copy per mat-vec program, in the order the program's lanes
// consume it: word (t, lane) of the copy is the V operand of program word (t, lane), same [T / 4][lanes][4] packing.
// Every thread only ever reads the words it wrote itself, so no fence is needed.  Loads / stores bypass L1 (.cg).
__device__ __forceinline__ float* slot_work(const Cta& c) {
  return c.work + (size_t)(blockIdx.x * (blockDim.x / kEnvThreads) + ESLOT) * (size_t)c.work_stride;
}
__device__ __forceinline__ void spill_section(const uint32_t* __restrict__ prog, int T, const float* __restrict__ V, float* __restrict__ g) {
  const char* Vb = reinterpret_cast<const char*>(V);
  const uint4* pp = reinterpret_cast<const uint4*>(prog) + ETID;
  float4* gp = reinterpret_cast<float4*>(g) + ETID;
  for (int t = 0; t < T; t += 4, pp += kEnvThreads, gp += kEnvThreads) {
    const uint4 w = *pp;
    __stcg(gp, make_float4(VNL_LDV(w.x), VNL_LDV(w.y), VNL_LDV(w.z), VNL_LDV(w.w)));
  }
}
// the inverse of spill_section for the ancestor program (it covers every off-diagonal entry exactly once; padding
// words point at the zero slot `pad` and are skipped)
__device__ __forceinline__ void restore_section(const uint32_t* __restrict__ prog, int T, float* __restrict__ V, const float* __restrict__ g, uint32_t pad) {
  char* Vb = reinterpret_cast<char*>(V);
  const uint4* pp = reinterpret_cast<const uint4*>(prog) + ETID;
  const float4* gp = reinterpret_cast<const float4*>(g) + ETID;
  for (int t = 0; t < T; t += 4, pp += kEnvThreads, gp += kEnvThreads) {
    const uint4 w = *pp;
    const float4 v = __ldcg(gp);
    const uint32_t e0 = w.x & 0x3ffcu, e1 = w.y & 0x3ffcu, e2 = w.z & 0x3ffcu, e3 = w.w & 0x3ffcu;
    if (e0 != pad) *reinterpret_cast<float*>(Vb + e0) = v.x;
    if (e1 != pad) *reinterpret_cast<float*>(Vb + e1) = v.y;
    if (e2 != pad) *reinterpret_cast<float*>(Vb + e2) = v.z;
    if (e3 != pad) *reinterpret_cast<float*>(Vb + e3) = v.w;
  }
}
// spmv_section with the V operands streamed from the workspace copy: eight terms (two 128-bit words) per batch, three
// batches of V words in flight (L2 latency is several batches long).  Can walk the ancestor and the descendant program
// back to back -- they and their workspace copies are contiguous -- so the stream never drains in between (T = TA + TD, a
// multiple of 8).  The flush slots of the steps from TA on are offset by `dslot0`.
__device__ __forceinline__ void spmv_stream_g(const uint32_t* __restrict__ prog, int T, int TA, const float* __restrict__ g,
                                              const float* __restrict__ x, float* __restrict__ part, int dslot0) {
  const char* xb = reinterpret_cast<const char*>(x);
  const uint4* pp = reinterpret_cast<const uint4*>(prog) + ETID;  // running pointers: every access is base + immediate
  const float4* gq = reinterpret_cast<const float4*>(g) + ETID;
  float acc = 0.0f;
  const float4 z4 = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  float4 q0a = __ldcg(gq), q0b = __ldcg(gq + kEnvThreads);
  float4 q1a = 8 < T ? __ldcg(gq + 2 * kEnvThreads) : z4, q1b = 8 < T ? __ldcg(gq + 3 * kEnvThreads) : z4;
  float4 q2a = 16 < T ? __ldcg(gq + 4 * kEnvThreads) : z4, q2b = 16 < T ? __ldcg(gq + 5 * kEnvThreads) : z4;
  gq += 6 * kEnvThreads;
#define VNL_BATCH(qa, qb, t0)                                                                     \
  if ((t0) < T) {                                                                                 \
    const float4 va = qa, vb = qb;                                                                \
    const uint4 wa = pp[0], wb = pp[kEnvThreads];                                                 \
    if ((t0) + 24 < T) { qa = __ldcg(gq); qb = __ldcg(gq + kEnvThreads); }                        \
    pp += 2 * kEnvThreads; gq += 2 * kEnvThreads;                                                 \
    const float x0 = VNL_LDX(wa.x), x1 = VNL_LDX(wa.y), x2 = VNL_LDX(wa.z), x3 = VNL_LDX(wa.w);   \
    const float x4 = VNL_LDX(wb.x), x5 = VNL_LDX(wb.y), x6 = VNL_LDX(wb.z), x7 = VNL_LDX(wb.w);   \
    float* const pt = (t0) >= TA ? part + dslot0 : part;                                          \
    acc += va.x * x0; VNL_FLUSHTO(pt, wa.x)                                                       \
    acc += va.y * x1; VNL_FLUSHTO(pt, wa.y)                                                       \
    acc += va.z * x2; VNL_FLUSHTO(pt, wa.z)                                                       \
    acc += va.w * x3; VNL_FLUSHTO(pt, wa.w)                                                       \
    acc += vb.x * x4; VNL_FLUSHTO(pt, wb.x)                                                       \
    acc += vb.y * x5; VNL_FLUSHTO(pt, wb.y)                                                       \
    acc += vb.z * x6; VNL_FLUSHTO(pt, wb.z)                                                       \
    acc += vb.w * x7; VNL_FLUSHTO(pt, wb.w)                                                       \
  }
  for (int t = 0; t < T; t += 24) {
    VNL_BATCH(q0a, q0b, t)
    VNL_BATCH(q1a, q1b, t + 8)
    VNL_BATCH(q2a, q2b, t + 16)
  }
#undef VNL_BATCH
}
#undef VNL_LDV
#undef VNL_LDX
#undef VNL_FLUSHTO

// out = M x   (tree-sparse symmetric M: diagonal + strict-ancestor terms + descendant terms)
__device__ __noinline__ void mul_m(int so, int xo, int outo) {
  VNL_SMEM
  const int nv = c.d.nv, lane = LANE, tid = ETID;
  const float* const Mdiag = s + c.L.Mdiag;
  const float* const x = s + xo;
  float* const pa = s + c.L.part;
  float* const pd = pa + c.d.naslot;
  if (kStream) {
    spmv_stream_g(TB32(prog_a), c.TA + c.TD, c.TA, slot_work(c), x, pa, c.d.naslot);  // PROG_D follows PROG_A in the staged tables
  } else {
    spmv_section(TB32(prog_a), c.TA, s + c.L.Ms, x, pa);
    spmv_section(TB32(prog_d), c.TD, s + c.L.Ms, x, pd);
  }
  env_sync();
  const uint8_t* const dpa = TB8(dpart_adr);
  const uint8_t* const apa = TB8(apart_adr);
  float* const out = s + outo;
  for (int i = tid; i < nv; i += kEnvThreads) {
    float acc = Mdiag[i] * x[i];
    for (int q = apa[i]; q < apa[i + 1]; ++q) acc += pa[q];
    for (int q = dpa[i]; q < dpa[i + 1]; ++q) acc += pd[q];
    out[i] = acc;
  }
  env_sync();
}

// L^T D L factorisation in place in the K region, then K = L^-1 in place.  `damp` = false: the region already holds M
// (forward() builds it there); `damp` = true: M + dt * damping is first put back from the workspace copy and Mdiag.
// Leaves: K off-diagonals in L.K, 1 / D in the diagonal slots.
__device__ __noinline__ void factor(int so, bool damp, bool invert, Prof pf) {
  VNL_SMEM
  const int nv = c.d.nv, nM = c.d.nM, lane = LANE, tid = ETID, maxdepth = c.d.maxdepth;
  float* const F = s + c.L.K;
  const uint16_t* const madr = TB16(madr);
  const uint16_t* const anc_start = TB16(anc_start);
  const uint8_t* const mrow = TB8(mrow);
  const uint8_t* const mcol = TB8(mcol);
  if (damp) {
    const float* damping = c.ff(VNL_F_DOF_DAMPING);
    const float dt = c.d.timestep;
    if (kStream) {
      restore_section(TB32(prog_a), c.TA, F, slot_work(c), 4u * (uint32_t)nM);
    } else {
      for (int e = tid; e < nM; e += kEnvThreads) F[e] = s[c.L.Ms + e];
      env_sync();
    }
    for (int i = tid; i < nv; i += kEnvThreads) F[madr[i]] = s[c.L.Mdiag + i] + dt * damping[i];
    if (tid == 0) F[nM] = 0.0f;
    env_sync();
  }
  // zero slots behind the entries: the padded tails of the descendant lists read F[nM] * F[nM + c], c < 40
  for (int i = tid; i < 40; i += kEnvThreads) F[nM + i] = 0.0f;
  env_sync();
  // Left-looking elimination by dof height, in Cholesky form.  A final row k holds C[k][a] = F[k][a] / sqrt(D_k)
  // (a >= 1) and 1 / sqrt(D_k) in its diagonal slot, so that row j (entries c = 0 .. dj) receives from every descendant
  // k at distance a just  F[j][c] -= C[k][a] * C[k][a + c].  Rows of one height are independent: one barrier per
  // level.  Inside a row the lanes are (group g, column c): the groups share out the descendants and are summed by
  // shuffles; the accumulation stays in registers, so no load ever waits on a store and the loop pipelines.
  const uint2* const erow = reinterpret_cast<const uint2*>(TB32(erow));
  const uint16_t* const elvl = TB16(elvl);
  const uint16_t* const dsrc = TB16(desc_src);
  {
    int r0 = elvl[0] & 255;
    for (int h = 0; h <= c.nheight; ++h) {
      const int r1 = elvl[h + 1] & 255;
      for (int r = r0 + EWARP; r < r1; r += kEnvWarps) {  // rows of the level are dealt to the env's warps
        const uint2 w = erow[r];
        const int base = w.x & 0x1fff, n = ((w.x >> 13) & 63) + 1, lg = (w.x >> 19) & 7;
        const int d1 = w.y >> 16;
        float* const Fb = F + base;
        if (n <= 32) {
          const int cc = lane & ((1 << lg) - 1), g = lane >> lg, G = 32 >> lg;
          const bool own = (g == 0) && (cc < n);
          const float* const Fc = F + (cc < n ? cc : 0);
          float acc = own ? Fb[cc] : 0.0f, accb = 0.0f;
          int t = (w.y & 0xffff) + g;
          for (; t < d1; t += 4 * G) {  // the host pads every list to a multiple of 4 G with the zero slot: no remainder
            const int s0 = dsrc[t], s1 = dsrc[t + G], s2 = dsrc[t + 2 * G], s3 = dsrc[t + 3 * G];
            const float u0 = F[s0], u1 = F[s1], u2 = F[s2], u3 = F[s3];
            const float v0 = Fc[s0], v1 = Fc[s1], v2 = Fc[s2], v3 = Fc[s3];
            acc = fmaf(-u0, v0, acc); accb = fmaf(-u1, v1, accb); acc = fmaf(-u2, v2, acc); accb = fmaf(-u3, v3, accb);
          }
          acc += accb;
          for (int o = 1 << lg; o < 32; o <<= 1) acc += __shfl_xor_sync(FULLMASK, acc, o);
          const float rs = VNL_RSQRT(__shfl_sync(FULLMASK, acc, 0));
          if (own) Fb[cc] = cc == 0 ? rs : acc * rs;
        } else {  // rows longer than a warp: lane owns columns lane and lane + 32 (few descendants down there)
          const bool on2 = lane + 32 < n;
          const int c1 = on2 ? lane + 32 : 0;
          float acc = Fb[lane], acc2 = on2 ? Fb[c1] : 0.0f;
          for (int t = w.y & 0xffff; t < d1; ++t) {
            const int s0 = dsrc[t];
            const float u = F[s0];
            acc = fmaf(-u, F[s0 + lane], acc);
            acc2 = fmaf(-u, F[s0 + c1], acc2);
          }
          const float rs = VNL_RSQRT(__shfl_sync(FULLMASK, acc, 0));
          Fb[lane] = lane == 0 ? rs : acc * rs;
          if (on2) Fb[c1] = acc2 * rs;
        }
      }
      r0 = r1;
      env_sync();
    }
  }
  pf.mark(16);
  // normalise rows: Lhat = C / sqrt(D), then 1 / D in the diagonal slots (they hold 1 / sqrt(D))
  for (int e = tid; e < nM; e += kEnvThreads) {
    const int b0 = madr[mrow[e]];
    if (e != b0) F[e] = F[e] * F[b0];
  }
  env_sync();
  for (int i = tid; i < nv; i += kEnvThreads) { const int m0 = madr[i]; const float rs = F[m0]; F[m0] = rs * rs; }
  env_sync();
  pf.mark(17);
  if (!invert) return;  // the caller solves by substitution (one right-hand side only)
  // K = Lhat^-1 in place by levels of dof depth:  K[i][cc] = -( Lhat[i][cc] + sum_{a<cc} Lhat[i][a] K[anc_a(i)][cc - a] ).
  // Items of a level are sorted by descending cc, so a later pass never reads a slot an earlier pass overwrote.
  const uint16_t* const kitem = TB16(kitem);
  const uint16_t* const klvl = TB16(klvl);
  int i0 = klvl[1];
  for (int dl = 1; dl <= maxdepth; ++dl) {
    const int i1 = klvl[dl + 1];
    for (int it0 = i0; it0 < i1; it0 += kEnvThreads) {
      const int it = it0 + tid;
      float val = 0.0f;
      float* dst = nullptr;
      if (it < i1) {
        const uint32_t w = kitem[it];
        const int cc = w & 255, base = madr[w >> 8];
        const float* const Fi = F + base;
        const uint16_t* const ai = anc_start + base;
        const float* const Fs = F + cc;  // K[anc_a][cc - a] = Fs[ai[a] - a]
        float a0 = Fi[cc], a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
        int a = 1;
        for (; a + 3 < cc; a += 4) {
          a0 += Fi[a] * Fs[ai[a] - a];
          a1 += Fi[a + 1] * Fs[ai[a + 1] - a - 1];
          a2 += Fi[a + 2] * Fs[ai[a + 2] - a - 2];
          a3 += Fi[a + 3] * Fs[ai[a + 3] - a - 3];
        }
        for (; a < cc; ++a) a0 += Fi[a] * Fs[ai[a] - a];
        val = -((a0 + a1) + (a2 + a3));
        dst = F + base + cc;
      }
      env_sync();
      if (dst) *dst = val;
      env_sync();
    }
    i0 = i1;
  }
  {  // K leaves shared memory: program-ordered copies for solve_m's two mat-vecs, 1 / D stays (Kdiag)
    if (kStream) {
      float* const wk = slot_work(c) + (c.TA + c.TD) * kEnvThreads;
      spill_section(TB32(prog_a), c.TA, F, wk);
      spill_section(TB32(prog_d), c.TD, F, wk + c.TA * kEnvThreads);
    } else {
      for (int e = tid; e <= nM; e += kEnvThreads) s[c.L.Ks + e] = F[e];  // incl. the zero slot the padded terms point at
    }
    for (int i = tid; i < nv; i += kEnvThreads) s[c.L.Kdiag + i] = F[madr[i]];
    env_sync();
  }
  pf.mark(18);
}

// out <- M^-1 x   via  K (D^-1 (K^T x)).
__device__ __noinline__ void solve_m(int so, int xo, int outo) {
  VNL_SMEM
  const int nv = c.d.nv, lane = LANE, tid = ETID;
  const float* const Kdiag = s + c.L.Kdiag;
  const float* const x = s + xo;
  float* const pa = s + c.L.part;
  float* const pd = pa + c.d.naslot;
  float* const tmp = s + c.L.tmpv;
  const uint8_t* const dpa = TB8(dpart_adr);
  const float* const wk = slot_work(c) + (c.TA + c.TD) * kEnvThreads;  // the program-ordered copies of K follow those of M
  if (kStream) spmv_stream_g(TB32(prog_d), c.TD, 0, wk + c.TA * kEnvThreads, x, pd, 0);
  else spmv_section(TB32(prog_d), c.TD, s + c.L.Ks, x, pd);
  env_sync();
  for (int j = tid; j < nv; j += kEnvThreads) {
    float acc = x[j];
    for (int q = dpa[j]; q < dpa[j + 1]; ++q) acc += pd[q];
    tmp[j] = acc * Kdiag[j];
  }
  env_sync();
  if (kStream) spmv_stream_g(TB32(prog_a), c.TA, c.TA, wk, tmp, pa, 0);
  else spmv_section(TB32(prog_a), c.TA, s + c.L.Ks, tmp, pa);
  env_sync();
  float* const out = s + outo;
  const uint8_t* const apa = TB8(apart_adr);
  for (int i = tid; i < nv; i += kEnvThreads) {
    float acc = tmp[i];
    for (int q = apa[i]; q < apa[i + 1]; ++q) acc += pa[q];
    out[i] = acc;
  }
  env_sync();
}

// out <- (L^T D L)^-1 x by substitution with the NON-inverted factor (Lhat off-diagonals, 1 / D in the diagonal slots):
// used where a factorisation serves a single right-hand side (the implicit-damping solve of forward.euler), which
// is cheaper than inverting the factor first.  mj_solveLD order: L^-T, D^-1, L^-1 -- both sweeps in gather form and
// level scheduled: L^-T by dof height (t[j] -= sum over descendants k of Lhat[k][a] t[k]), L^-1 by dof depth
// (t[i] -= sum over ancestors).  A level packs 32 >> lg rows per warp, each row on a 2^lg-lane segment.
__device__ __noinline__ void solve_ld(int so, int xo, int outo) {
  VNL_SMEM
  const int nv = c.d.nv, lane = LANE, tid = ETID;
  const float* const F = s + c.L.K;
  const float* const x = s + xo;
  float* const t = s + c.L.tmpv;
  const uint16_t* const madr = TB16(madr);
  const uint8_t* const mcol = TB8(mcol);
  for (int i = tid; i < nv; i += kEnvThreads) t[i] = x[i];
  env_sync();
  {
    const uint2* const erow = reinterpret_cast<const uint2*>(TB32(erow));
    const uint16_t* const elvl = TB16(elvl);
    const uint16_t* const dsrc = TB16(desc_src);
    const uint8_t* const dkk = TB8(desc_k);
    uint32_t lw = elvl[1];  // height 0 (leaves) has nothing to gather
    for (int h = 1; h <= c.nheight; ++h) {
      const uint32_t lw1 = elvl[h + 1];
      const int r0 = lw & 255, r1 = lw1 & 255, lg = lw >> 8;
      const int sl = lane & ((1 << lg) - 1), per = 32 >> lg, W = 1 << lg;
      for (int rs = r0 + EWARP * per; rs < r1; rs += per * kEnvWarps) {
        const int r = rs + (lane >> lg);
        float acc = 0.0f;
        int j = 0;
        if (r < r1) {
          const uint2 w = erow[r];
          j = w.x >> 22;
          const int d1 = w.y >> 16;
          for (int q = (w.y & 0xffff) + sl; q < d1; q += W) acc += F[dsrc[q]] * t[dkk[q]];
        }
        for (int o = W >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(FULLMASK, acc, o);
        if (r < r1 && sl == 0) t[j] -= acc;
      }
      lw = lw1;
      env_sync();
    }
  }
  for (int i = tid; i < nv; i += kEnvThreads) t[i] *= F[madr[i]];
  env_sync();
  {
    const uint8_t* const ddof = TB8(ddof);
    const uint16_t* const dlvl = TB16(dlvl);
    uint32_t lw = dlvl[0];
    for (int dl = 1; dl <= c.d.maxdepth; ++dl) {
      const uint32_t lw1 = dlvl[dl];
      const int r0 = lw & 255, r1 = lw1 & 255, lg = lw >> 8;
      const int sl = lane & ((1 << lg) - 1), per = 32 >> lg, W = 1 << lg;
      for (int rs = r0 + EWARP * per; rs < r1; rs += per * kEnvWarps) {
        const int r = rs + (lane >> lg);
        float acc = 0.0f;
        int i = 0;
        if (r < r1) {
          i = ddof[r];
          const int base = madr[i];
          for (int a = 1 + sl; a <= dl; a += W) acc += F[base + a] * t[mcol[base + a]];
        }
        for (int o = W >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(FULLMASK, acc, o);
        if (r < r1 && sl == 0) t[i] -= acc;
      }
      lw = lw1;
      env_sync();
    }
  }
  float* const out = s + outo;
  for (int i = tid; i < nv; i += kEnvThreads) out[i] = t[i];
  env_sync();
}

// ---------------------------------------------------------------------------------------------------------------------
// constraint Jacobian products on the compact active set
// ---------------------------------------------------------------------------------------------------------------------
// out[row] = (J x)[row].  Contacts: groups of G lanes walk the ancestor chain of the contact's body.
__device__ __noinline__ void jmul(int so, int xo, int outo) {
  VNL_SMEM
  const int* ints = (const int*)(s + c.L.ints);
  const int nl = ints[0], nc = ints[1], lane = LANE, tid = ETID;
  const float* const x = s + xo;
  float* const out = s + outo;
  const uint16_t* const madr = TB16(madr);
  const uint8_t* const mcol = TB8(mcol);
  const uint8_t* const lastdof = TB8(lastdof);
  const float* cdof = s + c.L.cdof;
  const int* cbody = (const int*)(s + c.L.cbody);
  const int* lim_dof = (const int*)(s + c.L.lim_dof);
  for (int r = tid; r < nl; r += kEnvThreads) { const int ld = lim_dof[r]; out[r] = ld < 0 ? -x[~ld] : x[ld]; }  // sign folded in: ~dof = upper limit
  if (nc > 0) {
    int G = 32;
    while (G > 1 && (32 / G) * kEnvWarps < nc) G >>= 1;
    const int per = 32 / G, sub = lane & (G - 1);
    for (int k0 = 0; k0 < nc; k0 += per * kEnvWarps) {  // contacts are dealt to the env's warps, `per` per warp per pass
      const int k = k0 + EWARP * per + lane / G;
      float sacc[6] = {0, 0, 0, 0, 0, 0};
      if (k < nc) {
        const int dl = lastdof[cbody[k]];
        if (dl != 0xFF) {
          const int ae = madr[dl + 1];
          for (int a = madr[dl] + sub; a < ae; a += G) {
            const int j = mcol[a];
            const float xj = x[j];
#pragma unroll
            for (int q = 0; q < 6; ++q) sacc[q] += cdof[j * 6 + q] * xj;
          }
        }
      }
      for (int o = G >> 1; o > 0; o >>= 1) {
#pragma unroll
        for (int q = 0; q < 6; ++q) sacc[q] += __shfl_xor_sync(FULLMASK, sacc[q], o);
      }
      if (k < nc && sub == 0) {
        const float* fr = s + c.L.cframe + 6 * k;  // [n, b]; the second tangent is n x b
        const V3 vel = v3(sacc[3], sacc[4], sacc[5]) + cross(v3(sacc[0], sacc[1], sacc[2]), ld3(s + c.L.crel + 3 * k));
        const V3 fn3 = ld3(fr), fb3 = ld3(fr + 3);
        const float un = dot(fn3, vel), u1 = dot(fb3, vel), u2 = dot(cross(fn3, fb3), vel);
        const float mu = s[c.L.cmu + k];
        float* o4 = out + nl + 4 * k;
        o4[0] = un + u1 * mu; o4[1] = un + u1 * -mu; o4[2] = un + u2 * mu; o4[3] = un + u2 * -mu;
      }
    }
  }
  env_sync();
}

// qfrc = J^T f with f[row] = -D Jaref [Jaref < 0]
__device__ __noinline__ void jtmul_force(int so) {
  VNL_SMEM
  const int* ints = (const int*)(s + c.L.ints);
  const int nl = ints[0], nc = ints[1], lane = LANE, tid = ETID, nv = c.d.nv;
  float* const qfrc = s + c.L.qfrc_con;
  float* const cwrench = s + c.L.Jv;  // per-contact wrench scratch: Jv is dead whenever the constraint forces are mapped back
  const uint8_t* const dof_body = TB8(dof_body);
  const uint8_t* const sub_end = TB8(sub_end);
  const float* D = s + c.L.efcD;
  const float* Jaref = s + c.L.Jaref;
  for (int k = tid; k < nc; k += kEnvThreads) {
    float f[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float ja = Jaref[nl + 4 * k + q];
      f[q] = (ja < 0.0f) ? -D[nl + 4 * k + q] * ja : 0.0f;
    }
    const float mu = s[c.L.cmu + k];
    const float fn = f[0] + f[1] + f[2] + f[3], f1 = mu * (f[0] - f[1]), f2 = mu * (f[2] - f[3]);
    const float* fr = s + c.L.cframe + 6 * k;
    const V3 fn3 = ld3(fr), fb3 = ld3(fr + 3);
    const V3 F = fn3 * fn + fb3 * f1 + cross(fn3, fb3) * f2;
    st3(cwrench + 6 * k, cross(ld3(s + c.L.crel + 3 * k), F));
    st3(cwrench + 6 * k + 3, F);
  }
  env_sync();
  const int* cbody = (const int*)(s + c.L.cbody);
  const int* limrow = (const int*)(s + c.L.limrow_of_dof);
  const int* lim_dof = (const int*)(s + c.L.lim_dof);
  for (int i = tid; i < nv; i += kEnvThreads) {
    const int b = dof_body[i], be = sub_end[b];
    const float* cd = s + c.L.cdof + 6 * i;
    float acc = 0.0f;
    for (int k = 0; k < nc; ++k) {
      const int cb = cbody[k];
      if (cb >= b && cb < be) acc += dot6(cd, cwrench + 6 * k);
    }
    const int r = limrow[i];
    if (r >= 0) {
      const float ja = Jaref[r];
      if (ja < 0.0f) acc += (lim_dof[r] < 0 ? -1.0f : 1.0f) * (-D[r] * ja);
    }
    qfrc[i] = acc;
  }
  env_sync();
}

// constraint._kbi  (the impedance power is 1 or 2 on every reference model: no powf on those paths)
__device__ __noinline__ float imp_pow(float x, float p) { return powf(x, p); }
__device__ __forceinline__ void kbi(const Dims& d, float sr0, float sr1, const float* solimp, float pos, float& k, float& b, float& imp) {
  const float timeconst = fmaxf(sr0, 2.0f * d.timestep), dampratio = sr1;
  const float dmin = fminf(fmaxf(solimp[0], VNL_MINIMP), VNL_MAXIMP), dmax = fminf(fmaxf(solimp[1], VNL_MINIMP), VNL_MAXIMP);
  const float width = fmaxf(VNL_MINVAL, solimp[2]), mid = fminf(fmaxf(solimp[3], VNL_MINIMP), VNL_MAXIMP), power = fmaxf(1.0f, solimp[4]);
  k = 1.0f / (dmax * dmax * timeconst * timeconst * dampratio * dampratio);
  b = 2.0f / (dmax * timeconst);
  if (sr0 <= 0.0f) k = -sr0 / (dmax * dmax);
  if (sr1 <= 0.0f) b = -sr1 / dmax;
  const float x = fabsf(pos) / width;
  float imp_a, imp_b;
  if (power == 1.0f) { imp_a = x; imp_b = 1.0f - (1.0f - x); }
  else if (power == 2.0f) { imp_a = (1.0f / mid) * (x * x); imp_b = 1.0f - (1.0f / (1.0f - mid)) * ((1.0f - x) * (1.0f - x)); }
  else { imp_a = (1.0f / imp_pow(mid, power - 1.0f)) * imp_pow(x, power); imp_b = 1.0f - (1.0f / imp_pow(1.0f - mid, power - 1.0f)) * imp_pow(1.0f - x, power); }
  const float imp_y = x < mid ? imp_a : imp_b;
  imp = dmin + imp_y * (dmax - dmin);
  imp = fminf(fmaxf(imp, dmin), dmax);
  if (x > 1.0f) imp = dmax;
}

// solver._update_gradient for the Newton solver: Mgrad = H^-1 grad with H = M + J^T diag(D [Jaref < 0]) J, dense
// (nv x nv) and Cholesky-factorised per call, as MJX does (opt.jacobian = dense on the reference path, envs/ant.py:50).
// The rows of J are never stored: a limit row is one-hot, the four pyramid rows of a contact are a +- mu b, a +- mu t
// with (a, b, t)_i = frame . (cdof_lin_i + cdof_ang_i x rel) on the dofs above the contact's body.
__device__ __noinline__ void newton_mgrad(int so) {
  VNL_SMEM
  const Lay& L = c.L;
  const int* ints = (const int*)(s + L.ints);
  const int nl = ints[0], nc = ints[1], nv = c.d.nv, nM = c.d.nM, tid = ETID, lane = LANE;
  float* const H = s + L.H;
  float* const jr = s + L.jr;
  const float* const D = s + L.efcD;
  const float* const Jaref = s + L.Jaref;
  const uint8_t* const mrow = TB8(mrow);
  const uint8_t* const mcol = TB8(mcol);
  for (int q = tid; q < nv * nv; q += kEnvThreads) H[q] = 0.0f;
  env_sync();
  for (int e = tid; e < nM; e += kEnvThreads) {
    const int i = mrow[e], j = mcol[e];
    const float v = s[L.Mn + e];
    H[i * nv + j] = v; H[j * nv + i] = v;
  }
  env_sync();
  const int* lim_dof = (const int*)(s + L.lim_dof);
  for (int r = tid; r < nl; r += kEnvThreads)  // one row per limited joint: distinct dofs, no collisions
    if (Jaref[r] < 0.0f) { const int ld = lim_dof[r], dof = ld < 0 ? ~ld : ld; H[dof * nv + dof] += D[r]; }
  env_sync();
  const int* cbody = (const int*)(s + L.cbody);
  const uint8_t* const dof_body = TB8(dof_body);
  const uint8_t* const sub_end = TB8(sub_end);
  for (int k = 0; k < nc; ++k) {
    const int cb = cbody[k], r = nl + 4 * k;
    const float* fr = s + L.cframe + 6 * k;
    const V3 fn3 = ld3(fr), fb3 = ld3(fr + 3), ft3 = cross(fn3, fb3), rel = ld3(s + L.crel + 3 * k);
    for (int i = tid; i < nv; i += kEnvThreads) {
      const int b = dof_body[i];
      float a = 0.0f, bb = 0.0f, t = 0.0f;
      if (cb >= b && cb < sub_end[b]) {
        const float* cd = s + L.cdof + 6 * i;
        const V3 p = ld3(cd + 3) + cross(ld3(cd), rel);
        a = dot(fn3, p); bb = dot(fb3, p); t = dot(ft3, p);
      }
      jr[i] = a; jr[nv + i] = bb; jr[2 * nv + i] = t;
    }
    env_sync();
    const float mu = s[L.cmu + k];
    const float w0 = Jaref[r] < 0.0f ? D[r] : 0.0f, w1 = Jaref[r + 1] < 0.0f ? D[r + 1] : 0.0f;
    const float w2 = Jaref[r + 2] < 0.0f ? D[r + 2] : 0.0f, w3 = Jaref[r + 3] < 0.0f ? D[r + 3] : 0.0f;
    for (int q = tid; q < nv * nv; q += kEnvThreads) {
      const int i = q / nv, j = q - i * nv;
      const float ai = jr[i], bi = mu * jr[nv + i], ti = mu * jr[2 * nv + i];
      const float aj = jr[j], bj = mu * jr[nv + j], tj = mu * jr[2 * nv + j];
      H[q] += w0 * (ai + bi) * (aj + bj) + w1 * (ai - bi) * (aj - bj) + w2 * (ai + ti) * (aj + tj) + w3 * (ai - ti) * (aj - tj);
    }
    env_sync();
  }
  // in-place Cholesky H = L L^T (lower triangle), right-looking
  for (int k = 0; k < nv; ++k) {
    const float dk = sqrtf(H[k * nv + k]);
    env_sync();
    if (tid == 0) H[k * nv + k] = dk;
    for (int i = k + 1 + tid; i < nv; i += kEnvThreads) H[i * nv + k] = H[i * nv + k] / dk;
    env_sync();
    const int m = nv - k - 1;
    for (int q = tid; q < m * m; q += kEnvThreads) {
      const int i = k + 1 + q / m, j = k + 1 + q % m;
      if (j <= i) H[i * nv + j] -= H[i * nv + k] * H[j * nv + k];
    }
    env_sync();
  }
  // Mgrad = L^-T L^-1 grad
  float* const y = s + L.Mgrad;
  for (int i = tid; i < nv; i += kEnvThreads) y[i] = s[L.grad + i];
  env_sync();
  for (int k = 0; k < nv; ++k) {
    const float yk = y[k] / H[k * nv + k];
    env_sync();
    if (tid == 0) y[k] = yk;
    for (int i = k + 1 + tid; i < nv; i += kEnvThreads) y[i] -= H[i * nv + k] * yk;
    env_sync();
  }
  for (int k = nv - 1; k >= 0; --k) {
    const float yk = y[k] / H[k * nv + k];
    env_sync();
    if (tid == 0) y[k] = yk;
    for (int i = tid; i < k; i += kEnvThreads) y[i] -= H[k * nv + i] * yk;
    env_sync();
  }
  (void)lane;
}

// solver state carried between _update_constraint calls
struct Sol { float cost, prev_cost, gauss, gradnorm; bool stop; };  // passed and returned by value: registers, not local memory

// solver._update_constraint + _update_gradient (CG: Mgrad = M^-1 grad)
// `last`: no iteration can follow (the iteration budget is spent).  Returns true when the solver stops after this update
// -- budget spent or converged by the test the next loop top would make -- in which case the gradient solve, whose
// only consumer is the next search direction, is skipped (the reference computes and discards it).
__device__ __noinline__ Sol update_constraint(int so, Sol st, Prof pf, bool last, float scale) {
  VNL_SMEM
  const Lay& L = c.L;
  const int* ints = (const int*)(s + L.ints);
  const int nrow = ints[0] + 4 * ints[1], lane = LANE, tid = ETID, nv = c.d.nv;
  float* qfrc_con = s + L.qfrc_con;
  pf.mark(11);
  jtmul_force(so);
  pf.mark(22);
  float v0 = 0.0f, v1 = 0.0f, g = 0.0f;
  // CG: the gradient goes straight into solve_m's scratch vector (solve_m is safe in place) and is otherwise re-formed as
  // Ma - qfrc_smooth - qfrc_constraint where it is read: its shared-memory slot holds the previous M^-1 grad instead
  const int go = c.d.solver == 2 ? L.grad : L.tmpv;
  // reductions: every warp of the env sums ALL elements (same order, same result, no exchange); the grad stores of the
  // warps carry identical values
  for (int r = lane; r < nrow; r += 32) { const float ja = s[L.Jaref + r]; if (ja < 0.0f) v0 += s[L.efcD + r] * ja * ja; }
  for (int i = lane; i < nv; i += 32) {
    const float ma = s[L.Ma + i], qs = s[L.qfrc_smooth + i];
    v1 += (ma - qs) * (s[L.qacc + i] - s[L.qacc_smooth + i]);
    const float gi = ma - qs - qfrc_con[i];
    s[go + i] = gi;
    g += gi * gi;
  }
  { float a4[4] = {v0, v1, g, 0.0f}; warp_sum_n<4>(a4); v0 = a4[0]; v1 = a4[1]; g = a4[2]; }
  st.gauss = 0.5f * v1;
  st.prev_cost = st.cost;
  st.cost = 0.5f * v0 + st.gauss;
  st.gradnorm = sqrtf(g);
  env_sync();
  pf.mark(23);
  bool stop = last;
  if (c.d.iterations != 1) stop |= ((st.prev_cost - st.cost) / scale < c.d.tolerance) || (st.gradnorm / scale < c.d.tolerance);
  if (!stop) {
    if (c.d.solver == 2) newton_mgrad(so);
    else solve_m(so, L.tmpv, L.Mgrad);
  }
  pf.mark(24);
  st.stop = stop;
  return st;
}

struct LSP { float alpha, cost, d0, d1; };

// ---------------------------------------------------------------------------------------------------------------------
// mjx.forward for the env held in this warp's shared-memory slice
// ---------------------------------------------------------------------------------------------------------------------
// `gx` != nullptr (the last substep of a call): xpos / xquat / qfrc_actuator of this forward pass are the ones the caller
// sees; they are stored to the env's rows of the output state right where they are produced (gx -> xpos, gq -> xquat,
// gf -> qfrc_actuator), because their shared-memory homes are recycled by the solver.
// `kin_only`: stop after smooth.kinematics (the clip-preprocessing mode: process_clip's set_position runs kinematics only).
template <bool DUMP>
__device__ __noinline__ void forward(int so, float* dump, Prof pf, float* gx, float* gq, float* gf, bool kin_only = false) {
  VNL_SMEM
  const Dims& d = c.d;
  const Lay& L = c.L;
  const int lane = LANE, tid = ETID;
  int* ints = (int*)(s + L.ints);
  int* stats = ints + 4;
  const bool ls3 = c.lockstep >= 3;  // CTA-uniform: barriers at every phase boundary
  const bool lsi = c.lockstep == 3 || c.lockstep == 5;  // ... and at the top of every solver iteration (VNL_LOCKSTEP=4: phases only; 5: every other iteration)
  const int lsi_mask = c.lockstep == 5 ? 1 : 0;
  const uint8_t* const lvl_start = TB8(lvl_start);
  const uint16_t* const lvl_bp = TB16(lvl_bp);
  const uint8_t* const body_tree = TB8(body_tree);
  const uint8_t* const dof_body = TB8(dof_body);

  // ---- smooth.kinematics ------------------------------------------------------------------------------------------
  // (1) per body, in parallel: the body's pose in its PARENT frame after its own joints (lq, lp) and each joint's
  //     anchor / axis in the parent frame; (2) compose down the tree level by level; (3) joint frames to world.
  {
    const int* jntadr = c.fi(VNL_F_BODY_JNTADR);
    const int* jntnum = c.fi(VNL_F_BODY_JNTNUM);
    const int* jtype = c.fi(VNL_F_JNT_TYPE);
    const int* jqadr = c.fi(VNL_F_JNT_QPOSADR);
    const float* bpos = c.ff(VNL_F_BODY_POS);
    const float* bquat = c.ff(VNL_F_BODY_QUAT);
    const float* jpos = c.ff(VNL_F_JNT_POS);
    const float* jaxis = c.ff(VNL_F_JNT_AXIS);
    const float* qpos0 = c.ff(VNL_F_QPOS0);
    for (int b = tid; b < d.nbody; b += kEnvThreads) {
      Q4 lq; lq.w = 1.0f; lq.x = lq.y = lq.z = 0.0f;
      V3 lp = v3(0.0f, 0.0f, 0.0f);
      if (b > 0) {
        lq = ld4(bquat + 4 * b);
        lp = ld3(bpos + 3 * b);
        const int ja = jntadr[b], jn = jntnum[b];
        for (int jj = 0; jj < jn; ++jj) {
          const int j = ja + jj, qa = jqadr[j];
          if (jtype[j] == 0) {  // free joint (its body hangs off the world): pose straight from qpos, quat normalised + written back
            lp = ld3(s + L.qpos + qa);
            lq = quat_normalize(ld4(s + L.qpos + qa + 3));
            st4(s + L.qpos + qa + 3, lq);
            st3(s + L.xanchor + 3 * j, lp);
            st3(s + L.xaxis + 3 * j, v3(0.0f, 0.0f, 1.0f));
          } else {
            const V3 jp = ld3(jpos + 3 * j), jax = ld3(jaxis + 3 * j);
            const V3 anchor = rotate(jp, lq) + lp;
            st3(s + L.xanchor + 3 * j, anchor);
            st3(s + L.xaxis + 3 * j, rotate(jax, lq));
            lq = quat_mul(lq, axis_angle_quat(jax, s[L.qpos + qa] - qpos0[qa]));
            lp = anchor - rotate(jp, lq);
          }
        }
      }
      st4(s + L.xquat + 4 * b, lq);
      st3(s + L.xpos + 3 * b, lp);
    }
    env_sync();
    pf.mark(25);
    int k0 = lvl_start[1];  // level 0 (children of the world) is already in world coordinates
    for (int lv = 1; lv < d.nlevel; ++lv) {
      const int k1 = lvl_start[lv + 1];
      if (k0 + tid < k1) {
        const uint32_t bp = lvl_bp[k0 + tid];
        const int b = bp & 255, p = bp >> 8;
        const Q4 pq = ld4(s + L.xquat + 4 * p);
        const V3 pp = ld3(s + L.xpos + 3 * p);
        const Q4 lq = ld4(s + L.xquat + 4 * b);
        const V3 lp = ld3(s + L.xpos + 3 * b);
        st4(s + L.xquat + 4 * b, quat_mul(pq, lq));
        st3(s + L.xpos + 3 * b, pp + rotate(lp, pq));
      }
      k0 = k1;
      env_sync();
    }
    pf.mark(26);
    if (gx) {
      for (int i = tid; i < d.nbody * 3; i += kEnvThreads) gx[i] = s[L.xpos + i];
      for (int i = tid; i < d.nbody * 4; i += kEnvThreads) gq[i] = s[L.xquat + i];
    }
    if (DUMP) {
      for (int i = tid; i < d.nbody * 3; i += kEnvThreads) dump[d.dump_xpos + i] = s[L.xpos + i];
      for (int i = tid; i < d.nbody * 4; i += kEnvThreads) dump[d.dump_xpos + d.nbody * 3 + i] = s[L.xquat + i];
    }
    const int* jbody = c.fi(VNL_F_JNT_BODYID);
    for (int j = tid; j < d.njnt; j += kEnvThreads) {
      const int p = TB8(parent)[jbody[j]];
      if (p > 0) {
        const Q4 pq = ld4(s + L.xquat + 4 * p);
        st3(s + L.xanchor + 3 * j, ld3(s + L.xpos + 3 * p) + rotate(ld3(s + L.xanchor + 3 * j), pq));
        st3(s + L.xaxis + 3 * j, rotate(ld3(s + L.xaxis + 3 * j), pq));
      }
    }
    env_sync();
  }
  pf.mark(0);
  if (kin_only) return;
  if (ls3) __syncthreads();
  // ---- smooth.com_pos: xipos, tree COM, cinert (t16[0..9]), cdof ------------------------------------------------------
  const int* dof_jnt = c.fi(VNL_F_DOF_JNTID);
  const int* jtype = c.fi(VNL_F_JNT_TYPE);
  const int* jdofadr = c.fi(VNL_F_JNT_DOFADR);
  {
    const float* ipos = c.ff(VNL_F_BODY_IPOS);
    const float* mass = c.ff(VNL_F_BODY_MASS);
    for (int b = tid; b < d.nbody; b += kEnvThreads)
      st3(s + L.xipos + 3 * b, ld3(s + L.xpos + 3 * b) + rotate(ld3(ipos + 3 * b), ld4(s + L.xquat + 4 * b)));
    env_sync();
    for (int t = 0; t < d.nroot; ++t) {  // subtree COM of each tree root = mass-weighted mean over its id range
      const int rb = TB8(roots)[t], re = TB8(sub_end)[rb];
      float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
      for (int q = rb + lane; q < re; q += 32) {
        const float mq = mass[q];
        a0 += s[L.xipos + 3 * q] * mq; a1 += s[L.xipos + 3 * q + 1] * mq; a2 += s[L.xipos + 3 * q + 2] * mq; a3 += mq;
      }
      a0 = warp_sum(a0); a1 = warp_sum(a1); a2 = warp_sum(a2); a3 = warp_sum(a3);
      if (lane < 3) {
        const float a = lane == 0 ? a0 : (lane == 1 ? a1 : a2);
        s[L.rcom + 3 * t + lane] = (a3 < VNL_MINVAL) ? s[L.xipos + 3 * rb + lane] : a / fmaxf(a3, VNL_MINVAL);
      }
    }
    env_sync();
    const float* iquat = c.ff(VNL_F_BODY_IQUAT);
    const float* inertia = c.ff(VNL_F_BODY_INERTIA);
    for (int b = tid; b < d.nbody; b += kEnvThreads) {
      float* ci = s + L.t16 + kTS * b;
      if (b == 0) {
#pragma unroll
        for (int q = 0; q < 16; ++q) ci[q] = 0.0f;
        continue;
      }
      float R[9];
      quat_to_mat(quat_mul(ld4(s + L.xquat + 4 * b), ld4(iquat + 4 * b)), R);
      const V3 off = ld3(s + L.xipos + 3 * b) - ld3(s + L.rcom + 3 * body_tree[b]);
      const float I0 = inertia[3 * b], I1 = inertia[3 * b + 1], I2 = inertia[3 * b + 2], ms = mass[b];
      const float oo = dot(off, off);
      const float o[3] = {off.x, off.y, off.z};
      // (ximat * inertia) @ ximat.T + h @ h.T * mass, h = cross(off, -I): entries [00 11 22 01 02 12]
      const int rr[6] = {0, 1, 2, 0, 0, 1}, cc[6] = {0, 1, 2, 1, 2, 2};
#pragma unroll
      for (int q = 0; q < 6; ++q) {
        const int r = rr[q], cl = cc[q];
        float v = R[3 * r] * I0 * R[3 * cl] + R[3 * r + 1] * I1 * R[3 * cl + 1] + R[3 * r + 2] * I2 * R[3 * cl + 2];
        v += (((r == cl) ? oo : 0.0f) - o[r] * o[cl]) * ms;
        ci[q] = v;
      }
      ci[6] = off.x * ms; ci[7] = off.y * ms; ci[8] = off.z * ms; ci[9] = ms;
    }
    const int* jbody = c.fi(VNL_F_JNT_BODYID);
    for (int j = tid; j < d.njnt; j += kEnvThreads) {
      const int b = jbody[j], da = jdofadr[j];
      const V3 off = ld3(s + L.rcom + 3 * body_tree[b]) - ld3(s + L.xanchor + 3 * j);
      if (jtype[j] == 0) {
        float R[9];
        quat_to_mat(ld4(s + L.xquat + 4 * b), R);
#pragma unroll
        for (int a = 0; a < 3; ++a) {
          float* ct = s + L.cdof + 6 * (da + a);
#pragma unroll
          for (int q = 0; q < 6; ++q) ct[q] = 0.0f;
          ct[3 + a] = 1.0f;
          const V3 ax = v3(R[a], R[3 + a], R[6 + a]);
          st3(s + L.cdof + 6 * (da + 3 + a), ax);
          st3(s + L.cdof + 6 * (da + 3 + a) + 3, cross(ax, off));
        }
      } else {
        const V3 ax = ld3(s + L.xaxis + 3 * j);
        st3(s + L.cdof + 6 * da, ax);
        st3(s + L.cdof + 6 * da + 3, cross(ax, off));
      }
    }
    env_sync();
    if (DUMP) {
      for (int i = tid; i < d.nbody * 3; i += kEnvThreads) dump[d.dump_xipos + i] = s[L.xipos + i];
      for (int i = tid; i < d.njnt * 3; i += kEnvThreads) { dump[d.dump_xanchor + i] = s[L.xanchor + i]; dump[d.dump_xanchor + d.njnt * 3 + i] = s[L.xaxis + i]; }
      for (int i = tid; i < d.nbody * 10; i += kEnvThreads) dump[d.dump_cinert + i] = s[L.t16 + kTS * (i / 10) + i % 10];
      for (int t = tid; t < d.nroot; t += kEnvThreads) st3(dump + d.dump_subtree_com + 3 * TB8(roots)[t], ld3(s + L.rcom + 3 * t));
    }
  }
  pf.mark(1);
  if (ls3) __syncthreads();
  // ---- smooth.com_vel + the forward half of smooth.rne: cvel, cacc down the tree (cdof_dot stays in registers) ---------
  {
    if (lane < 6) {
      s[L.cvel + lane] = 0.0f;
      s[L.cacc + lane] = (lane == 3) ? -d.gx : ((lane == 4) ? -d.gy : ((lane == 5) ? -d.gz : 0.0f));
    }
    env_sync();
    int k0 = 0;
    for (int lv = 0; lv < d.nlevel; ++lv) {
      const int k1 = lvl_start[lv + 1];
      if (k0 + tid < k1) {
        const uint32_t bp = lvl_bp[k0 + tid];
        const int b = bp & 255, p = bp >> 8;
        float cv[6], ca[6], cd[6];
#pragma unroll
        for (int q = 0; q < 6; ++q) { cv[q] = s[L.cvel + 6 * p + q]; ca[q] = s[L.cacc + 6 * p + q]; }
        const int dn = TB8(body_dofnum)[b];
        int i = TB8(body_dofadr)[b];
        const int ie = i + (dn & 0x7f);
        if (dn & 0x80) {  // free joint: translations first (cdof_dot = 0), the three rotations all see that velocity
#pragma unroll
          for (int a = 0; a < 3; ++a) {
            const float qv = s[L.qvel + i + a];
#pragma unroll
            for (int q = 0; q < 6; ++q) cv[q] += s[L.cdof + 6 * (i + a) + q] * qv;
          }
          float cv0[6];
#pragma unroll
          for (int q = 0; q < 6; ++q) cv0[q] = cv[q];
#pragma unroll
          for (int a = 3; a < 6; ++a) {
            const float qv = s[L.qvel + i + a];
            motion_cross(cv0, s + L.cdof + 6 * (i + a), cd);
#pragma unroll
            for (int q = 0; q < 6; ++q) { ca[q] += cd[q] * qv; cv[q] += s[L.cdof + 6 * (i + a) + q] * qv; }
          }
          i += 6;
        }
        for (; i < ie; ++i) {
          const float qv = s[L.qvel + i];
          motion_cross(cv, s + L.cdof + 6 * i, cd);
#pragma unroll
          for (int q = 0; q < 6; ++q) { ca[q] += cd[q] * qv; cv[q] += s[L.cdof + 6 * i + q] * qv; }
        }
#pragma unroll
        for (int q = 0; q < 6; ++q) { s[L.cvel + 6 * b + q] = cv[q]; s[L.cacc + 6 * b + q] = ca[q]; }
      }
      k0 = k1;
      env_sync();
    }
    pf.mark(27);
    // local RNE force of each body: cfrc = I cacc + cvel x* (I cvel)   -> t16[10..15]
    for (int b = tid; b < d.nbody; b += kEnvThreads) {
      float f1[6], iv[6], f2[6];
      inert_mul(s + L.t16 + kTS * b, s + L.cacc + 6 * b, f1);
      inert_mul(s + L.t16 + kTS * b, s + L.cvel + 6 * b, iv);
      motion_cross_force(s + L.cvel + 6 * b, iv, f2);
#pragma unroll
      for (int q = 0; q < 6; ++q) s[L.t16 + kTS * b + 10 + q] = f1[q] + f2[q];
    }
    env_sync();
    pf.mark(28);
    // one pass up the tree: composite inertia (crb, in place over cinert) and subtree-summed RNE force
    for (int lv = d.nlevel - 2; lv >= 0; --lv) {
      const int q0 = lvl_start[lv], n16 = (lvl_start[lv + 1] - q0) * 16;
      for (int it = tid; it < n16; it += kEnvThreads) {
        const int b = lvl_bp[q0 + (it >> 4)] & 255, q = it & 15;
        const int ce = TB8(child_adr)[b + 1];
        int ch = TB8(child_adr)[b];
        if (ch < ce) {
          float acc = s[L.t16 + kTS * b + q];
          for (; ch < ce; ++ch) acc += s[L.t16 + kTS * TB8(child_list)[ch] + q];
          s[L.t16 + kTS * b + q] = acc;
        }
      }
      env_sync();
    }
    if (DUMP) {
      for (int i = tid; i < d.nbody * 10; i += kEnvThreads) dump[d.dump_cinert + d.nbody * 10 + d.nv * 6 + i] = s[L.t16 + kTS * (i / 10) + i % 10];
      for (int i = tid; i < d.nbody * 6; i += kEnvThreads) dump[d.dump_cvel + i] = s[L.cvel + i];
    }
  }
  pf.mark(2);
  if (ls3) __syncthreads();
  // ---- qfrc_smooth = passive - bias + actuator; act_dot -----------------------------------------------------------------
  {
    const int* jqadr = c.fi(VNL_F_JNT_QPOSADR);
    const float* stiff = c.ff(VNL_F_JNT_STIFFNESS);
    const float* qspring = c.ff(VNL_F_QPOS_SPRING);
    const float* damping = c.ff(VNL_F_DOF_DAMPING);
    const int* actadr = c.fi(VNL_F_DOF_ACTADR);
    const int* actlist = c.fi(VNL_F_DOF_ACTLIST);
    const int* aadr = c.fi(VNL_F_ACT_ACTADR);
    const int* flim = c.fi(VNL_F_ACT_FORCELIMITED);
    const float* gain = c.ff(VNL_F_ACT_GAIN);
    const float* gear = c.ff(VNL_F_ACT_GEAR);
    const float* frange = c.ff(VNL_F_ACT_FORCERANGE);
    const float* dynprm = c.ff(VNL_F_ACT_DYNPRM);
    for (int i = tid; i < d.nv; i += kEnvThreads) {
      float acc = 0.0f;
      for (int t = actadr[i]; t < actadr[i + 1]; ++t) {  // actuators of this dof in actuator order (no atomics)
        const int u = actlist[t];
        const float ctrl = s[L.ctrl + u];
        float ca = ctrl;
        const int aa = aadr[u];
        if (aa >= 0) {
          s[L.act_dot + aa] = (ctrl - s[L.act + aa]) / fmaxf(dynprm[u], VNL_MINVAL);
          ca = s[L.act + aa];
        }
        float force = gain[u] * ca;
        if (flim[u]) force = fminf(fmaxf(force, frange[2 * u]), frange[2 * u + 1]);
        acc += gear[u] * force;
      }
      if (gf) gf[i] = acc;
      if (DUMP) dump[d.dump_passive + 2 * d.nv + i] = acc;
      const int j = dof_jnt[i];
      float pas;
      if (jtype[j] == 0) {
        const int a = i - jdofadr[j];
        pas = (a < 3) ? -stiff[j] * (s[L.qpos + jqadr[j] + a] - qspring[jqadr[j] + a]) : 0.0f;
      } else {
        pas = -stiff[j] * (s[L.qpos + jqadr[j]] - qspring[jqadr[j]]);
      }
      pas -= damping[i] * s[L.qvel + i];
      const float bias = dot6(s + L.cdof + 6 * i, s + L.t16 + kTS * dof_body[i] + 10);
      s[L.qfrc_smooth + i] = pas - bias + acc;
      if (DUMP) { dump[d.dump_passive + i] = pas; dump[d.dump_passive + d.nv + i] = bias; }
    }
    env_sync();
  }
  pf.mark(3);
  if (ls3) __syncthreads();
  // ---- joint-space inertia (tree sparse): M[i][a] = cdof[anc_a(i)] . (crb[body_i] cdof_i) --------------------------
  {
    const float* armature = c.ff(VNL_F_DOF_ARMATURE);
    float* fd = s + L.cacc;  // cacc is dead: reuse as crb * cdof
    for (int i = tid; i < d.nv; i += kEnvThreads) inert_mul(s + L.t16 + kTS * dof_body[i], s + L.cdof + 6 * i, fd + 6 * i);
    env_sync();
    float* const F = s + L.K;  // built straight into the factorisation's workspace (region A's head is dead by now)
    for (int e = tid; e < d.nM; e += kEnvThreads) {
      const int i = TB8(mrow)[e], j = TB8(mcol)[e];
      float v = dot6(fd + 6 * i, s + L.cdof + 6 * j);
      if (i == j) { v += armature[i]; s[L.Mdiag + i] = v; }
      F[e] = v;
      if (d.solver == 2) s[L.Mn + e] = v;
    }
    if (tid == 0) F[d.nM] = 0.0f;  // the zero entry padded program terms point at
    env_sync();
    if (DUMP) {
      for (int i = tid; i < d.nv * d.nv; i += kEnvThreads) dump[d.dump_qM + i] = 0.0f;
      env_sync();
      for (int q = tid; q < d.nM; q += kEnvThreads) {
        dump[d.dump_qM + TB8(mrow)[q] * d.nv + TB8(mcol)[q]] = F[q];
        dump[d.dump_qM + TB8(mcol)[q] * d.nv + TB8(mrow)[q]] = F[q];
      }
    }
    if (kStream) {  // program-ordered copies of M for the solver's mat-vecs and for the integrator's second factorisation
      float* const wk = slot_work(c);
      spill_section(TB32(prog_a), c.TA, F, wk);
      spill_section(TB32(prog_d), c.TD, F, wk + c.TA * kEnvThreads);
    } else {
      for (int e = tid; e <= d.nM; e += kEnvThreads) s[L.Ms + e] = F[e];
    }
    if (kEnvWarps > 1 || !kStream) env_sync();  // the factorisation rewrites F: every thread of the env must be done copying
  }
  pf.mark(4);
  if (ls3) __syncthreads();
  factor(so, false, true, pf);
  pf.mark(5);
  if (ls3) __syncthreads();
  solve_m(so, L.qfrc_smooth, L.qacc_smooth);
  pf.mark(6);
  if (ls3) __syncthreads();

  // ---- collision + constraint rows, compacted to the active set ----------------------------------------------------------
  float* arefv = s + L.Jv;  // aref lives in the Jv slot until the solver iterations start
  {
    if (lane == 0) { ints[0] = 0; ints[1] = 0; }
    for (int i = tid; i < d.nv; i += kEnvThreads) ((int*)(s + L.limrow_of_dof))[i] = -1;
    env_sync();
    // joint limits (constraint._instantiate_limit_slide_hinge): their rows come first
    {
      const int* ljnt = c.fi(VNL_F_LIMIT_JNT);
      const int* jqadr = c.fi(VNL_F_JNT_QPOSADR);
      const float* range = c.ff(VNL_F_JNT_RANGE);
      const float* margin = c.ff(VNL_F_JNT_MARGIN);
      const float* solref = c.ff(VNL_F_JNT_SOLREF);
      const float* solimp = c.ff(VNL_F_JNT_SOLIMP);
      const float* invw = c.ff(VNL_F_DOF_INVWEIGHT0);
      int base = 0;
      for (int r0 = 0; r0 < d.nlimit; r0 += 32) {
        const int r = r0 + lane;
        bool active = false;
        float pos = 0.0f, sign = 0.0f;
        int j = 0;
        if (r < d.nlimit) {
          j = ljnt[r];
          const float q = s[L.qpos + jqadr[j]];
          const float dmin = q - range[2 * j], dmax = range[2 * j + 1] - q;
          pos = fminf(dmin, dmax) - margin[j];
          active = pos < 0.0f;
          sign = (dmin < dmax) ? 1.0f : -1.0f;
        }
        const unsigned m = __ballot_sync(FULLMASK, active);
        if (active) {
          const int slot = base + __popc(m & ((1u << lane) - 1u));
          const int dof = jdofadr[j];
          ((int*)(s + L.lim_dof))[slot] = sign > 0.0f ? dof : ~dof;
          ((int*)(s + L.limrow_of_dof))[dof] = slot;
          float k, b, imp;
          kbi(d, solref[2 * j], solref[2 * j + 1], solimp + 5 * j, pos, k, b, imp);
          const float R = fmaxf(invw[dof] * (1.0f - imp) / imp, VNL_MINVAL);
          s[L.efcD + slot] = 1.0f / R;
          arefv[slot] = -b * (sign * s[L.qvel + dof]) - k * imp * pos;
          if (DUMP) { dump[d.dump_efc + r] = pos; dump[d.dump_efc + d.nefc + r] = 1.0f / R; dump[d.dump_efc + 2 * d.nefc + r] = arefv[slot]; }
        }
        base += __popc(m);
      }
      if (lane == 0) ints[0] = base;
    }
    env_sync();
    {  // contacts (collision_driver + constraint._instantiate_contact, pyramidal condim 3)
      const int nl = ints[0];
      const int* cpair = c.fi(VNL_F_CON_PAIR);
      const float* csign = c.ff(VNL_F_CON_SIGN);
      const int* ptype = c.fi(VNL_F_PAIR_TYPE);
      const int* g1 = c.fi(VNL_F_PAIR_GEOM1);
      const int* g2 = c.fi(VNL_F_PAIR_GEOM2);
      const int* gbody = c.fi(VNL_F_GEOM_BODYID);
      const float* gpos = c.ff(VNL_F_GEOM_POS);
      const float* gquat = c.ff(VNL_F_GEOM_QUAT);
      const float* gsize = c.ff(VNL_F_GEOM_SIZE);
      const float* pfric = c.ff(VNL_F_PAIR_FRICTION);
      const float* psolref = c.ff(VNL_F_PAIR_SOLREF);
      const float* psolimp = c.ff(VNL_F_PAIR_SOLIMP);
      const float* pmargin = c.ff(VNL_F_PAIR_INCLUDEMARGIN);
      const float* binvw = c.ff(VNL_F_BODY_INVWEIGHT0);
      int base = 0;
      for (int c0 = 0; c0 < d.ncon; c0 += 32) {
        const int ci = c0 + lane;
        bool active = false;
        float dist = 0.0f;
        V3 cp = v3(0, 0, 0), n = v3(0, 0, 1), fb = v3(0, 1, 0);
        int p = 0, body = 0;
        if (ci < d.ncon) {
          p = cpair[ci];
          const int ga = g1[p], gb = g2[p];
          body = gbody[gb];
          float Pm[9], Gm[9];  // the plane is attached to the world body: world frame = local frame
          quat_to_mat(ld4(gquat + 4 * ga), Pm);
          n = v3(Pm[2], Pm[5], Pm[8]);
          const V3 ppos = ld3(gpos + 3 * ga);
          const Q4 bq = ld4(s + L.xquat + 4 * body);
          const V3 gp = ld3(s + L.xpos + 3 * body) + rotate(ld3(gpos + 3 * gb), bq);
          quat_to_mat(quat_mul(bq, ld4(gquat + 4 * gb)), Gm);
          const float* sz = gsize + 3 * gb;
          const int ty = ptype[p];
          if (ty == 2) {  // plane_sphere
            dist = dot(gp - ppos, n) - sz[0];
            cp = gp - n * (sz[0] + 0.5f * dist);
          } else if (ty == 3) {  // plane_capsule end
            const V3 axis = v3(Gm[2], Gm[5], Gm[8]);
            V3 b = axis - n * dot(n, axis);
            const float bn = normalize3(b);
            if (bn < 0.5f) b = (-0.5f < n.y && n.y < 0.5f) ? v3(0, 1, 0) : v3(0, 0, 1);
            fb = b;
            const V3 sp = gp + axis * (csign[ci] * sz[1]);
            dist = dot(sp - ppos, n) - sz[0];
            cp = sp - n * (sz[0] + 0.5f * dist);
          } else {  // plane_ellipsoid
            const V3 ln = v3(Gm[0] * n.x + Gm[3] * n.y + Gm[6] * n.z, Gm[1] * n.x + Gm[4] * n.y + Gm[7] * n.z, Gm[2] * n.x + Gm[5] * n.y + Gm[8] * n.z);
            V3 sup = v3(ln.x * sz[0], ln.y * sz[1], ln.z * sz[2]);
            normalize3(sup);
            sup = v3(-sup.x * sz[0], -sup.y * sz[1], -sup.z * sz[2]);
            const V3 pt = gp + v3(Gm[0] * sup.x + Gm[1] * sup.y + Gm[2] * sup.z, Gm[3] * sup.x + Gm[4] * sup.y + Gm[5] * sup.z, Gm[6] * sup.x + Gm[7] * sup.y + Gm[8] * sup.z);
            dist = dot(n, pt - ppos);
            cp = pt - n * (dist * 0.5f);
          }
          if (ty != 3) {  // math.make_frame
            V3 nn = n;
            normalize3(nn);
            n = nn;
            V3 b = (-0.5f < n.y && n.y < 0.5f) ? v3(0, 1, 0) : v3(0, 0, 1);
            b = b - n * dot(n, b);
            normalize3(b);
            fb = b;
          }
          if (DUMP) {
            dump[d.dump_con + ci] = dist;
            st3(dump + d.dump_con + d.ncon + 3 * ci, cp);
            st3(dump + d.dump_con + 4 * d.ncon + 9 * ci, n); st3(dump + d.dump_con + 4 * d.ncon + 9 * ci + 3, fb);
            st3(dump + d.dump_con + 4 * d.ncon + 9 * ci + 6, cross(n, fb));
          }
          dist -= pmargin[p];
          active = dist < 0.0f;
        }
        const unsigned m = __ballot_sync(FULLMASK, active);
        if (active) {
          const int k = base + __popc(m & ((1u << lane) - 1u));
          ((int*)(s + L.cbody))[k] = body;
          const V3 rel = cp - ld3(s + L.rcom + 3 * body_tree[body]);
          st3(s + L.crel + 3 * k, rel);
          const V3 t2 = cross(n, fb);
          st3(s + L.cframe + 6 * k, n); st3(s + L.cframe + 6 * k + 3, fb);
          const float mu = pfric[5 * p];
          s[L.cmu + k] = mu;
          float kk, bb, imp;
          kbi(d, psolref[2 * p], psolref[2 * p + 1], psolimp + 5 * p, dist, kk, bb, imp);
          const float t = binvw[2 * body];
          const float invweight = (t + mu * mu * t) * 2.0f * mu * mu / d.impratio;
          const float R = fmaxf(invweight * (1.0f - imp) / imp, VNL_MINVAL);
          // J qvel for the four pyramid rows = frame . point velocity (cvel is the body's spatial velocity)
          const float* cv = s + L.cvel + 6 * body;
          const V3 vel = ld3(cv + 3) + cross(ld3(cv), rel);
          const float un = dot(n, vel), u1 = dot(fb, vel), u2 = dot(t2, vel);
          const float ref = -kk * imp * dist;
          const int r = nl + 4 * k;
          s[L.efcD + r] = s[L.efcD + r + 1] = s[L.efcD + r + 2] = s[L.efcD + r + 3] = 1.0f / R;
          arefv[r] = -bb * (un + mu * u1) + ref;
          arefv[r + 1] = -bb * (un - mu * u1) + ref;
          arefv[r + 2] = -bb * (un + mu * u2) + ref;
          arefv[r + 3] = -bb * (un - mu * u2) + ref;
          if (DUMP) {
            const int rr = d.nlimit + 4 * ci;
            for (int q = 0; q < 4; ++q) {
              dump[d.dump_efc + rr + q] = dist; dump[d.dump_efc + d.nefc + rr + q] = 1.0f / R;
              dump[d.dump_efc + 2 * d.nefc + rr + q] = arefv[r + q];
            }
          }
        }
        base += __popc(m);
      }
      if (lane == 0) ints[1] = base;
    }
    env_sync();
  }
  pf.mark(7);
  if (ls3) __syncthreads();
  const int nl = ints[0], nc = ints[1], nrow = nl + 4 * nc;
  if (tid == 0) { stats[2] += nc; stats[3] += nl; }

  // ---- solver.solve (CG with the MJX line search) ------------------------------------------------------------------------
  float* qacc = s + L.qacc;
  float* Ma = s + L.Ma;
  float* Jaref = s + L.Jaref;
  float* Jv = s + L.Jv;
  const float* efcD = s + L.efcD;
  float* const Mgp = s + L.grad;  // CG: previous M^-1 grad (Polak-Ribiere) in the gradient's slot (see update_constraint)
  const float* const qfrc_con = s + L.qfrc_con;
#define VNL_GRAD(i) (Ma[i] - qfrc_smooth[i] - qfrc_con[i])
  float* Mgrad = s + L.Mgrad;
  float* search = s + L.search;
  float* Mv = s + L.Mv;
  const float* qfrc_smooth = s + L.qfrc_smooth;
  const float* qacc_smooth = s + L.qacc_smooth;
  int niter = 0, lsiter = 0;
  {
    // candidate cost: 0.5 sum D Jaref^2 [Jaref<0] + 0.5 (Ma - qfrc_smooth).(qacc - qacc_smooth)
    // The smooth candidate is evaluated FIRST: the warm start wins in all but the first substep after a reset, and the
    // winner's Ma / Jaref are then already in place (the loser's would have to be recomputed).
    float cost_w, cost_s;
    {
      // its Gauss term is (M qacc_smooth - qfrc_smooth) . (qacc_smooth - qacc_smooth) = 0 whatever M qacc_smooth rounds to,
      // so the mat-vec is only done if this candidate wins (below)
      jmul(so, L.qacc_smooth, L.Jaref);
      float w0 = 0.0f;
      for (int r = lane; r < nrow; r += 32) { const float ja = Jaref[r] - arefv[r]; if (ja < 0.0f) w0 += efcD[r] * ja * ja; }
      w0 = warp_sum(w0);
      cost_s = 0.5f * w0;
      env_sync();
      mul_m(so, L.warm, L.Ma);
      jmul(so, L.warm, L.Jaref);
      float v0 = 0.0f, v1 = 0.0f;
      for (int r = lane; r < nrow; r += 32) { const float ja = Jaref[r] - arefv[r]; if (ja < 0.0f) v0 += efcD[r] * ja * ja; }
      for (int i = lane; i < d.nv; i += 32) v1 += (Ma[i] - qfrc_smooth[i]) * (s[L.warm + i] - qacc_smooth[i]);
      v0 = warp_sum(v0); v1 = warp_sum(v1);
      cost_w = 0.5f * v0 + 0.5f * v1;
      env_sync();
    }
    if (cost_w < cost_s) {
      for (int i = tid; i < d.nv; i += kEnvThreads) qacc[i] = s[L.warm + i];  // Ma, Jaref already hold the warm-start candidate
    } else {
      for (int i = tid; i < d.nv; i += kEnvThreads) qacc[i] = qacc_smooth[i];
      env_sync();
      mul_m(so, L.qacc, L.Ma);
      jmul(so, L.qacc, L.Jaref);
    }
    env_sync();
    for (int r = tid; r < nrow; r += kEnvThreads) Jaref[r] -= arefv[r];
    env_sync();
    pf.mark(8);
    if (ls3) __syncthreads();
    const float scale = d.meaninertia * (float)max(1, d.nv);
    Sol st;
    st.cost = INFINITY; st.prev_cost = 0.0f; st.gauss = 0.0f; st.gradnorm = 0.0f;
    st.stop = false;
    st = update_constraint(so, st, pf, d.iterations < 1, scale);
    bool done = st.stop;  // true: converged before the first iteration
    // CG: Mgrad = M^-1 grad, so M search needs no mat-vec: M (-Mgrad) = -grad, and Polak-Ribiere's search = -Mgrad + beta search
    // carries it along as Mv = -grad + beta Mv (MJX multiplies by M every iteration; the two agree to rounding).
    if (!done) for (int i = tid; i < d.nv; i += kEnvThreads) { search[i] = -Mgrad[i]; Mv[i] = -VNL_GRAD(i); }
    env_sync();
    pf.mark(9);
    for (int itn = 0; itn < d.iterations; ++itn) {
      if (lsi && (itn & lsi_mask) == 0) __syncthreads();
      if (!done && d.iterations != 1) {
        const float improvement = (st.prev_cost - st.cost) / scale;
        const float gradient = st.gradnorm / scale;
        done = (improvement < d.tolerance) || (gradient < d.tolerance);
      }
      if (done) { if (lsi) continue; break; }
      // ---- _linesearch ----
      if (d.solver == 2) mul_m(so, L.search, L.Mv);  // Newton: Mgrad = H^-1 grad, no such shortcut
      pf.mark(19);
      jmul(so, L.search, L.Jv);
      pf.mark(20);
      float q0s = 0.0f, q1s = 0.0f, q2s = 0.0f, q3s = 0.0f;
      for (int i = lane; i < d.nv; i += 32) {
        const float si = search[i];
        q0s += si * si; q1s += si * Ma[i]; q2s += si * qfrc_smooth[i]; q3s += si * Mv[i];
      }
      { float a4[4] = {q0s, q1s, q2s, q3s}; warp_sum_n<4>(a4); q0s = a4[0]; q1s = a4[1]; q2s = a4[2]; q3s = a4[3]; }
      const float gtol = d.tolerance * d.ls_tolerance * (sqrtf(q0s) * scale);
      const float g0 = st.gauss, g1 = q1s - q2s, g2 = 0.5f * q3s;
      // One evaluation site for all line-search points: phase 0 evaluates alpha = 0, phase 1 the Newton step from
      // it, later phases the three candidates (lo_next, hi_next, mid) of one bracketing round.
      LSP p0, lo, hi;
      p0.alpha = p0.cost = p0.d0 = p0.d1 = 0.0f;
      lo = p0; hi = p0;
      bool swap = true;
      int it = 0;
      for (int phase = 0;; ++phase) {
        float al0, al1, al2;
        if (phase == 0) { al0 = al1 = al2 = 0.0f; }
        else if (phase == 1) { al0 = al1 = al2 = p0.alpha - p0.d0 / p0.d1; }
        else {
          bool ldone = it >= d.ls_iterations;
          ldone |= !swap;
          ldone |= (lo.d0 < 0.0f) && (lo.d0 > -gtol);
          ldone |= (hi.d0 > 0.0f) && (hi.d0 < gtol);
          if (ldone) break;
          al0 = lo.alpha - lo.d0 / lo.d1;
          al1 = hi.alpha - hi.d0 / hi.d1;
          al2 = 0.5f * (lo.alpha + hi.alpha);
        }
        float acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
        for (int r = lane; r < nrow; r += 32) {
          const float x = Jaref[r], jv = Jv[r], D = efcD[r];
          const float q0 = 0.5f * x * x * D, q1 = jv * x * D, q2 = 0.5f * jv * jv * D;
          if (x + al0 * jv < 0.0f) { acc[0] += q0; acc[1] += q1; acc[2] += q2; }
          if (x + al1 * jv < 0.0f) { acc[3] += q0; acc[4] += q1; acc[5] += q2; }
          if (x + al2 * jv < 0.0f) { acc[6] += q0; acc[7] += q1; acc[8] += q2; }
        }
        if (phase < 2) {  // a single alpha: three sums
          float a4[4] = {acc[0], acc[1], acc[2], 0.0f};
          warp_sum_n<4>(a4);
          acc[0] = a4[0]; acc[1] = a4[1]; acc[2] = a4[2];
        } else {
          float a8[8] = {acc[0], acc[1], acc[2], acc[3], acc[4], acc[5], acc[6], acc[7]};
          warp_sum_n<8>(a8);
#pragma unroll
          for (int q = 0; q < 8; ++q) acc[q] = a8[q];
          acc[8] = warp_sum(acc[8]);
        }
        LSP pt[3];
        const float als[3] = {al0, al1, al2};
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const float q0 = acc[3 * k] + g0, q1 = acc[3 * k + 1] + g1, q2 = acc[3 * k + 2] + g2, a = als[k];
          pt[k].alpha = a;
          pt[k].cost = a * a * q2 + a * q1 + q0;
          pt[k].d0 = 2.0f * a * q2 + q1;
          pt[k].d1 = 2.0f * q2 + (q2 == 0.0f ? VNL_MINVAL : 0.0f);
        }
        if (phase == 0) { p0 = pt[0]; continue; }
        if (phase == 1) {
          const bool lesser = pt[0].d0 < p0.d0;
          hi = lesser ? p0 : pt[0];
          lo = lesser ? pt[0] : p0;
          continue;
        }
        const LSP lo_next = pt[0], hi_next = pt[1], mid = pt[2];
        const bool s1 = (lo.d0 > 0.0f) || (lo.d0 < lo_next.d0);
        if (s1) lo = lo_next;
        const bool s2 = (mid.d0 < 0.0f) && (lo.d0 < mid.d0);
        if (s2) lo = mid;
        const bool s3 = (hi_next.d0 < 0.0f) && (lo.d0 < hi_next.d0);
        if (s3) lo = hi_next;
        const bool s4 = (hi.d0 < 0.0f) || (hi.d0 > hi_next.d0);
        if (s4) hi = hi_next;
        const bool s5 = (mid.d0 > 0.0f) && (hi.d0 > mid.d0);
        if (s5) hi = mid;
        const bool s6 = (lo_next.d0 > 0.0f) && (hi.d0 > lo_next.d0);
        if (s6) hi = lo_next;
        swap = s1 || s2 || s3 || s4 || s5 || s6;
        ++it;
      }
      lsiter += it;
      pf.mark(21);
      const bool improved = (lo.cost < p0.cost) || (hi.cost < p0.cost);
      const float alpha = lo.cost < hi.cost ? lo.alpha : hi.alpha;
      const float ia = improved ? alpha : 0.0f * alpha;
      float pg = 0.0f;  // previous grad . Mgrad before they are overwritten
      if (d.solver != 2) for (int i = lane; i < d.nv; i += 32) pg += VNL_GRAD(i) * Mgrad[i];
      pg = warp_sum(pg);
      env_sync();  // (pg re-forms the gradient from Ma, which the update below advances)
      if (d.solver == 2) { for (int i = tid; i < d.nv; i += kEnvThreads) { qacc[i] += search[i] * ia; Ma[i] += Mv[i] * ia; } }
      else { for (int i = tid; i < d.nv; i += kEnvThreads) { qacc[i] += search[i] * ia; Ma[i] += Mv[i] * ia; Mgp[i] = Mgrad[i]; } }
      for (int r = tid; r < nrow; r += kEnvThreads) Jaref[r] += Jv[r] * ia;
      env_sync();
      st = update_constraint(so, st, pf, itn == d.iterations - 1, scale);
      done = st.stop;
      if (done) {
        // no further iteration: the search direction is not needed
      } else if (d.solver == 2) {
        for (int i = tid; i < d.nv; i += kEnvThreads) search[i] = -Mgrad[i];
      } else {  // Polak-Ribiere
        float nb = 0.0f;
        for (int i = lane; i < d.nv; i += 32) nb += VNL_GRAD(i) * (Mgrad[i] - Mgp[i]);
        nb = warp_sum(nb);
        const float beta = fmaxf(0.0f, nb / fmaxf(VNL_MINVAL, pg));
        for (int i = tid; i < d.nv; i += kEnvThreads) { search[i] = -Mgrad[i] + beta * search[i]; Mv[i] = -VNL_GRAD(i) + beta * Mv[i]; }
      }
      env_sync();
      pf.mark(11);
      ++niter;
    }
  }
#undef VNL_GRAD
  if (tid == 0) { stats[0] += niter; stats[1] += lsiter; }
  for (int i = tid; i < d.nv; i += kEnvThreads) s[L.warm + i] = qacc[i];  // qacc_warmstart <- qacc
  env_sync();
}

// ---------------------------------------------------------------------------------------------------------------------
// forward.euler (implicit joint damping when enabled) + _advance
// ---------------------------------------------------------------------------------------------------------------------
__device__ __noinline__ void euler(int so, Prof pf) {
  VNL_SMEM
  const Dims& d = c.d;
  const Lay& L = c.L;
  const int lane = LANE, tid = ETID;
  const float dt = d.timestep;
  float* qacc = s + L.qacc;
  pf.mark(12);
  if (d.eulerdamp) {
    factor(so, true, false, pf);
    pf.mark(13);
    for (int i = tid; i < d.nv; i += kEnvThreads) s[L.grad + i] = s[L.qfrc_smooth + i] + s[L.qfrc_con + i];
    env_sync();
    solve_ld(so, L.grad, L.Mgrad);
    qacc = s + L.Mgrad;
  }
  for (int a = tid; a < d.na; a += kEnvThreads) s[L.act + a] += s[L.act_dot + a] * dt;
  for (int i = tid; i < d.nv; i += kEnvThreads) s[L.qvel + i] += qacc[i] * dt;
  env_sync();
  const int* jtype = c.fi(VNL_F_JNT_TYPE);
  const int* jqadr = c.fi(VNL_F_JNT_QPOSADR);
  const int* jdofadr = c.fi(VNL_F_JNT_DOFADR);
  for (int j = tid; j < d.njnt; j += kEnvThreads) {
    const int qa = jqadr[j], da = jdofadr[j];
    if (jtype[j] == 0) {
      for (int k = 0; k < 3; ++k) s[L.qpos + qa + k] += s[L.qvel + da + k] * dt;
      V3 w = ld3(s + L.qvel + da + 3);
      const float norm = normalize3(w);
      const Q4 q = quat_normalize(quat_mul(ld4(s + L.qpos + qa + 3), axis_angle_quat(w, dt * norm)));
      st4(s + L.qpos + qa + 3, q);
    } else {
      s[L.qpos + qa] += s[L.qvel + da] * dt;
    }
  }
  env_sync();
  pf.mark(14);
}

__device__ __forceinline__ float nan_to_num(float v) {
  if (isnan(v)) return 0.0f;
  if (isinf(v)) return v > 0.0f ? 3.402823466e+38f : -3.402823466e+38f;
  return v;
}

// The reward terms that depend on (qvel, qpos, qfrc_actuator, subtree_com) of ONE state: the post-step state for the
// rodent (rodent.py:266-316), the pre-step state for the humanoid (humanoid.py:264-311).  Warp-cooperative.
struct RewardTerms { float rcom, rvel, rquat, ract, healthy; };
__device__ __noinline__ RewardTerms reward_state_terms(const uint32_t* tb, int nv, int f, const float* qvel, const float* qpos,
                                                       const float* qfrc, const float* com) {
  const int lane = LANE;
  const int ntrack = vnl_hdr_i(tb, VNL_TH_NTRACK);
  const float* rvel = vnl_field_f(tb, VNL_T_VELOCITY) + (size_t)f * 3;
  const float* rang = vnl_field_f(tb, VNL_T_ANGULAR_VELOCITY) + (size_t)f * 3;
  const float* rjv = vnl_field_f(tb, VNL_T_JOINTS_VELOCITY) + (size_t)f * (nv - 6);
  float v0 = 0.0f, v1 = 0.0f;
  for (int i = lane; i < nv; i += 32) {
    const float ref = i < 3 ? rvel[i] : (i < 6 ? rang[i - 3] : rjv[i - 6]);
    const float df = qvel[i] - ref;
    v0 += df * df;
    const float qa = qfrc[i];
    v1 += qa * qa;
  }
  v0 = warp_sum(v0); v1 = warp_sum(v1);
  const float* cref = vnl_hdr_i(tb, VNL_TH_COM_FROM_FIELD)
                          ? vnl_field_f(tb, VNL_T_CENTER_OF_MASS) + (size_t)f * 3
                          : vnl_field_f(tb, VNL_T_BODY_POSITIONS) + ((size_t)f * ntrack + vnl_hdr_i(tb, VNL_TH_COM_REF_IDX)) * 3;
  const V3 dc = ld3(com) - ld3(cref);
  RewardTerms r;
  r.rcom = expf(-100.0f * sqrtf(dot(dc, dc)));
  r.rvel = expf(-0.1f * sqrtf(v0));
  const Q4 qc = quat_normalize(ld4(qpos + 3));
  const Q4 qr = quat_normalize(ld4(vnl_field_f(tb, VNL_T_QUATERNION) + (size_t)f * 4));
  const float dq = qc.w * qr.w + qc.x * qr.x + qc.y * qr.y + qc.z * qr.z;
  const float dist = fminf(1.0f, 2.0f * dq * dq - 1.0f);
  r.rquat = expf(-2.0f * fabsf(0.5f * acosf(dist)));
  r.ract = -0.015f * (v1 / (float)nv);
  const float z = qpos[2];
  r.healthy = z < vnl_hdr_f(tb, VNL_TH_HEALTHY_LO) ? 0.0f : 1.0f;
  if (z > vnl_hdr_f(tb, VNL_TH_HEALTHY_HI)) r.healthy = 0.0f;
  return r;
}

// Philox4x32-10 (Salmon et al., SC 2011; the constants of Random123): the draws of the resampling reset (DESIGN §3h)
__device__ __forceinline__ uint4 philox4x32_10(uint4 x, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t lo0 = 0xD2511F53u * x.x, hi0 = __umulhi(0xD2511F53u, x.x);
    const uint32_t lo1 = 0xCD9E8D57u * x.z, hi1 = __umulhi(0xCD9E8D57u, x.z);
    x = make_uint4(hi1 ^ x.y ^ k0, lo1, hi0 ^ x.w ^ k1, lo0);
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return x;
}

// ---------------------------------------------------------------------------------------------------------------------
// one env, one env group.  MODE 0 = env step, 1 = env reset tail, 2 = physics only, 3 = forward stage dump,
// 4 = kinematics only (clip preprocessing: qpos -> normalised qpos, xpos, xquat), 5 = reset to a fresh draw (the envs
// listed in p.rs.scratch: the resampling AutoReset, DESIGN §3h) -- mode 1 with the qpos / qvel / clip / start frame drawn
// in-kernel, no reward / done / metrics / stats writes
// ---------------------------------------------------------------------------------------------------------------------
template <int MODE>
__device__ __forceinline__ void env_run(int so, const Params& p, int e, bool active) {
  VNL_SMEM
  constexpr bool kReset = MODE == 1 || MODE == 5;
  const Dims& d = c.d;
  const Lay& L = c.L;
  const int lane = LANE, tid = ETID;
  if (MODE == 4) {  // preprocessing/mjx_preprocess.py:109-134 `extract_features`: set_position -> smooth.kinematics, per frame
    if (!active) return;  // no CTA-wide barriers on this path
    Prof pf4; pf4.p = nullptr; pf4.t0o = 0;
    for (int i = tid; i < d.nq; i += kEnvThreads) s[L.qpos + i] = p.in.qpos[(size_t)e * d.nq + i];
    env_sync();
    forward<false>(so, nullptr, pf4, p.out.xpos + (size_t)e * d.nbody * 3, p.out.xquat + (size_t)e * d.nbody * 4, nullptr, true);
    for (int i = tid; i < d.nq; i += kEnvThreads) p.out.qpos[(size_t)e * d.nq + i] = s[L.qpos + i];  // free-joint quaternion normalised
    env_sync();
    return;
  }
  if (!active) {  // a warp without an env in this round only keeps the CTA's phase barriers company
    if (p.lockstep) {
      const int ns = (kReset || MODE == 3) ? 1 : p.nsteps;
      for (int st = 0; st < ns; ++st) { group_sync(p.lsgroups); if (kReset || MODE == 3) break; if (p.lockstep > 1) group_sync(p.lsgroups); }
    }
    return;
  }
  Prof pf;
  pf.p = (c.prof && e == c.prof_env) ? c.prof : nullptr;
  pf.t0o = so + c.L.ints + 12;  // ints[12..13]: 8-byte aligned (the slice and every array start on 16 bytes)
  int* ints = (int*)(s + L.ints);
  if (lane < 16) ints[lane] = 0;
  if (pf.p) { env_sync(); if (ETID == 0) *reinterpret_cast<long long*>(smem + pf.t0o) = clock64(); }

  const uint32_t* tb = p.task;
  // ---- load state -------------------------------------------------------------------------------------------------------
  int rclip = 0, rstart = 0, rcount = 0;
  if (MODE == 5) {
    // the draw (include/vnl_b200.h, VnlResample): block 0 = clip and start frame, blocks 1 .. = four qpos normals each;
    // qpos / qvel = the clip row (clip, start) as the env classes' reset() stack it, plus the noise
    const VnlResample& rs = p.rs;
    const uint32_t k0 = (uint32_t)rs.seed, k1 = (uint32_t)(rs.seed >> 32), g = (uint32_t)(rs.env_offset + e);
    rcount = rs.reset_count[e];
    const uint4 x = philox4x32_10(make_uint4(g, (uint32_t)rcount, 0u, 0u), k0, k1);
    rclip = (int)(((uint64_t)x.x * (uint64_t)max(1, vnl_hdr_i(tb, VNL_TH_NCLIPS))) >> 32);
    rstart = (int)(((uint64_t)x.y * (uint64_t)rs.start_frame_hi) >> 32);
    const size_t row = (size_t)rclip * vnl_hdr_i(tb, VNL_TH_CLIP_LEN) + rstart;
    const int nj = d.nq - 7, nvj = d.nv - 6;
    for (int i = tid; i < d.nq; i += kEnvThreads)
      s[L.qpos + i] = i < 3 ? vnl_field_f(tb, VNL_T_POSITION)[row * 3 + i]
                      : i < 7 ? vnl_field_f(tb, VNL_T_QUATERNION)[row * 4 + i - 3] : vnl_field_f(tb, VNL_T_JOINTS)[row * nj + i - 7];
    for (int i = tid; i < d.nv; i += kEnvThreads)
      s[L.qvel + i] = i < 3 ? vnl_field_f(tb, VNL_T_VELOCITY)[row * 3 + i]
                      : i < 6 ? vnl_field_f(tb, VNL_T_ANGULAR_VELOCITY)[row * 3 + i - 3] : vnl_field_f(tb, VNL_T_JOINTS_VELOCITY)[row * nvj + i - 6];
    env_sync();
    if (rs.noise_scale != 0.0f) {
      for (int j = 1 + tid; 4 * (j - 1) < d.nq; j += kEnvThreads) {  // the lanes draw the noise blocks in parallel
        const uint4 y = philox4x32_10(make_uint4(g, (uint32_t)rcount, (uint32_t)j, 0u), k0, k1);
        const float u[4] = {(float)((y.x >> 8) + 1u) * 0x1p-24f, (float)((y.y >> 8) + 1u) * 0x1p-24f,
                            (float)((y.z >> 8) + 1u) * 0x1p-24f, (float)((y.w >> 8) + 1u) * 0x1p-24f};
        float nrm[4];
        for (int h = 0; h < 2; ++h) {
          const float r = sqrtf(-2.0f * logf(u[2 * h]));
          float sn, cs;
          sincospif(2.0f * u[2 * h + 1], &sn, &cs);
          nrm[2 * h] = r * cs; nrm[2 * h + 1] = r * sn;
        }
        for (int k = 0; k < 4; ++k) {
          const int i = 4 * (j - 1) + k;
          if (i < d.nq) s[L.qpos + i] = fmaf(rs.noise_scale, nrm[k], s[L.qpos + i]);
        }
      }
    }
  } else {
    for (int i = tid; i < d.nq; i += kEnvThreads) s[L.qpos + i] = p.in.qpos[(size_t)e * d.nq + i];
    for (int i = tid; i < d.nv; i += kEnvThreads) s[L.qvel + i] = p.in.qvel[(size_t)e * d.nv + i];
  }
  if (kReset) {
    for (int i = tid; i < d.na; i += kEnvThreads) s[L.act + i] = 0.0f;
    for (int i = tid; i < d.nv; i += kEnvThreads) s[L.warm + i] = 0.0f;
    for (int i = tid; i < d.nu; i += kEnvThreads) s[L.ctrl + i] = 0.0f;
  } else {
    for (int i = tid; i < d.na; i += kEnvThreads) s[L.act + i] = p.in.act ? p.in.act[(size_t)e * d.na + i] : 0.0f;
    for (int i = tid; i < d.nv; i += kEnvThreads) s[L.warm + i] = p.in.qacc_warmstart ? p.in.qacc_warmstart[(size_t)e * d.nv + i] : 0.0f;
    const int* climited = c.fi(VNL_F_ACT_CTRLLIMITED);
    const float* crange = c.ff(VNL_F_ACT_CTRLRANGE);
    for (int u = tid; u < d.nu; u += kEnvThreads) {
      float v = p.ctrl ? p.ctrl[(size_t)e * d.nu + u] : 0.0f;
      if (climited[u]) v = fminf(fmaxf(v, crange[2 * u]), crange[2 * u + 1]);
      s[L.ctrl + u] = v;
    }
  }
  env_sync();
  // termination error of the PREVIOUS state and frame (envs/rodent.py:241-264, quirks Q2 / Q9): depends only on
  // inputs, so evaluate it before the physics overwrites them.
  float rtrunk = 0.0f;
  int frame_old = 0;
  // multi-clip task tables (SURVEY 8 row f4): every clip table is [nclips, T, ...]; the env's clip only offsets the row
  int fbase = 0, clip = 0;
  if (MODE == 0 || kReset) {
    const int nclips = max(1, vnl_hdr_i(tb, VNL_TH_NCLIPS));
    clip = MODE == 5 ? rclip : p.in.clip_id ? min(max(p.in.clip_id[e], 0), nclips - 1) : 0;
    fbase = clip * vnl_hdr_i(tb, VNL_TH_CLIP_LEN);
  }
  RewardTerms rt;
  rt.rcom = rt.rvel = rt.rquat = rt.ract = rt.healthy = 0.0f;
  if (MODE == 0) {
    frame_old = p.in.cur_frame[e];
    const int T = vnl_hdr_i(tb, VNL_TH_CLIP_LEN), ntrack = vnl_hdr_i(tb, VNL_TH_NTRACK), nj = d.nq - 7;
    const int f = min(max(frame_old, 0), T - 1);
    const float* rj = vnl_field_f(tb, VNL_T_JOINTS) + (size_t)(fbase + f) * nj;
    const float* rb = vnl_field_f(tb, VNL_T_BODY_POSITIONS) + (size_t)(fbase + f) * ntrack * 3;
    const int* bidx = vnl_field_i(tb, VNL_T_BODY_IDXS);
    const float* xold = p.in.xpos + (size_t)e * d.nbody * 3;
    float v0 = 0.0f, v1 = 0.0f, v2 = 0.0f, v3_ = 0.0f;
    for (int j = lane; j < nj; j += 32) v0 += fabsf(rj[j] - s[L.qpos + 7 + j]);
    for (int b = lane; b < ntrack; b += 32) {
      v1 += fabsf(rb[3 * b] - xold[3 * bidx[b]]);
      v2 += fabsf(rb[3 * b + 1] - xold[3 * bidx[b] + 1]);
      v3_ += fabsf(rb[3 * b + 2] - xold[3 * bidx[b] + 2]);
    }
    v0 = warp_sum(v0); v1 = warp_sum(v1); v2 = warp_sum(v2); v3_ = warp_sum(v3_);
    float eb = fmaxf(v1, fmaxf(v2, v3_));
    if (vnl_hdr_i(tb, VNL_TH_TERM_MEAN)) { v0 = v0 / (float)nj; eb = (v1 + v2 + v3_) / (float)(3 * ntrack); }  // humanoid.py:256-258
    const float err = 0.5f * vnl_hdr_f(tb, VNL_TH_BODY_ERR_MULT) * eb + 0.5f * v0;
    rtrunk = 1.0f - err / vnl_hdr_f(tb, VNL_TH_TERM_THRESHOLD);
    if (vnl_hdr_i(tb, VNL_TH_REWARD_OLD_STATE))  // humanoid.py:275: the whole reward reads the pre-step state
      rt = reward_state_terms(tb, d.nv, fbase + f, s + L.qvel, s + L.qpos, p.in.qfrc_actuator + (size_t)e * d.nv, p.in.subtree_com + (size_t)e * 3);
  }

  int* stats = ints + 4;  // [4..7]
  float* dump = (MODE == 3) ? p.dump + (size_t)e * d.dump_total : nullptr;
  const int nsteps = (kReset || MODE == 3) ? 1 : p.nsteps;
  for (int st = 0; st < nsteps; ++st) {
    // Optional lockstep: the warps of a CTA start each substep together, so that they walk the (large) instruction
    // footprint of a substep as one group instead of seven independent streams.
    if (p.lockstep) group_sync(p.lsgroups);
    {
      const bool last = (MODE != 3) && (st == nsteps - 1);  // MODE 3 has no output state
      forward<MODE == 3>(so, dump, pf, last ? p.out.xpos + (size_t)e * d.nbody * 3 : nullptr,
                         last ? p.out.xquat + (size_t)e * d.nbody * 4 : nullptr, last ? p.out.qfrc_actuator + (size_t)e * d.nv : nullptr);
    }
    if (kReset || MODE == 3) break;
    if (p.lockstep > 1) group_sync(p.lsgroups);
    euler(so, pf);
  }

  if (MODE == 3) {
    // stage dump (layout = oracle.dump_layout); arrays this formulation never materialises stay NaN
    auto put = [&](int off, const float* src, int n) { for (int i = tid; i < n; i += kEnvThreads) dump[off + i] = src[i]; };
    put(d.dump_cinert + d.nbody * 10, s + L.cdof, d.nv * 6);
    put(d.dump_passive + 3 * d.nv, s + L.act_dot, d.na);
    put(d.dump_passive + 3 * d.nv + d.na, s + L.qfrc_smooth, d.nv);
    put(d.dump_passive + 4 * d.nv + d.na, s + L.qacc_smooth, d.nv);
    put(d.dump_qacc, s + L.qacc, d.nv);
    put(d.dump_qacc + d.nv, s + L.qfrc_con, d.nv);
    if (lane < 4) dump[d.dump_total - 4 + lane] = (float)stats[lane];
    env_sync();
    return;
  }

  // ---- write state ------------------------------------------------------------------------------------------------------
  const VnlState& o = p.out;
  for (int i = tid; i < d.nq; i += kEnvThreads) o.qpos[(size_t)e * d.nq + i] = s[L.qpos + i];
  for (int i = tid; i < d.nv; i += kEnvThreads) o.qvel[(size_t)e * d.nv + i] = s[L.qvel + i];
  for (int i = tid; i < d.na; i += kEnvThreads) o.act[(size_t)e * d.na + i] = s[L.act + i];
  for (int i = tid; i < d.nv; i += kEnvThreads) o.qacc_warmstart[(size_t)e * d.nv + i] = s[L.warm + i];
  // xpos / xquat / qfrc_actuator were stored by the last forward pass; the task code below reads them back (same warp,
  // ordered by the env barriers in between)
  const float* const gxp = o.xpos + (size_t)e * d.nbody * 3;
  const float* const gxq = o.xquat + (size_t)e * d.nbody * 4;
  const float* const gfa = o.qfrc_actuator + (size_t)e * d.nv;
  const int torso = (MODE == 2) ? 1 : vnl_hdr_i(tb, VNL_TH_TORSO_BODY);
  const float* rcom = s + L.rcom + 3 * TB8(body_tree)[torso];  // subtree_com[torso]: torso is the root of its tree
  if (lane < 3) o.subtree_com[(size_t)e * 3 + lane] = rcom[lane];
  if (MODE == 2) {
    if (p.stats && lane < 4) p.stats[4 * e + lane] = stats[lane];
    env_sync();
    return;
  }

  // ---- task outputs: obs, traj, reward, done (envs/rodent.py:178-239 / 149-176) ---------------------------------------
  const int T = vnl_hdr_i(tb, VNL_TH_CLIP_LEN), ref_len = vnl_hdr_i(tb, VNL_TH_REF_LEN), ntrack = vnl_hdr_i(tb, VNL_TH_NTRACK);
  const int njidx = vnl_hdr_i(tb, VNL_TH_NJIDX), napp = vnl_hdr_i(tb, VNL_TH_NAPP);
  const int obs_size = vnl_hdr_i(tb, VNL_TH_OBS_SIZE), traj_size = vnl_hdr_i(tb, VNL_TH_TRAJ_SIZE), nj = d.nq - 7;
  const int* bidx = vnl_field_i(tb, VNL_T_BODY_IDXS);
  const int* eeidx = vnl_field_i(tb, VNL_T_EE_IDX);
  const int* appidx = vnl_field_i(tb, VNL_T_APP_IDX);
  const int* apprefidx = vnl_field_i(tb, VNL_T_APP_REF_IDX);
  const int* jcol = vnl_field_i(tb, VNL_T_JOINT_COL);
  const float* rbody = vnl_field_f(tb, VNL_T_BODY_POSITIONS);
  const float* rpos = vnl_field_f(tb, VNL_T_POSITION);
  const float* rjoints = vnl_field_f(tb, VNL_T_JOINTS);
  int cur_frame, sub_clip_frame;
  if (MODE == 0) { cur_frame = frame_old + 1; sub_clip_frame = p.in.sub_clip_frame[e] + 1; }
  else { cur_frame = MODE == 5 ? rstart : p.in.cur_frame[e]; sub_clip_frame = 0; }
  if (lane == 0) { o.cur_frame[e] = cur_frame; o.sub_clip_frame[e] = sub_clip_frame; if (o.clip_id) o.clip_id[e] = clip; }
  {
    float* obs = p.outputs.obs + (size_t)e * obs_size;
    for (int i = tid; i < obs_size; i += kEnvThreads) {  // [qpos, qvel (, qfrc_actuator, xpos[end effectors])]
      float v;
      if (i < d.nq) v = s[L.qpos + i];
      else if (i < d.nq + d.nv) v = s[L.qvel + i - d.nq];
      else if (i < d.nq + 2 * d.nv) v = gfa[i - d.nq - d.nv];
      else { const int k = i - d.nq - 2 * d.nv; v = gxp[3 * eeidx[k / 3] + k % 3]; }
      obs[i] = (MODE == 0) ? nan_to_num(v) : v;
    }
    float R[9];
    quat_to_mat(ld4(gxq + 4 * vnl_hdr_i(tb, VNL_TH_ROT_BODY)), R);  // rodent.py:385 xmat[1]; ant.py:333 xmat[0]
    // window start: NEW cur_frame + 1 (rodent.py:188-190); the ant hands the not yet incremented info to _get_obs (ant.py:182)
    const int wf = (MODE == 0 && vnl_hdr_i(tb, VNL_TH_TRAJ_OLD_FRAME)) ? frame_old : cur_frame;
    const int ws = fbase + min(max(wf + 1, 0), T - ref_len);
    float* traj = p.outputs.traj + (size_t)e * traj_size;
    const int n_app = ref_len * napp * 3, n_bod = ref_len * ntrack * 3, n_root = ref_len * 3;
    for (int i = tid; i < traj_size; i += kEnvThreads) {
      float v;
      if (i < n_app) {
        const int w = i / (napp * 3), r = i - w * napp * 3;
        v = rbody[((size_t)(ws + w) * ntrack + apprefidx[r / 3]) * 3 + r % 3];
      } else if (i < n_app + n_bod) {
        const int q = i - n_app, w = q / (ntrack * 3), r = q - w * ntrack * 3, b = r / 3, cl = r % 3;
        const float* rb = rbody + ((size_t)(ws + w) * ntrack + b) * 3;
        const float* xp = gxp + 3 * bidx[b];
        v = (rb[0] - xp[0]) * R[cl] + (rb[1] - xp[1]) * R[3 + cl] + (rb[2] - xp[2]) * R[6 + cl];
      } else if (i < n_app + 2 * n_bod) {
        const int q = i - n_app - n_bod, w = q / (ntrack * 3), r = q - w * ntrack * 3, b = r / 3, k = r % 3;
        v = rbody[((size_t)(ws + w) * ntrack + b) * 3 + k] - gxp[3 * bidx[b] + k];
      } else if (i < n_app + 2 * n_bod + n_root) {
        const int q = i - n_app - 2 * n_bod, w = q / 3, cl = q % 3;
        const float* rp = rpos + (size_t)(ws + w) * 3;
        v = (rp[0] - s[L.qpos]) * R[cl] + (rp[1] - s[L.qpos + 1]) * R[3 + cl] + (rp[2] - s[L.qpos + 2]) * R[6 + cl];
      } else {
        const int q = i - n_app - 2 * n_bod - n_root, w = q / njidx, j = jcol[q - w * njidx];
        v = rjoints[(size_t)(ws + w) * nj + j] - s[L.qpos + 7 + j];
      }
      traj[i] = v;
    }
  }
  if (MODE == 5) {  // the step's reward, done, metrics and stats stay; the env's next draw takes the next counter
    env_sync();
    if (tid == 0) p.rs.reset_count[e] = rcount + 1;
    return;
  }
  if (MODE == 1) {
    // info["termination_error"] of the fresh state (rodent.py:169)
    const int f = fbase + min(max(cur_frame, 0), T - 1);
    float v0 = 0.0f, v1 = 0.0f, v2 = 0.0f, v3_ = 0.0f;
    for (int j = lane; j < nj; j += 32) v0 += fabsf(rjoints[(size_t)f * nj + j] - s[L.qpos + 7 + j]);
    for (int b = lane; b < ntrack; b += 32) {
      const float* rb = rbody + ((size_t)f * ntrack + b) * 3;
      const float* xp = gxp + 3 * bidx[b];
      v1 += fabsf(rb[0] - xp[0]); v2 += fabsf(rb[1] - xp[1]); v3_ += fabsf(rb[2] - xp[2]);
    }
    v0 = warp_sum(v0); v1 = warp_sum(v1); v2 = warp_sum(v2); v3_ = warp_sum(v3_);
    float eb = fmaxf(v1, fmaxf(v2, v3_));
    if (vnl_hdr_i(tb, VNL_TH_TERM_MEAN)) { v0 = v0 / (float)nj; eb = (v1 + v2 + v3_) / (float)(3 * ntrack); }
    const float err = 0.5f * vnl_hdr_f(tb, VNL_TH_BODY_ERR_MULT) * eb + 0.5f * v0;
    if (lane == 0) {
      p.outputs.reward[e] = 0.0f; p.outputs.done[e] = 0.0f;
      float* mt = p.outputs.metrics + 7 * (size_t)e;
      for (int k = 0; k < 6; ++k) mt[k] = 0.0f;
      mt[6] = 1.0f - err / vnl_hdr_f(tb, VNL_TH_TERM_THRESHOLD);
    }
    if (p.outputs.stats && lane < 4) p.outputs.stats[4 * e + lane] = stats[lane];
    env_sync();
    return;
  }
  // _calculate_reward (rodent.py:266-316 / humanoid.py:264-311): every reference lookup uses the OLD cur_frame
  {
    const int f = fbase + min(max(frame_old, 0), T - 1);
    if (!vnl_hdr_i(tb, VNL_TH_REWARD_OLD_STATE)) rt = reward_state_terms(tb, d.nv, f, s + L.qvel, s + L.qpos, gfa, rcom);
    float v2 = 0.0f, v3_ = 0.0f;  // |app - ref|^2, nan count
    for (int i = lane; i < d.nv; i += 32)
      if (isnan(s[L.qvel + i]) || isnan(s[L.warm + i]) || isnan(gfa[i])) v3_ += 1.0f;
    for (int i = lane; i < napp * 3; i += 32) {
      const int a = i / 3, k = i % 3;
      const float df = gxp[3 * appidx[a] + k] - rbody[((size_t)f * ntrack + apprefidx[a]) * 3 + k];
      v2 += df * df;
    }
    for (int i = lane; i < d.nq; i += 32) if (isnan(s[L.qpos + i])) v3_ += 1.0f;
    for (int i = lane; i < d.nbody * 3; i += 32) if (isnan(gxp[i])) v3_ += 1.0f;
    for (int i = lane; i < d.na; i += 32) if (isnan(s[L.act + i])) v3_ += 1.0f;
    v2 = warp_sum(v2); v3_ = warp_sum(v3_);
    float r_com = rt.rcom, rvl = rt.rvel, rquat = rt.rquat, ract = rt.ract;
    if (vnl_hdr_i(tb, VNL_TH_RACT_ACTION)) {  // ant.py:251: 0.01 * -0.015 * sum(action^2) / nu on the RAW action
      float sa = 0.0f;
      for (int u = lane; u < d.nu; u += 32) { const float au = p.ctrl[(size_t)e * d.nu + u]; sa += au * au; }
      sa = warp_sum(sa);
      ract = 0.01f * -0.015f * sa / (float)d.nu;
    }
    float rapp = napp > 0 ? expf(-400.0f * sqrtf(v2)) : 0.0f;  // no appendage term in humanoid.py:200-205
    float done = rtrunk < vnl_hdr_f(tb, VNL_TH_DONE_RTRUNK) ? 1.0f : 0.0f;  // rodent.py:213 / humanoid.py:199 (before scaling)
    const float raw0 = r_com, raw1 = rvl, raw3 = rquat, raw4 = ract, raw5 = rapp;
    r_com *= vnl_hdr_f(tb, VNL_TH_W_RCOM); rvl *= vnl_hdr_f(tb, VNL_TH_W_RVEL); rapp *= vnl_hdr_f(tb, VNL_TH_W_RAPP);
    const float rtr = rtrunk * vnl_hdr_f(tb, VNL_TH_W_RTRUNK);
    rquat *= vnl_hdr_f(tb, VNL_TH_W_RQUAT); ract *= vnl_hdr_f(tb, VNL_TH_W_RACT);
    const float total = r_com + rvl + rtr + rquat + ract + rapp;
    const float sub_healthy = (!vnl_hdr_i(tb, VNL_TH_USE_SUBCLIP) || sub_clip_frame < vnl_hdr_i(tb, VNL_TH_SUB_CLIP_LEN)) ? 1.0f : 0.0f;
    done = fmaxf(1.0f - rt.healthy, done);
    done = fmaxf(1.0f - sub_healthy, done);
    if (v3_ > 0.0f) done = 1.0f;
    if (p.episode.steps_out) {  // brax EpisodeWrapper.step inside AutoResetWrapper.step (envs/wrappers/training.py)
      const float steps = (p.episode.done_in[e] > 0.0f ? 0.0f : p.episode.steps_in[e]) + 1.0f;
      const bool over = steps >= p.episode.episode_length;
      const float trunc = over ? 1.0f - done : 0.0f;
      if (over) done = 1.0f;
      if (lane == 0) { p.episode.steps_out[e] = steps; p.episode.truncation_out[e] = trunc; }
    }
    if (lane == 0) {
      p.outputs.reward[e] = nan_to_num(total);
      p.outputs.done[e] = done;
      float* mt = p.outputs.metrics + 7 * (size_t)e;
      mt[0] = r_com; mt[1] = rvl; mt[2] = rtr; mt[3] = rquat; mt[4] = ract; mt[5] = rapp; mt[6] = rtr;
      if (vnl_hdr_i(tb, VNL_TH_METRICS_RAW)) { mt[0] = raw0; mt[1] = raw1; mt[2] = rtrunk; mt[3] = raw3; mt[4] = raw4; mt[5] = raw5; mt[6] = rtrunk; }  // ant.py:203-210
    }
    if (p.outputs.stats && lane < 4) p.outputs.stats[4 * e + lane] = stats[lane];
    // brax AutoResetWrapper.step fused in: where done, the pipeline-state leaves and obs are replaced by the cached
    // first ones; info (frames, traj), reward, done and metrics are kept (SURVEY quirk Q7).
    env_sync();  // every read of the stored xpos / xquat / qfrc_actuator rows above precedes the restore below
    if (p.first.qpos && done > 0.0f) {
      const VnlState& f1 = p.first;
      for (int i = tid; i < d.nq; i += kEnvThreads) o.qpos[(size_t)e * d.nq + i] = f1.qpos[(size_t)e * d.nq + i];
      for (int i = tid; i < d.nv; i += kEnvThreads) o.qvel[(size_t)e * d.nv + i] = f1.qvel[(size_t)e * d.nv + i];
      for (int i = tid; i < d.na; i += kEnvThreads) o.act[(size_t)e * d.na + i] = f1.act[(size_t)e * d.na + i];
      for (int i = tid; i < d.nv; i += kEnvThreads) o.qacc_warmstart[(size_t)e * d.nv + i] = f1.qacc_warmstart[(size_t)e * d.nv + i];
      for (int i = tid; i < d.nbody * 3; i += kEnvThreads) o.xpos[(size_t)e * d.nbody * 3 + i] = f1.xpos[(size_t)e * d.nbody * 3 + i];
      for (int i = tid; i < d.nbody * 4; i += kEnvThreads) o.xquat[(size_t)e * d.nbody * 4 + i] = f1.xquat[(size_t)e * d.nbody * 4 + i];
      for (int i = tid; i < d.nv; i += kEnvThreads) o.qfrc_actuator[(size_t)e * d.nv + i] = f1.qfrc_actuator[(size_t)e * d.nv + i];
      if (lane < 3) o.subtree_com[(size_t)e * 3 + lane] = f1.subtree_com[(size_t)e * 3 + lane];
      if (p.first_obs)
        for (int i = tid; i < obs_size; i += kEnvThreads) p.outputs.obs[(size_t)e * obs_size + i] = p.first_obs[(size_t)e * obs_size + i];
    }
  }
  env_sync();
  pf.mark(15);
}

template <int MODE>
__global__ void __launch_bounds__(kMaxEnvs * kEnvThreads, 1) vnl_env_kernel(Params p) {
  extern __shared__ __align__(16) float smem[];
  Cta& c = *reinterpret_cast<Cta*>(smem);
  uint32_t* ktab = reinterpret_cast<uint32_t*>(smem + kCtaFloats);
  const int tid = threadIdx.x, nt = blockDim.x;
  const uint32_t* g_ktab = (const uint32_t*)vnl_field_i(p.model, VNL_F_KTAB);
  for (int i = tid; i < p.dims.ktab_words; i += nt) ktab[i] = g_ktab[i];
  for (int f = tid; f < VNL_F_MODEL_COUNT; f += nt) c.foff[f] = p.model[VNL_TABLE_OFF + 2 * f];
  if (tid == 0) {
    c.d = p.dims;
    make_layout(c.d, c.L);
    c.mb = p.model;
    c.prof = p.prof; c.prof_env = p.prof_env; c.lockstep = p.lockstep;
    c.work = p.work; c.work_stride = p.work_stride;
    const uint32_t kb = (uint32_t)(kCtaFloats * 4);  // byte offset of the staged tables in shared memory
#define TOFF(name, id) c.o_##name = kb + g_ktab[id]
    TOFF(lvl_start, VNL_KT_LVL_START); TOFF(lvl_bp, VNL_KT_LVL_BP); TOFF(parent, VNL_KT_PARENT); TOFF(child_adr, VNL_KT_CHILD_ADR);
    TOFF(child_list, VNL_KT_CHILD_LIST); TOFF(body_dofadr, VNL_KT_BODY_DOFADR); TOFF(body_dofnum, VNL_KT_BODY_DOFNUM);
    TOFF(body_tree, VNL_KT_BODY_TREE); TOFF(lastdof, VNL_KT_BODY_LASTDOF); TOFF(sub_end, VNL_KT_SUB_END); TOFF(roots, VNL_KT_ROOTS);
    TOFF(mrow, VNL_KT_MROW); TOFF(mcol, VNL_KT_MCOL); TOFF(dof_body, VNL_KT_DOF_BODY); TOFF(dpart_adr, VNL_KT_DPART_ADR); TOFF(apart_adr, VNL_KT_APART_ADR);
    TOFF(madr, VNL_KT_MADR); TOFF(erow, VNL_KT_EROW); TOFF(elvl, VNL_KT_ELVL); TOFF(desc_adr, VNL_KT_DESC_ADR); TOFF(desc_src, VNL_KT_DESC_SRC);
    TOFF(desc_k, VNL_KT_DESC_K); TOFF(ddof, VNL_KT_DDOF); TOFF(dlvl, VNL_KT_DLVL); TOFF(anc_start, VNL_KT_ANC_START); TOFF(kitem, VNL_KT_KITEM);
    TOFF(klvl, VNL_KT_KLVL); TOFF(prog_a, VNL_KT_PROG_A); TOFF(prog_d, VNL_KT_PROG_D);
#undef TOFF
    c.TA = (int)g_ktab[VNL_KT_COUNT + VNL_KS_TA]; c.TD = (int)g_ktab[VNL_KT_COUNT + VNL_KS_TD];
    c.ndslot = (int)g_ktab[VNL_KT_COUNT + VNL_KS_NDSLOT];
    c.nheight = (int)g_ktab[VNL_KT_COUNT + VNL_KS_NHEIGHT];
  }
  __syncthreads();
  const int W = nt / kEnvThreads, warp = tid / kEnvThreads;  // env slots of this CTA, this thread's slot
  const int so = kCtaFloats + align4(c.d.ktab_words) + warp * c.L.total;
  // mode 5 walks the list of envs to reset (count, then the env indices), the other modes envs 0 .. B-1.  Every CTA reads
  // the same count, so all warps of a CTA agree on the number of rounds and the lockstep barriers stay matched.
  const int n = MODE == 5 ? p.rs.scratch[0] : p.B;
  const int stride = gridDim.x * W, rounds = (n + stride - 1) / stride;
  for (int r = 0; r < rounds; ++r) {
    // slot-major env numbering: a partial last round thins out EVERY CTA (fewer co-resident envs each, all faster)
    // instead of leaving whole SMs idle next to full ones
    const int i = r * stride + warp * gridDim.x + blockIdx.x;
    env_run<MODE>(so, p, MODE == 5 ? (i < n ? p.rs.scratch[1 + i] : 0) : i, i < n);
  }
}

template __global__ void vnl_env_kernel<0>(Params);
template __global__ void vnl_env_kernel<1>(Params);
template __global__ void vnl_env_kernel<2>(Params);
template __global__ void vnl_env_kernel<3>(Params);
template __global__ void vnl_env_kernel<4>(Params);
template __global__ void vnl_env_kernel<5>(Params);

// (name, offset, size) of every array of the per-env layout, for tests/test_layout.py (sizes as make_layout reserves them)
int layout_table(const Dims& d, LayoutEntry* out, int cap) {
  Lay L;
  make_layout(d, L);
  const int nb = d.nbody, nv = d.nv, big = (nb > nv ? nb : nv) * 6;
  const LayoutEntry e[] = {
      {"qpos", L.qpos, d.nq}, {"qvel", L.qvel, nv}, {"act", L.act, d.na}, {"ctrl", L.ctrl, d.nu}, {"warm", L.warm, nv},
      {"cdof", L.cdof, 6 * nv}, {"Mdiag", L.Mdiag, nv}, {"Kdiag", L.Kdiag, nv}, {"rcom", L.rcom, 3 * d.nroot},
      {"qfrc_smooth", L.qfrc_smooth, nv}, {"qacc_smooth", L.qacc_smooth, nv}, {"act_dot", L.act_dot, d.na}, {"ints", L.ints, 16},
      {"Ms", L.Ms, d.stream ? 0 : d.nM + 1}, {"Ks", L.Ks, d.stream ? 0 : d.nM + 1},
      {"Mn", L.Mn, d.solver == 2 ? d.nM : 0}, {"H", L.H, d.solver == 2 ? nv * nv : 0}, {"jr", L.jr, d.solver == 2 ? 3 * nv : 0},
      {"xpos", L.xpos, 3 * nb}, {"xquat", L.xquat, 4 * nb}, {"cvel", L.cvel, 6 * nb},
      {"Jaref", L.Jaref, d.nefc}, {"qacc", L.qacc, nv}, {"Ma", L.Ma, nv}, {"grad", L.grad, nv}, {"Mgrad", L.Mgrad, nv},
      {"search", L.search, nv}, {"Mv", L.Mv, nv}, {"qfrc_con", L.qfrc_con, nv},
      {"xipos", L.xipos, 3 * nb}, {"xanchor", L.xanchor, 3 * d.njnt}, {"xaxis", L.xaxis, 3 * d.njnt}, {"cacc", L.cacc, big},
      {"t16", L.t16, kTS * nb}, {"part", L.part, d.naslot + d.ndslot}, {"tmpv", L.tmpv, nv},
      {"lim_dof", L.lim_dof, d.nlimit}, {"limrow_of_dof", L.limrow_of_dof, nv}, {"cbody", L.cbody, d.ncon}, {"crel", L.crel, 3 * d.ncon},
      {"cframe", L.cframe, 6 * d.ncon}, {"cmu", L.cmu, d.ncon}, {"efcD", L.efcD, d.nefc},
      {"Jv", L.Jv, d.nefc > 6 * d.ncon ? d.nefc : 6 * d.ncon}, {"K", L.K, d.nM + 40}, {"total", L.total, 0}};
  const int n = (int)(sizeof(e) / sizeof(e[0]));
  for (int i = 0; i < n && i < cap; ++i) out[i] = e[i];
  return n;
}

static int max_envs_per_cta(const Dims& d) {
  Lay L;
  make_layout(d, L);
  const int w = (227 * 1024 - (kCtaFloats + align4(d.ktab_words)) * 4) / (L.total * 4);
  return w > kMaxEnvs ? kMaxEnvs : w;
}

void decide_stream(Dims& d) {
  Dims r = d, g = d;
  r.stream = 0; g.stream = 1;
  d.stream = max_envs_per_cta(r) >= max_envs_per_cta(g) ? 0 : 1;  // resident inertia only where it costs no resident env
  static int force = -2;
  if (force == -2) { const char* ev = getenv("VNL_STREAM"); force = ev ? atoi(ev) : -1; }
  if (force == 0 || force == 1) d.stream = force;
}

LaunchInfo launch_info(const Dims& d, int B) {
  Lay L;
  make_layout(d, L);
  const int fixed = (kCtaFloats + align4(d.ktab_words)) * 4, per = L.total * 4;
  int wmax = (227 * 1024 - fixed) / per;
  if (wmax > kMaxEnvs) wmax = kMaxEnvs;
  static int env_w = -1;
  if (env_w < 0) { const char* ev = getenv("VNL_WARPS"); env_w = ev ? atoi(ev) : 0; }
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
  }
  LaunchInfo best;
  best.warps_per_cta = wmax; best.smem_bytes = fixed + (wmax > 0 ? wmax : 1) * per; best.ctas = 0;
  if (wmax < 1) return best;
  // The grid is persistent: every warp walks ceil(B / resident warps) envs.  More warps per SM only pay when they save a
  // whole round (a warp sharing the SM with more neighbours runs each env slower), so take the fewest rounds and, on a
  // tie, the fewest warps.
  long best_rounds = -1;
  for (int W = wmax; W >= 1 && (env_w > 0 || W >= wmax - 2); --W) {
    if (env_w > 0 && W != (env_w < wmax ? env_w : wmax)) continue;
    const int smem = fixed + W * per;
    int resident = (227 * 1024) / (smem + 1024);
    if (resident < 1) resident = 1;
    if (resident > 2048 / (W * kEnvThreads)) resident = 2048 / (W * kEnvThreads);
    if (resident > 65536 / (W * kEnvThreads * 128)) resident = 65536 / (W * kEnvThreads * 128);  // register file (<= 128 / thread)
    if (resident < 1) resident = 1;
    const int need = (B + W - 1) / W;
    const int ctas = need < sms * resident ? need : sms * resident;
    const long rounds = ((long)B + (long)ctas * W - 1) / ((long)ctas * W);
    if (best_rounds < 0 || rounds <= best_rounds) {
      best_rounds = rounds;
      best.warps_per_cta = W; best.smem_bytes = smem; best.ctas = ctas;
    }
  }
  return best;
}

cudaError_t launch(int mode, const Params& p, cudaStream_t stream) {
  const LaunchInfo li = launch_info(p.dims, p.B);
  if (li.warps_per_cta < 1) return cudaErrorInvalidConfiguration;  // one env does not fit in shared memory
  if (p.dims.env_warps != kEnvWarps) return cudaErrorInvalidValue;   // the blob's lane programs are for another group width
  if ((p.dims.stream != 0) != kStream) return cudaErrorInvalidValue;  // dispatched to the wrong instantiation
  void (*k)(Params) = mode == 0 ? vnl_env_kernel<0> : mode == 1 ? vnl_env_kernel<1> : mode == 2 ? vnl_env_kernel<2> : mode == 3 ? vnl_env_kernel<3>
                      : mode == 4 ? vnl_env_kernel<4> : vnl_env_kernel<5>;
  cudaError_t err = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, li.smem_bytes);
  if (err != cudaSuccess) return err;
  static int lockstep = -1;
  if (lockstep < 0) { const char* ev = getenv("VNL_LOCKSTEP"); lockstep = ev ? atoi(ev) : 3; }
  Params q = p;
  q.lockstep = lockstep;
  static int lsgroups = -1;
  if (lsgroups < 0) { const char* ev = getenv("VNL_LSGROUPS"); lsgroups = ev ? atoi(ev) : 1; }
  q.lsgroups = lsgroups < 1 ? 1 : (lsgroups > li.warps_per_cta ? li.warps_per_cta : (lsgroups > 7 ? 7 : lsgroups));
  if (q.lsgroups > 1 && lockstep >= 3) q.lockstep = 2;  // the per-phase barriers are CTA wide
  k<<<li.ctas, li.warps_per_cta * kEnvThreads, li.smem_bytes, stream>>>(q);
  return cudaGetLastError();
}

}  // namespace ewN
}  // namespace vnl
