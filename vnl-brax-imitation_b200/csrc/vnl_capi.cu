// vnl_capi.cu -- extern "C" boundary of include/vnl_b200.h.
//
// STATELESS: the model dimensions needed for the launch geometry travel with every call in a caller-owned host struct
// (VnlContext: host copies of the blobs' scalar headers + the device workspace; for the XLA custom calls the same bytes
// arrive in `opaque` and the workspace is a scratch buffer).  There is no registry, no lock and no global: the model /
// task blobs are plain device operands that may sit at a different address on every call.  No call on the step path
// copies, allocates or synchronises.
#include <cuda_runtime.h>
#include <math.h>
#include <string.h>

#include "../../include/vnl_blob.h"
#include "vnl_kernels.h"
#include "vnl_xla_status.h"

namespace {

void fill_dims(const uint32_t* w, vnl::Dims& d) {
  d.nq = vnl_hdr_i(w, VNL_MH_NQ); d.nv = vnl_hdr_i(w, VNL_MH_NV); d.nu = vnl_hdr_i(w, VNL_MH_NU); d.na = vnl_hdr_i(w, VNL_MH_NA);
  d.nbody = vnl_hdr_i(w, VNL_MH_NBODY); d.njnt = vnl_hdr_i(w, VNL_MH_NJNT); d.ngeom = vnl_hdr_i(w, VNL_MH_NGEOM);
  d.npair = vnl_hdr_i(w, VNL_MH_NPAIR); d.ncon = vnl_hdr_i(w, VNL_MH_NCON); d.nlimit = vnl_hdr_i(w, VNL_MH_NLIMIT);
  d.nefc = vnl_hdr_i(w, VNL_MH_NEFC); d.nM = vnl_hdr_i(w, VNL_MH_NM); d.nlevel = vnl_hdr_i(w, VNL_MH_NLEVEL);
  d.maxdepth = vnl_hdr_i(w, VNL_MH_MAXDEPTH); d.nroot = vnl_hdr_i(w, VNL_MH_NROOT); d.ndslot = vnl_hdr_i(w, VNL_MH_NDSLOT); d.env_warps = vnl_hdr_i(w, VNL_MH_ENV_WARPS); d.naslot = vnl_hdr_i(w, VNL_MH_NASLOT); d.TA = vnl_hdr_i(w, VNL_MH_TA); d.TD = vnl_hdr_i(w, VNL_MH_TD); d.ktab_words = (int)w[VNL_TABLE_OFF + 2 * VNL_F_KTAB + 1];
  d.solver = vnl_hdr_i(w, VNL_MH_SOLVER); d.iterations = vnl_hdr_i(w, VNL_MH_ITERATIONS);
  d.ls_iterations = vnl_hdr_i(w, VNL_MH_LS_ITERATIONS); d.eulerdamp = vnl_hdr_i(w, VNL_MH_EULERDAMP);
  d.timestep = vnl_hdr_f(w, VNL_MH_TIMESTEP); d.gx = vnl_hdr_f(w, VNL_MH_GRAVITY_X); d.gy = vnl_hdr_f(w, VNL_MH_GRAVITY_Y);
  d.gz = vnl_hdr_f(w, VNL_MH_GRAVITY_Z); d.tolerance = vnl_hdr_f(w, VNL_MH_TOLERANCE); d.ls_tolerance = vnl_hdr_f(w, VNL_MH_LS_TOLERANCE);
  d.impratio = vnl_hdr_f(w, VNL_MH_IMPRATIO); d.meaninertia = vnl_hdr_f(w, VNL_MH_MEANINERTIA);
  const int nb = d.nbody, nv = d.nv;
  d.dump_xpos = 0;
  d.dump_xipos = nb * 3 + nb * 4 + nb * 9;
  d.dump_xanchor = d.dump_xipos + nb * 3 + nb * 9;
  d.dump_subtree_com = d.dump_xanchor + d.njnt * 6;
  d.dump_cinert = d.dump_subtree_com + nb * 3;
  d.dump_qM = d.dump_cinert + nb * 10 + nv * 6 + nb * 10;
  d.dump_cvel = d.dump_qM + nv * nv;
  d.dump_passive = d.dump_cvel + nb * 6 + nv * 6;
  d.dump_con = d.dump_passive + 5 * nv + d.na;
  d.dump_efc = d.dump_con + 13 * d.ncon;
  d.dump_qacc = d.dump_efc + 3 * d.nefc + d.nefc * nv;
  d.dump_total = d.dump_qacc + 2 * nv + d.nefc + 4;
  vnl::any_decide_stream(d);
}

int check_blob(const void* host, size_t nbytes, uint32_t magic, int nfields) {
  if (!host || nbytes < sizeof(uint32_t) * VNL_DATA_OFF) return -1;
  const uint32_t* w = (const uint32_t*)host;
  if (w[0] != magic) return -2;
  if (w[1] != VNL_BLOB_VERSION) return -3;
  if ((size_t)w[2] * 4 != nbytes) return -4;
  if ((int)w[3] != nfields) return -5;
  for (int f = 0; f < nfields; ++f) {
    const uint64_t off = w[VNL_TABLE_OFF + 2 * f], n = w[VNL_TABLE_OFF + 2 * f + 1];
    if (off < VNL_DATA_OFF || off + n > w[2]) return -6;
  }
  return 0;
}

// Argument checks + launch parameters common to every entry point.  `B` is the ACTUAL batch: the workspace bound is
// checked against the geometry this very launch will use.
int prepare(const VnlContext* ctx, const void* model, const void* task, bool need_task, int B, vnl::Params& p) {
  if (!ctx || !model) return -10;
  if (ctx->model_hdr[0] != VNL_MAGIC_MODEL || ctx->model_hdr[1] != VNL_BLOB_VERSION) return -11;
  fill_dims(ctx->model_hdr, p.dims);
  if (p.dims.stream) {
    if (!ctx->workspace) return -20;
    const vnl::LaunchInfo li = vnl::any_launch_info(p.dims, B);
    p.work_stride = vnl::work_stride(p.dims);
    if ((uint64_t)li.ctas * li.warps_per_cta * p.work_stride * sizeof(float) > ctx->workspace_bytes) return -21;
    p.work = static_cast<float*>(ctx->workspace);
  }
  p.model = (const uint32_t*)model;
  p.task = (const uint32_t*)task;
  if (need_task) {
    if (!task) return -12;
    if (ctx->task_hdr[0] != VNL_MAGIC_TASK || ctx->task_hdr[1] != VNL_BLOB_VERSION) return -13;
  }
  return 0;
}

}  // namespace

__global__ void vnl_ffma_probe_kernel(int iters, float* out) {
  float a[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) a[k] = 1.0f + 1e-3f * (float)(threadIdx.x + k);
  const float m = 0.9999f, c = 1e-4f;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int k = 0; k < 16; ++k) a[k] = fmaf(a[k], m, c);
  }
  float s = 0.0f;
#pragma unroll
  for (int k = 0; k < 16; ++k) s += a[k];
  if (s == 123.456f) out[blockIdx.x * blockDim.x + threadIdx.x] = s;  // keeps the chains alive; practically never true
}

// compute_velocity_from_kinematics + the joint-velocity clip of process_clip (preprocessing/mjx_preprocess.py:88-105,
// 170-193; quaternion helpers preprocessing/transformations.py:86-139), one thread per (clip, frame, column block).
// The trajectory is padded with its last frame (mjx_preprocess.py:91), so the last frame's velocity is zero.  Works on the
// RAW qpos (the reference differentiates mocap_qpos, not the kinematics-normalised copy).
__global__ void clip_velocity_kernel(const float* __restrict__ qpos, int nclips, int T, int nq, float dt, float max_qvel,
                                     float* __restrict__ qvel) {
  const int nv = nq - 1;
  const long long total = (long long)nclips * T * nv;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int col = (int)(idx % nv);
    const long long row = idx / nv;
    const int t = (int)(row % T);
    const float* q0 = qpos + row * nq;
    const float* q1 = (t + 1 < T) ? q0 + nq : q0;  // padded frame = the last one
    float v;
    if (col < 3) {
      v = (q1[col] - q0[col]) / dt;
    } else if (col < 6) {
      // quat_diff(source, target) = conj(source) * target, normalised, then quat_to_axisangle / dt
      const float sw = q0[3], sx = -q0[4], sy = -q0[5], sz = -q0[6];
      const float tw = q1[3], tx = q1[4], ty = q1[5], tz = q1[6];
      float d[4] = {sw * tw - sx * tx - sy * ty - sz * tz, sw * tx + sx * tw + sy * tz - sz * ty,
                    sw * ty - sx * tz + sy * tw + sz * tx, sw * tz + sx * ty - sy * tx + sz * tw};
      const float n = sqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2] + d[3] * d[3]);
      for (int k = 0; k < 4; ++k) d[k] /= n;
      float angle = 2.0f * acosf(fminf(fmaxf(d[0], -1.0f), 1.0f));
      if (angle < 1e-10f) {
        v = 0.0f;
      } else {
        const float qn = sinf(angle / 2.0f);
        const float pi = 3.14159265358979323846f, x = angle + pi;
        angle = (x - floorf(x / (2.0f * pi)) * (2.0f * pi)) - pi;  // python floor-mod
        v = d[1 + col - 3] / qn * angle / dt;
      }
    } else {
      v = (q1[col + 1] - q0[col + 1]) / dt;
      v = fminf(fmaxf(v, -max_qvel), max_qvel);
    }
    qvel[row * nv + col] = v;
  }
}

// The envs a step finished, in ascending order: list[0] = their count, list[1 ..] = their indices (the work list of the
// resampling reset, env-kernel mode 5).  One CTA walks the batch 1024 envs at a time with a block-wide ballot scan, so the
// list -- and with it which warp resets which env -- is the same on every run.
__global__ void __launch_bounds__(1024) done_list_kernel(const float* __restrict__ done, int B, int32_t* __restrict__ list) {
  __shared__ int wsum[32];
  __shared__ int base;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  if (tid == 0) base = 0;
  __syncthreads();
  for (int i0 = 0; i0 < B; i0 += 1024) {
    const int i = i0 + tid;
    const bool f = i < B && done[i] > 0.0f;
    const unsigned m = __ballot_sync(0xffffffffu, f);
    if (lane == 0) wsum[w] = __popc(m);
    __syncthreads();
    int off = base;
    for (int k = 0; k < w; ++k) off += wsum[k];
    if (f) list[1 + off + __popc(m & ((1u << lane) - 1u))] = i;
    __syncthreads();
    if (tid == 0) { int t = base; for (int k = 0; k < 32; ++k) t += wsum[k]; base = t; }
    __syncthreads();
  }
  if (tid == 0) list[0] = base;
}

extern "C" {

const char* vnl_version(void) { return "vnl_b200 0.1 (sm_100a)"; }

int vnl_check_model(const void* model_host, size_t nbytes) { return check_blob(model_host, nbytes, VNL_MAGIC_MODEL, VNL_F_MODEL_COUNT); }
int vnl_check_task(const void* task_host, size_t nbytes) { return check_blob(task_host, nbytes, VNL_MAGIC_TASK, VNL_TASK_COUNT); }

int vnl_context_init(VnlContext* ctx, const void* model_host, size_t model_bytes, const void* task_host, size_t task_bytes) {
  if (!ctx) return -1;
  memset(ctx, 0, sizeof(*ctx));
  int rc = vnl_check_model(model_host, model_bytes);
  if (rc) return rc;
  memcpy(ctx->model_hdr, model_host, sizeof(ctx->model_hdr));
  if (task_host) {
    rc = vnl_check_task(task_host, task_bytes);
    if (rc) return rc - 100;
    memcpy(ctx->task_hdr, task_host, sizeof(ctx->task_hdr));
  }
  return 0;
}

size_t vnl_workspace_bytes(const void* model_host) {
  vnl::Dims d;
  fill_dims((const uint32_t*)model_host, d);
  if (!d.stream) return 0;
  // bound over every geometry launch_info can pick on this device: batch sizes from one CTA's worth to many rounds
  size_t best = 0;
  for (int B = 1; B <= (1 << 20); B <<= 1) {
    const vnl::LaunchInfo li = vnl::any_launch_info(d, B);
    const size_t n = (size_t)li.ctas * li.warps_per_cta;
    if (n > best) best = n;
  }
  const vnl::LaunchInfo li = vnl::any_launch_info(d, (1 << 20) + 12345);
  if ((size_t)li.ctas * li.warps_per_cta > best) best = (size_t)li.ctas * li.warps_per_cta;
  return best * vnl::work_stride(d) * sizeof(float);
}

int vnl_step_smem_bytes(const void* model_host) {
  vnl::Dims d;
  fill_dims((const uint32_t*)model_host, d);
  return vnl::any_launch_info(d, 1 << 20).smem_bytes;
}

int vnl_envs_per_cta(const void* model_host) {
  vnl::Dims d;
  fill_dims((const uint32_t*)model_host, d);
  return vnl::any_launch_info(d, 1 << 20).warps_per_cta;
}

int vnl_resident_envs(const void* model_host) {
  vnl::Dims d;
  fill_dims((const uint32_t*)model_host, d);
  const vnl::LaunchInfo li = vnl::any_launch_info(d, 1 << 20);
  return li.ctas * li.warps_per_cta;
}

int vnl_debug_layout(const void* model_host, const char** names, int32_t* offsets, int32_t* sizes, int cap) {
  vnl::Dims d;
  fill_dims((const uint32_t*)model_host, d);
  vnl::LayoutEntry e[64];
  const int n = vnl::ew1s1::layout_table(d, e, 64);
  for (int i = 0; i < n && i < cap; ++i) { names[i] = e[i].name; offsets[i] = e[i].offset; sizes[i] = e[i].size; }
  return n;
}

size_t vnl_dump_size(const void* model_host) {
  vnl::Dims d;
  fill_dims((const uint32_t*)model_host, d);
  return (size_t)d.dump_total;
}

int vnl_step(const VnlContext* ctx, const void* model, const void* task, int B, const VnlState* in, const float* action, const VnlState* out,
             const VnlOutputs* outputs, void* stream) {
  if (B <= 0 || !in || !out || !outputs || !action) return -1;
  vnl::Params p;
  memset(&p, 0, sizeof(p));
  int rc = prepare(ctx, model, task, true, B, p);
  if (rc) return rc;
  p.B = B; p.nsteps = vnl_hdr_i(ctx->task_hdr, VNL_TH_NFRAMES); p.in = *in; p.out = *out; p.ctrl = action; p.outputs = *outputs;
  return (int)vnl::any_launch(0, p, (cudaStream_t)stream);
}

int vnl_step_autoreset(const VnlContext* ctx, const void* model, const void* task, int B, const VnlState* in, const float* action, const VnlState* out,
                       const VnlOutputs* outputs, const VnlState* first, const float* first_obs, void* stream) {
  if (B <= 0 || !in || !out || !outputs || !action || !first || !first->qpos) return -1;
  vnl::Params p;
  memset(&p, 0, sizeof(p));
  int rc = prepare(ctx, model, task, true, B, p);
  if (rc) return rc;
  p.B = B; p.nsteps = vnl_hdr_i(ctx->task_hdr, VNL_TH_NFRAMES); p.in = *in; p.out = *out; p.ctrl = action; p.outputs = *outputs;
  p.first = *first; p.first_obs = first_obs;
  return (int)vnl::any_launch(0, p, (cudaStream_t)stream);
}

int vnl_step_training(const VnlContext* ctx, const void* model, const void* task, int B, const VnlState* in, const float* action, const VnlState* out,
                      const VnlOutputs* outputs, const VnlState* first, const float* first_obs, const VnlEpisode* episode,
                      void* stream) {
  if (B <= 0 || !in || !out || !outputs || !action || !first || !first->qpos || !episode) return -1;
  if (!episode->steps_in || !episode->done_in || !episode->steps_out || !episode->truncation_out) return -1;
  vnl::Params p;
  memset(&p, 0, sizeof(p));
  int rc = prepare(ctx, model, task, true, B, p);
  if (rc) return rc;
  p.B = B; p.nsteps = vnl_hdr_i(ctx->task_hdr, VNL_TH_NFRAMES); p.in = *in; p.out = *out; p.ctrl = action; p.outputs = *outputs;
  p.first = *first; p.first_obs = first_obs; p.episode = *episode;
  return (int)vnl::any_launch(0, p, (cudaStream_t)stream);
}

int vnl_step_training_resample(const VnlContext* ctx, const void* model, const void* task, int B, const VnlState* in, const float* action,
                               const VnlState* out, const VnlOutputs* outputs, const VnlEpisode* episode, const VnlResample* rs,
                               void* stream) {
  if (B <= 0 || !in || !out || !outputs || !outputs->done || !action || !episode || !rs) return -1;
  if (!episode->steps_in || !episode->done_in || !episode->steps_out || !episode->truncation_out) return -1;
  if (!rs->reset_count || !rs->scratch || rs->start_frame_hi <= 0 || !(rs->noise_scale >= 0.0f) || !isfinite(rs->noise_scale)) return -1;
  // every drawn start must have its whole reference window (frames start + 1 .. start + ref_len) inside the clip, so that no
  // lookup of the reset has to be clamped: start_frame_hi <= clip length - ref_len (host-side header, no CUDA call)
  if (ctx && rs->start_frame_hi > vnl_hdr_i(ctx->task_hdr, VNL_TH_CLIP_LEN) - vnl_hdr_i(ctx->task_hdr, VNL_TH_REF_LEN)) return -1;
  vnl::Params p;
  memset(&p, 0, sizeof(p));
  int rc = prepare(ctx, model, task, true, B, p);
  if (rc) return rc;
  const cudaStream_t st = (cudaStream_t)stream;
  p.B = B; p.nsteps = vnl_hdr_i(ctx->task_hdr, VNL_TH_NFRAMES); p.in = *in; p.out = *out; p.ctrl = action; p.outputs = *outputs;
  p.episode = *episode;  // p.first stays empty: no first-state restore
  cudaError_t err = vnl::any_launch(0, p, st);
  if (err != cudaSuccess) return (int)err;
  done_list_kernel<<<1, 1024, 0, st>>>(outputs->done, B, rs->scratch);
  err = cudaGetLastError();
  if (err != cudaSuccess) return (int)err;
  p.rs = *rs;  // the launch geometry stays that of B envs; the kernel walks only the listed ones
  return (int)vnl::any_launch(5, p, st);
}

// Developer hook: vnl_step with per-phase clock64 accumulation for CTA `block` into prof[32].
int vnl_step_profiled(const VnlContext* ctx, const void* model, const void* task, int B, const VnlState* in, const float* action, const VnlState* out,
                      const VnlOutputs* outputs, void* stream, long long* prof, int block) {
  if (B <= 0 || !in || !out || !outputs || !action) return -1;
  vnl::Params p;
  memset(&p, 0, sizeof(p));
  int rc = prepare(ctx, model, task, true, B, p);
  if (rc) return rc;
  p.B = B; p.nsteps = vnl_hdr_i(ctx->task_hdr, VNL_TH_NFRAMES); p.in = *in; p.out = *out; p.ctrl = action; p.outputs = *outputs;
  p.prof = prof; p.prof_env = block;
  return (int)vnl::any_launch(0, p, (cudaStream_t)stream);
}

int vnl_reset(const VnlContext* ctx, const void* model, const void* task, int B, const VnlState* in, const VnlState* out, const VnlOutputs* outputs,
              void* stream) {
  if (B <= 0 || !in || !out || !outputs) return -1;
  vnl::Params p;
  memset(&p, 0, sizeof(p));
  int rc = prepare(ctx, model, task, true, B, p);
  if (rc) return rc;
  p.B = B; p.nsteps = 1; p.in = *in; p.out = *out; p.outputs = *outputs;
  return (int)vnl::any_launch(1, p, (cudaStream_t)stream);
}

int vnl_pipeline_step(const VnlContext* ctx, const void* model, int B, int nsteps, const VnlState* in, const float* ctrl, const VnlState* out,
                      int32_t* stats, void* stream) {
  if (B <= 0 || nsteps <= 0 || !in || !out) return -1;
  vnl::Params p;
  memset(&p, 0, sizeof(p));
  int rc = prepare(ctx, model, nullptr, false, B, p);
  if (rc) return rc;
  p.B = B; p.nsteps = nsteps; p.in = *in; p.out = *out; p.ctrl = ctrl; p.stats = stats;
  return (int)vnl::any_launch(2, p, (cudaStream_t)stream);
}

int vnl_forward_dump(const VnlContext* ctx, const void* model, int B, const VnlState* in, const float* ctrl, float* dump, void* stream) {
  if (B <= 0 || !in || !dump) return -1;
  vnl::Params p;
  memset(&p, 0, sizeof(p));
  int rc = prepare(ctx, model, nullptr, false, B, p);
  if (rc) return rc;
  p.B = B; p.nsteps = 1; p.in = *in; p.ctrl = ctrl; p.dump = dump;
  cudaError_t err = cudaMemsetAsync(dump, 0xFF, (size_t)B * p.dims.dump_total * sizeof(float), (cudaStream_t)stream);
  if (err != cudaSuccess) return (int)err;
  return (int)vnl::any_launch(3, p, (cudaStream_t)stream);
}

// process_clip on the GPU (SURVEY 8 row f4): kinematics of every frame with the env kernel's own kinematic pass (mode 4:
// one warp per frame) + one elementwise kernel for the finite-difference velocities.
int vnl_process_clip(const VnlContext* ctx, const void* model, int nclips, int T, const float* qpos, float dt, float max_qvel,
                     float* qpos_out, float* body_positions, float* body_quaternions, float* qvel_out, void* stream) {
  if (nclips <= 0 || T <= 0 || !qpos || !qpos_out || !body_positions || !body_quaternions || !qvel_out || !(dt > 0.0f)) return -1;
  if ((long long)nclips * T > (1 << 24)) return -2;
  const int B = nclips * T;
  vnl::Params p;
  memset(&p, 0, sizeof(p));
  int rc = prepare(ctx, model, nullptr, false, B, p);
  if (rc) return rc;
  p.B = B; p.nsteps = 1;
  p.in.qpos = const_cast<float*>(qpos);
  p.out.qpos = qpos_out; p.out.xpos = body_positions; p.out.xquat = body_quaternions;
  cudaError_t err = vnl::any_launch(4, p, (cudaStream_t)stream);
  if (err != cudaSuccess) return (int)err;
  const long long total = (long long)B * (p.dims.nq - 1);
  const int threads = 256;
  long long blocks = (total + threads - 1) / threads;
  if (blocks > 148 * 16) blocks = 148 * 16;
  clip_velocity_kernel<<<(int)blocks, threads, 0, (cudaStream_t)stream>>>(qpos, nclips, T, p.dims.nq, dt, max_qvel, qvel_out);
  return (int)cudaGetLastError();
}

// XLA custom calls (status-returning legacy ABI), stateless: see include/vnl_b200.h for the buffer list.
static void unpack(void** b, int first, VnlState& s) {
  s.qpos = (float*)b[first]; s.qvel = (float*)b[first + 1]; s.act = (float*)b[first + 2]; s.qacc_warmstart = (float*)b[first + 3];
  s.xpos = (float*)b[first + 4]; s.xquat = (float*)b[first + 5]; s.subtree_com = (float*)b[first + 6];
  s.qfrc_actuator = (float*)b[first + 7]; s.cur_frame = (int32_t*)b[first + 8]; s.sub_clip_frame = (int32_t*)b[first + 9];
  s.clip_id = (int32_t*)b[first + 10];
}
static int xla_call(bool reset, void* stream, void** buffers, const char* opaque, size_t opaque_len) {
  if (!buffers || !opaque || opaque_len < sizeof(VnlXlaOpaque)) return -30;
  VnlXlaOpaque op;  // opaque bytes carry no alignment guarantee
  memcpy(&op, opaque, sizeof(op));
  if (op.version != VNL_XLA_OPAQUE_VERSION) return -31;
  VnlContext ctx;
  memcpy(ctx.model_hdr, op.model_hdr, sizeof(ctx.model_hdr));
  memcpy(ctx.task_hdr, op.task_hdr, sizeof(ctx.task_hdr));
  ctx.workspace = buffers[VNL_XLA_STEP_NBUF - 1];
  ctx.workspace_bytes = op.workspace_bytes;
  VnlState in, out;
  unpack(buffers, 2, in);
  unpack(buffers, 14, out);
  VnlOutputs o;
  o.obs = (float*)buffers[25]; o.traj = (float*)buffers[26]; o.reward = (float*)buffers[27]; o.done = (float*)buffers[28];
  o.metrics = (float*)buffers[29]; o.stats = (int32_t*)buffers[30];
  if (reset) return vnl_reset(&ctx, buffers[0], buffers[1], op.B, &in, &out, &o, stream);
  return vnl_step(&ctx, buffers[0], buffers[1], op.B, &in, (const float*)buffers[13], &out, &o, stream);
}
int vnl_xla_step_rc(void* stream, void** buffers, const char* opaque, size_t opaque_len) { return xla_call(false, stream, buffers, opaque, opaque_len); }
int vnl_xla_reset_rc(void* stream, void** buffers, const char* opaque, size_t opaque_len) { return xla_call(true, stream, buffers, opaque, opaque_len); }
void vnl_xla_step(void* stream, void** buffers, const char* opaque, size_t opaque_len, void* status) {
  vnl::xla_report(status, "vnl_xla_step", xla_call(false, stream, buffers, opaque, opaque_len));
}
void vnl_xla_reset(void* stream, void** buffers, const char* opaque, size_t opaque_len, void* status) {
  vnl::xla_report(status, "vnl_xla_reset", xla_call(true, stream, buffers, opaque, opaque_len));
}
int vnl_xla_make_opaque(const VnlContext* ctx, int B, VnlXlaOpaque* opaque) {
  if (!ctx || !opaque || B <= 0) return -1;
  memset(opaque, 0, sizeof(*opaque));
  opaque->B = B; opaque->version = VNL_XLA_OPAQUE_VERSION;
  memcpy(opaque->model_hdr, ctx->model_hdr, sizeof(opaque->model_hdr));
  memcpy(opaque->task_hdr, ctx->task_hdr, sizeof(opaque->task_hdr));
  opaque->workspace_bytes = ctx->workspace_bytes;
  return 0;
}

// Measurement helper for bench.py: an FFMA-saturating microkernel (8 independent chains per thread) that gives the
// FP32 CUDA-core roofline denominator on the device the benchmark runs on.  flops = blocks * 256 * iters * 16 * 2.
int vnl_ffma_probe(int blocks, int iters, float* out, void* stream) {
  if (blocks <= 0 || iters <= 0 || !out) return -1;
  vnl_ffma_probe_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(iters, out);
  return (int)cudaGetLastError();
}

}  // extern "C"
