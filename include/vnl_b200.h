/*
 * vnl_b200.h -- C ABI of the B200-native fused MJX-style physics + imitation-reward step.
 *
 * This is the drop-in boundary for the hot path of talmolab/VNL-Brax-Imitation:
 *
 *   vnl_step   replaces  RodentTracking.step          (reference envs/rodent.py:178-239)
 *              = PipelineEnv.pipeline_step (n_frames x mjx.step, envs/rodent.py:181)
 *              + _get_obs / _get_traj      (envs/rodent.py:318-382)
 *              + _calculate_reward / _calculate_termination (envs/rodent.py:241-316)
 *              + done / NaN guard          (envs/rodent.py:207-225)
 *   vnl_reset  replaces  RodentTracking.reset after the RNG draw
 *              = pipeline_init (mjx.forward, envs/rodent.py:148) + obs/traj/termination
 *              (envs/rodent.py:149-176)
 *
 * The reference has no FFI of its own (it is pure Python/JAX; the arithmetic lives in
 * mujoco-mjx, reached through brax).  The binding a maintainer adds is a jax.ffi / XLA
 * custom call whose operands are exactly the device buffers below (INTEGRATION.md).
 *
 * Conventions
 *   - every array is a caller-allocated DEVICE buffer, fp32 / int32, batch-major contiguous
 *     [B, n]; the library allocates nothing per call, keeps NO global state (no registry, no lock), only
 *     enqueues work on `stream` (a cudaStream_t passed as void*), never synchronises and is
 *     CUDA-graph capturable.
 *   - `model` and `task` are device copies of the flat blobs described below (constant
 *     tables; pass them as operands so the caller owns their lifetime).  They may live at a
 *     different device address on every call (XLA copies / donates / replicates operands).
 *   - `ctx` is a small HOST struct (VnlContext) the caller fills once per model: the host copy
 *     of the blobs' scalar headers (launch geometry) and the caller-owned device workspace.
 *     It is read-only for the library: nothing is cached between calls, there is no registry,
 *     no lock and no global state; two host threads may call concurrently as long as each
 *     passes its own workspace (one workspace serves one stream at a time).
 *   - return value 0 = ok, negative = argument error, positive = cudaError_t of the launch.
 *     Numerical failure is data, not an error (nan flag -> done = 1, NaN -> 0).
 */
#ifndef VNL_B200_H_
#define VNL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------
 * Blob container: an array of 32-bit words.
 *   words[0]            magic  (VNL_MAGIC_MODEL / VNL_MAGIC_TASK)
 *   words[1]            version
 *   words[2]            total number of words
 *   words[3]            number of fields in the table
 *   words[4 .. 63]      scalar header (ints, and floats stored by bit pattern), see enums
 *   words[64 + 2f]      word offset of field f (16-byte aligned)   } f < VNL_MAX_FIELDS
 *   words[64 + 2f + 1]  element count of field f                   }
 *   words[VNL_DATA_OFF ..] data
 * ---------------------------------------------------------------------------------------- */
#define VNL_MAGIC_MODEL 0x4d4c4e56u /* "VNLM" */
#define VNL_MAGIC_TASK 0x544c4e56u  /* "VNLT" */
#define VNL_BLOB_VERSION 7
#define VNL_TABLE_OFF 64
#define VNL_MAX_FIELDS 96
#define VNL_DATA_OFF (VNL_TABLE_OFF + 2 * VNL_MAX_FIELDS)

/* scalar header slots of a MODEL blob (word index) */
enum VnlModelHdr {
  VNL_MH_NQ = 4, VNL_MH_NV, VNL_MH_NU, VNL_MH_NA, VNL_MH_NBODY, VNL_MH_NJNT, VNL_MH_NGEOM,
  VNL_MH_NPAIR,       /* static geom pairs */
  VNL_MH_NCON,        /* contacts always emitted (capsule pair = 2) */
  VNL_MH_NLIMIT,      /* limited hinge joints */
  VNL_MH_NEFC,        /* nlimit + 4 * ncon (pyramidal, condim 3) */
  VNL_MH_SOLVER,      /* 1 = CG, 2 = Newton */
  VNL_MH_ITERATIONS, VNL_MH_LS_ITERATIONS,
  VNL_MH_EULERDAMP,   /* 1 = implicit joint damping in the Euler integrator */
  VNL_MH_NM,          /* tree-sparse entries of the joint-space inertia */
  VNL_MH_NLEVEL,      /* body-tree depth (levels below the world body) */
  VNL_MH_MAXDEPTH,    /* longest dof ancestor chain */
  VNL_MH_NROOT,       /* kinematic trees (bodies whose parent is the world) */
  VNL_MH_NDSLOT,      /* partial-sum slots of the descendant mat-vec program (= KTAB scalar VNL_KS_NDSLOT) */
  VNL_MH_ENV_WARPS,   /* warps cooperating on one env (1 or 2): the mat-vec lane programs have 32 * this many lanes */
  VNL_MH_NASLOT,      /* partial-sum slots of the ancestor mat-vec program */
  VNL_MH_TA,          /* steps of the ancestor / descendant mat-vec programs (= KTAB scalars VNL_KS_TA / VNL_KS_TD) */
  VNL_MH_TD,
  /* floats (bit patterns) */
  VNL_MH_TIMESTEP = 32, VNL_MH_GRAVITY_X, VNL_MH_GRAVITY_Y, VNL_MH_GRAVITY_Z,
  VNL_MH_TOLERANCE, VNL_MH_LS_TOLERANCE, VNL_MH_IMPRATIO, VNL_MH_MEANINERTIA
};

/* fields of a MODEL blob.  i = int32, f = float32; shapes in comments */
enum VnlModelField {
  VNL_F_BODY_PARENTID = 0, /* i [nbody] */
  VNL_F_BODY_ROOTID,       /* i [nbody] */
  VNL_F_BODY_JNTADR,       /* i [nbody] */
  VNL_F_BODY_JNTNUM,       /* i [nbody] */
  VNL_F_BODY_DOFADR,       /* i [nbody] */
  VNL_F_BODY_DOFNUM,       /* i [nbody] */
  VNL_F_BODY_POS,          /* f [nbody,3] */
  VNL_F_BODY_QUAT,         /* f [nbody,4] */
  VNL_F_BODY_IPOS,         /* f [nbody,3] */
  VNL_F_BODY_IQUAT,        /* f [nbody,4] */
  VNL_F_BODY_MASS,         /* f [nbody] */
  VNL_F_BODY_INERTIA,      /* f [nbody,3] */
  VNL_F_BODY_INVWEIGHT0,   /* f [nbody,2] */
  VNL_F_JNT_TYPE,          /* i [njnt] 0 free, 3 hinge */
  VNL_F_JNT_QPOSADR,       /* i [njnt] */
  VNL_F_JNT_DOFADR,        /* i [njnt] */
  VNL_F_JNT_BODYID,        /* i [njnt] */
  VNL_F_JNT_LIMITED,       /* i [njnt] */
  VNL_F_JNT_POS,           /* f [njnt,3] */
  VNL_F_JNT_AXIS,          /* f [njnt,3] */
  VNL_F_JNT_STIFFNESS,     /* f [njnt] */
  VNL_F_JNT_RANGE,         /* f [njnt,2] */
  VNL_F_JNT_MARGIN,        /* f [njnt] */
  VNL_F_JNT_SOLREF,        /* f [njnt,2] */
  VNL_F_JNT_SOLIMP,        /* f [njnt,5] */
  VNL_F_DOF_BODYID,        /* i [nv] */
  VNL_F_DOF_JNTID,         /* i [nv] */
  VNL_F_DOF_PARENTID,      /* i [nv] */
  VNL_F_DOF_ARMATURE,      /* f [nv] */
  VNL_F_DOF_DAMPING,       /* f [nv] */
  VNL_F_DOF_INVWEIGHT0,    /* f [nv] */
  VNL_F_QPOS0,             /* f [nq] */
  VNL_F_QPOS_SPRING,       /* f [nq] */
  VNL_F_GEOM_TYPE,         /* i [ngeom] */
  VNL_F_GEOM_BODYID,       /* i [ngeom] */
  VNL_F_GEOM_POS,          /* f [ngeom,3] */
  VNL_F_GEOM_QUAT,         /* f [ngeom,4] */
  VNL_F_GEOM_SIZE,         /* f [ngeom,3] */
  VNL_F_ACT_DOFADR,        /* i [nu] */
  VNL_F_ACT_CTRLLIMITED,   /* i [nu] */
  VNL_F_ACT_FORCELIMITED,  /* i [nu] */
  VNL_F_ACT_DYNTYPE,       /* i [nu] 0 none, 2 filter */
  VNL_F_ACT_ACTADR,        /* i [nu] -1 if stateless */
  VNL_F_ACT_GAIN,          /* f [nu] */
  VNL_F_ACT_GEAR,          /* f [nu] */
  VNL_F_ACT_CTRLRANGE,     /* f [nu,2] */
  VNL_F_ACT_FORCERANGE,    /* f [nu,2] */
  VNL_F_ACT_DYNPRM,        /* f [nu] */
  VNL_F_PAIR_GEOM1,        /* i [npair] the plane */
  VNL_F_PAIR_GEOM2,        /* i [npair] */
  VNL_F_PAIR_TYPE,         /* i [npair] geom type of geom2 */
  VNL_F_PAIR_FRICTION,     /* f [npair,5] */
  VNL_F_PAIR_SOLREF,       /* f [npair,2] */
  VNL_F_PAIR_SOLIMP,       /* f [npair,5] */
  VNL_F_PAIR_INCLUDEMARGIN,/* f [npair] */
  /* ---- derived tables used by the CUDA kernels (host-precomputed, see model_blob.py) ---- */
  VNL_F_LEVEL_START,       /* i [nlevel+1] offsets into LEVEL_BODY (level 0 = children of world) */
  VNL_F_LEVEL_BODY,        /* i [nbody-1] bodies sorted by depth */
  VNL_F_DOF_MADR,          /* i [nv+1] start of dof i's row in the sparse inertia (diagonal first,
                              then ancestors walking to the root -- MuJoCo qM order) */
  VNL_F_M_COL,             /* i [nM] column (ancestor dof) of each sparse entry */
  VNL_F_DOF_DEPTH,         /* i [nv] number of ancestors */
  VNL_F_BODY_SUBTREE_END,  /* i [nbody] bodies b .. end-1 are b's subtree (ids are DFS preorder) */
  VNL_F_LIMIT_JNT,         /* i [nlimit] joint id of each limit row */
  VNL_F_CON_PAIR,          /* i [ncon] pair of each emitted contact */
  VNL_F_CON_SIGN,          /* f [ncon] capsule end (+1 / -1), 0 for single-contact geoms */
  VNL_F_GEOMC_BODY,        /* i [npair] body of geom2 */
  VNL_F_GEOMC_POS,         /* f [npair,3] geom2 frame in its body */
  VNL_F_GEOMC_MAT,         /* f [npair,9] */
  VNL_F_PLANE_POS,         /* f [npair,3] plane (geom1) world frame; planes are static */
  VNL_F_PLANE_MAT,         /* f [npair,9] */
  VNL_F_BODY_IMAT,         /* f [nbody,9] rotation of body_iquat */
  VNL_F_M_ROW,             /* i [nM] row (dof) of each sparse entry */
  VNL_F_BODY_LASTDOF,      /* i [nbody] last dof of the body or of its nearest jointed ancestor, -1 if none */
  VNL_F_DESC_ADR,          /* i [nv+1] CSR over strict descendants of each dof */
  VNL_F_DESC_ENTRY,        /* i [nM-nv] sparse-entry index e with M_COL[e] == dof, M_ROW[e] = the descendant */
  VNL_F_DOFLEVEL_START,    /* i [maxdepth+2] CSR of dofs grouped by ancestor count */
  VNL_F_DOFLEVEL_DOF,      /* i [nv] */
  VNL_F_DOF_ACTADR,        /* i [nv+1] CSR over the actuators driving each dof */
  VNL_F_DOF_ACTLIST,       /* i [nu] */
  VNL_F_KTAB,              /* packed u8 / u16 index tables the kernel stages in shared memory, see VnlKtab */
  VNL_F_MODEL_COUNT
};

/* VNL_F_KTAB: words [0 .. VNL_KT_COUNT) hold the BYTE offset of each table from the start of the field, the next
 * VNL_KT_NSCALAR words hold scalars (VnlKtabScalar); every table is 4-byte aligned.  Built by model_blob.py. */
enum VnlKtab {
  VNL_KT_LVL_START = 0, /* u8  [nlevel+1] offsets into LVL_BP */
  VNL_KT_LVL_BP,        /* u16 [nbody-1]  body | parent << 8, bodies sorted by tree level */
  VNL_KT_PARENT,        /* u8  [nbody] */
  VNL_KT_CHILD_ADR,     /* u8  [nbody+1] CSR over children */
  VNL_KT_CHILD_LIST,    /* u8  [nbody-1] children of each body, descending id */
  VNL_KT_BODY_DOFADR,   /* u8  [nbody] */
  VNL_KT_BODY_DOFNUM,   /* u8  [nbody] number of dofs | 0x80 when the body's first joint is a free joint */
  VNL_KT_BODY_TREE,     /* u8  [nbody] index of the body's kinematic tree */
  VNL_KT_BODY_LASTDOF,  /* u8  [nbody] last dof of the body or of its nearest jointed ancestor, 0xFF if none */
  VNL_KT_SUB_END,       /* u8  [nbody] bodies b .. end-1 are b's subtree */
  VNL_KT_ROOTS,         /* u8  [nroot] root body of each tree */
  VNL_KT_MROW,          /* u8  [nM] */
  VNL_KT_MCOL,          /* u8  [nM] */
  VNL_KT_DOF_BODY,      /* u8  [nv] */
  VNL_KT_DPART_ADR,     /* u8  [nv+1] CSR: partial-sum slots of PROG_D that make up each dof's descendant sum */
  VNL_KT_APART_ADR,     /* u8  [nv+1] CSR: partial-sum slots of PROG_A that make up each dof's strict-ancestor sum */
  VNL_KT_MADR,          /* u16 [nv+1] */
  /* Level schedule of the L^T D L factorisation (left-looking) and of the L^-T sweep: rows (dofs) with descendants,
   * grouped by dof HEIGHT (longest chain of descendants below the dof, leaves = 0) -- rows of one height are independent. */
  VNL_KT_EROW,          /* u32 [2 nv] per row, by height, descending dof inside: madr | (row length - 1) << 13 |
                         * lg2ceil(row length) << 19 | dof << 22; then DESC range begin | end << 16.  8-byte aligned. */
  VNL_KT_ELVL,          /* u16 [nheight+2] first EROW row of heights 0.. | lg2ceil(most descendants of a row there) << 8 */
  VNL_KT_DESC_ADR,      /* u16 [nv+1] CSR over the descendant lists */
  VNL_KT_DESC_SRC,      /* u16 [sum of dof depths] entry madr[k] + a of descendant k (a = depth(k) - depth(row)), k descending */
  VNL_KT_DESC_K,        /* u8  [sum of dof depths] the descendant dof k */
  VNL_KT_DDOF,          /* u8  [dofs of depth >= 1] dofs grouped by depth (L^-1 sweep: gather from the ancestors) */
  VNL_KT_DLVL,          /* u16 [maxdepth+1] first DDOF index of depths 1.. | lg2ceil(depth) << 8 */
  VNL_KT_ANC_START,     /* u16 [nM] madr[mcol[e]]: row start of the entry's column dof */
  VNL_KT_KITEM,         /* u16 [sum of dof depths] c | dof << 8, grouped by dof depth, descending c inside a group */
  VNL_KT_KLVL,          /* u16 [maxdepth+2] offsets into KITEM by dof depth */
  /* Lane programs of the sparse mat-vecs with M and with the inverse factor K (same sparsity).  A program is
   * [T / 4][32 * env_warps][4] words (the four consecutive steps of a lane form one 16-byte word; T a multiple of 8),
   * one term per lane per step: bits 0-13 entry * 4, bits 14-23 x index * 4, bits 24-31 the
   * partial-sum slot to flush into after this term (0xFF = keep accumulating).  PROG_A: strict-ancestor terms
   * (row i, entries madr[i]+1 ..), PROG_D: descendant terms (column j); long rows / columns are split into chunks,
   * the chunks' slots are listed by APART_ADR / DPART_ADR.  Lanes are load balanced on the host; lists are padded with a zero term. */
  VNL_KT_PROG_A,        /* u32 [TA*32*env_warps] */
  VNL_KT_PROG_D,        /* u32 [TD*32*env_warps] */
  VNL_KT_COUNT
};
enum VnlKtabScalar { VNL_KS_TA = 0, VNL_KS_TD, VNL_KS_NDSLOT, VNL_KS_NHEIGHT /* largest dof height */, VNL_KT_NSCALAR };

/* scalar header slots of a TASK blob (imitation task: clip + index tables) */
enum VnlTaskHdr {
  VNL_TH_KIND = 4,        /* 0 = rodent (envs/rodent.py), 1 = humanoid (envs/humanoid.py); informative, the switches below decide */
  VNL_TH_CLIP_LEN,        /* frames in the clip tables (T) */
  VNL_TH_REF_LEN,         /* ref_traj_length (5) */
  VNL_TH_SUB_CLIP_LEN,    /* sub_clip_length (10) */
  VNL_TH_NTRACK,          /* tracked bodies (18) */
  VNL_TH_NJIDX,           /* joint_names (33) */
  VNL_TH_NAPP,            /* appendage_names (5) */
  VNL_TH_NEE,             /* end_eff_names (4) */
  VNL_TH_NFRAMES,         /* physics substeps per env step (5) */
  VNL_TH_OBS_SIZE,        /* 232 */
  VNL_TH_TRAJ_SIZE,       /* 795 */
  VNL_TH_COM_REF_IDX,     /* column of the filtered body table used as COM reference (quirk Q4) */
  VNL_TH_TORSO_BODY,      /* body whose xmat defines the egocentric frame (1) */
  /* variant switches: rodent (envs/rodent.py) = all 0 except OBS_QFRC / USE_SUBCLIP; humanoid (envs/humanoid.py) see below */
  VNL_TH_REWARD_OLD_STATE,/* 1: every reward term reads the PRE-step state (humanoid.py:275, `data_c = state.pipeline_state`) */
  VNL_TH_TERM_MEAN,       /* 1: termination error = mean |.| over joints and over all body coordinates (humanoid.py:256-258);
                             0: L1 sum over joints + max column abs-sum over tracked bodies (rodent.py:256-258) */
  VNL_TH_USE_SUBCLIP,     /* 1: done when sub_clip_frame reaches sub_clip_length (rodent.py:207-215) */
  VNL_TH_OBS_QFRC,        /* 1: obs carries qfrc_actuator and the end-effector positions (rodent.py:337-344) */
  VNL_TH_COM_FROM_FIELD,  /* 1: COM reference = VNL_T_CENTER_OF_MASS (humanoid.py:279); 0: filtered body table column (quirk Q4) */
  VNL_TH_ROT_BODY,        /* body whose xmat rotates into the egocentric frame: 1 = torso (rodent.py:385), 0 = world for the ant
                           * (ant.py:333 reads data.xmat[0], i.e. the identity) */
  VNL_TH_TRAJ_OLD_FRAME,  /* 1: the step's reference window starts at OLD cur_frame + 1 (ant.py:182 hands state.info to _get_obs
                           * before the increment); 0: at NEW cur_frame + 1 (rodent.py:188-190) */
  VNL_TH_RACT_ACTION,     /* 1: ract = 0.01 * -0.015 * sum(action^2) / nu (ant.py:251); 0: -0.015 * mean(qfrc_actuator^2) */
  VNL_TH_METRICS_RAW,     /* 1: metrics hold the UNWEIGHTED reward terms (ant.py:203-210); 0: the weighted ones (rodent.py:193-199) */
  VNL_TH_NCLIPS,          /* clips stacked in the tables (SURVEY 8 row f4): every VNL_T_* clip table is [nclips, T, ...], the env's
                           * VnlState.clip_id picks one; 0 or 1 = the single-clip task of the reference */
  VNL_TH_HEALTHY_LO = 32, VNL_TH_HEALTHY_HI, VNL_TH_TERM_THRESHOLD, VNL_TH_BODY_ERR_MULT,
  VNL_TH_W_RCOM, VNL_TH_W_RVEL, VNL_TH_W_RTRUNK, VNL_TH_W_RQUAT, VNL_TH_W_RACT, VNL_TH_W_RAPP, /* reward weights:
                           * rodent / humanoid 0.01 x4, 1e-4, 0.01 (rodent.py:193-199); ant 0.05 0.01 0.20 0.01 0.001 0 (ant.py:186-192) */
  VNL_TH_DONE_RTRUNK      /* done when the UNSCALED rtrunk is below this (0 for the rodent, 0.5 for the humanoid: humanoid.py:199) */
};

enum VnlTaskField {
  VNL_T_POSITION = 0,     /* f [T,3]      ReferenceClip.position */
  VNL_T_QUATERNION,       /* f [T,4] */
  VNL_T_JOINTS,           /* f [T,nq-7] */
  VNL_T_BODY_POSITIONS,   /* f [T,ntrack,3] already filtered to walker_body_names (rodent.py:114) */
  VNL_T_VELOCITY,         /* f [T,3] */
  VNL_T_ANGULAR_VELOCITY, /* f [T,3] */
  VNL_T_JOINTS_VELOCITY,  /* f [T,nv-6] */
  VNL_T_BODY_IDXS,        /* i [ntrack]  model body ids (rodent.py:81-86) */
  VNL_T_EE_IDX,           /* i [nee]     model body ids (rodent.py:65-70) */
  VNL_T_APP_IDX,          /* i [napp]    model body ids (rodent.py:71-76) */
  VNL_T_APP_REF_IDX,      /* i [napp]    app ids clamped into the filtered table (quirk Q5) */
  VNL_T_JOINT_COL,        /* i [njidx]   joint ids clamped into the nq-7 joint columns (quirk Q6) */
  VNL_T_CENTER_OF_MASS,   /* f [T,3]     ReferenceClip.center_of_mass (old 13-field clip format, humanoid.py:279); zeros if absent */
  VNL_TASK_COUNT
};

/* ------------------------------------------------------------------------------------------
 * Per-env state crossing the boundary.  Mirrors the leaves of the brax `State` the
 * reference's callers read (SURVEY section 8b): pipeline_state.{qpos,qvel,act,
 * qacc_warmstart,xpos,xquat,subtree_com[1],qfrc_actuator} and info.{cur_frame,sub_clip_frame}.
 * xpos/xquat/subtree_com/qfrc_actuator lag qpos by one physics substep exactly as
 * mjx.step leaves them (forward, then euler).
 * ---------------------------------------------------------------------------------------- */
typedef struct VnlState {
  float* qpos;           /* [B,nq] */
  float* qvel;           /* [B,nv] */
  float* act;            /* [B,na] */
  float* qacc_warmstart; /* [B,nv] */
  float* xpos;           /* [B,nbody,3] */
  float* xquat;          /* [B,nbody,4] */
  float* subtree_com;    /* [B,3]  subtree_com[torso] */
  float* qfrc_actuator;  /* [B,nv] */
  int32_t* cur_frame;      /* [B] info["cur_frame"] */
  int32_t* sub_clip_frame; /* [B] info["sub_clip_frame"] */
  int32_t* clip_id;        /* [B] which clip of a multi-clip task blob the env tracks (SURVEY 8 row f4); NULL = clip 0.
                              Read from `in`, copied to `out` when both are given; never changed by a step. */
} VnlState;

/* Host-side call context: everything the host needs to size a launch, so that no call depends on a registry keyed by
 * device pointers.  Fill it once with vnl_context_init and set the workspace; pass it to every call (read-only). */
typedef struct VnlContext {
  uint32_t model_hdr[VNL_DATA_OFF]; /* host copy of the first VNL_DATA_OFF words of the MODEL blob (scalars + field table) */
  uint32_t task_hdr[VNL_TABLE_OFF]; /* host copy of the scalar header of the TASK blob; task_hdr[0] == 0: physics only */
  void* workspace;                  /* device scratch of vnl_workspace_bytes() bytes (inertia of the resident envs); the
                                       kernels write before they read, so it may be uninitialised (an XLA scratch result) */
  uint64_t workspace_bytes;
} VnlContext;

/* Validates the two host blobs (vnl_check_model / vnl_check_task) and copies their headers; `task_host` may be NULL.
 * Leaves workspace = NULL.  0 = ok. */
int vnl_context_init(VnlContext* ctx, const void* model_host, size_t model_bytes, const void* task_host, size_t task_bytes);

typedef struct VnlOutputs {
  float* obs;     /* [B,obs_size]  State.obs (rodent.py:318-344), NaN -> 0 */
  float* traj;    /* [B,traj_size] info["traj"] (rodent.py:346-382) */
  float* reward;  /* [B] */
  float* done;    /* [B] 0/1 */
  float* metrics; /* [B,7] rcom rvel rtrunk rquat ract rapp termination_error (scaled, rodent.py:227-235) */
  int32_t* stats; /* [B,4] solver iterations, line-search iterations, active contacts, active limits
                     (summed over the substeps of the call); may be NULL */
} VnlOutputs;

/* One env step for B envs: `in` is read, `out` and `outputs` are written (in and out may alias
 * buffer by buffer).  Replaces RodentTracking.step (envs/rodent.py:178-239). */
int vnl_step(const VnlContext* ctx, const void* model, const void* task, int B, const VnlState* in, const float* action,
             const VnlState* out, const VnlOutputs* outputs, void* stream);

/* vnl_step followed by brax's AutoResetWrapper.step (brax/envs/wrappers/training.py, installed around the env at
 * ppo_imitation/train.py:204-214), in the same launch: where the step's done flag is set, the state leaves written to
 * `out` (qpos .. qfrc_actuator) and `outputs->obs` are replaced by `first` / `first_obs` (the cached reset state);
 * info (cur_frame, sub_clip_frame, traj), reward, done and metrics are NOT restored (SURVEY quirk Q7). */
int vnl_step_autoreset(const VnlContext* ctx, const void* model, const void* task, int B, const VnlState* in, const float* action,
                       const VnlState* out, const VnlOutputs* outputs, const VnlState* first, const float* first_obs,
                       void* stream);

/* Episode bookkeeping of brax's EpisodeWrapper + AutoResetWrapper (`envs.training.wrap`, reached from
 * ppo_imitation/train.py:204-214 with action_repeat = 1, train.py:121): info["steps"] and info["truncation"]. */
typedef struct VnlEpisode {
  const float* steps_in;  /* [B] info["steps"] of the incoming state */
  const float* done_in;   /* [B] done of the incoming state: AutoResetWrapper zeroes the counter of a finished episode */
  float* steps_out;       /* [B] (may alias steps_in) */
  float* truncation_out;  /* [B] info["truncation"] = 1 - done where the episode length is reached, else 0 */
  float episode_length;   /* train_config.yaml:7 (150) */
} VnlEpisode;

/* vnl_step wrapped the way the reference trains (ppo_imitation/train.py:204-214): AutoResetWrapper(EpisodeWrapper(env)),
 * action_repeat 1, all in the one launch.  steps = (done_in ? 0 : steps_in) + 1; where steps >= episode_length:
 * truncation = 1 - done, done = 1; then the AutoReset restore of vnl_step_autoreset on that final done flag. */
int vnl_step_training(const VnlContext* ctx, const void* model, const void* task, int B, const VnlState* in, const float* action,
                      const VnlState* out, const VnlOutputs* outputs, const VnlState* first, const float* first_obs,
                      const VnlEpisode* episode, void* stream);

/* Resampling AutoReset (DESIGN §3h): where an episode ends, the env starts a new one from a fresh draw instead of the cached
 * first state.  The draw: Philox4x32-10 with key (seed low 32 bits, seed high 32 bits) and counter (g, n, j, 0), g =
 * env_offset + e the global env index, n = reset_count[e], j the block.  Block 0: clip = (x0 * nclips) >> 32, start =
 * (x1 * start_frame_hi) >> 32 (64-bit products).  Blocks j >= 1, only when noise_scale != 0: u = ((x >> 8) + 1) 2^-24,
 * Box-Muller on (u0, u1) and (u2, u3) -> (r cos t, r sin t), r = sqrt(-2 ln u_a), t = 2 pi u_b: the normals of qpos
 * coordinates 4 (j - 1) .. 4 (j - 1) + 3. */
typedef struct VnlResample {
  uint64_t seed;          /* Philox key */
  int32_t env_offset;     /* global index of env 0 of this call (a shard's first env): a sharded run draws what one process would */
  int32_t start_frame_hi; /* start frame uniform in [0, start_frame_hi); 0 < start_frame_hi <= clip length - ref_traj_length, so
                             that the reset's reference window lies inside the clip */
  float noise_scale;      /* qpos += noise_scale * N(0, 1) on every coordinate (finite, >= 0; 0 = no noise) */
  int32_t* reset_count;   /* [B] resets of each env so far (the draw's counter n); incremented on every env reset */
  int32_t* scratch;       /* [B + 1] caller-owned device scratch: the count of done envs, then their indices */
} VnlResample;

/* vnl_step_training without the first-state restore, then, where the final done flag is set, the env reset in place to a fresh
 * draw (clip, start frame, qpos noise): what vnl_reset of the drawn qpos / qvel / start frame / clip would write goes to the
 * state leaves of `out`, cur_frame = start, sub_clip_frame = 0, clip_id = clip (where `out` has one), and to the obs / traj rows
 * of `outputs`.  The step's reward, done, metrics, stats, steps and truncation are kept.  Three launches (step, compaction of
 * the done envs into rs->scratch, reset of the listed envs): enqueue-only, no allocation, capturable. */
int vnl_step_training_resample(const VnlContext* ctx, const void* model, const void* task, int B, const VnlState* in,
                               const float* action, const VnlState* out, const VnlOutputs* outputs, const VnlEpisode* episode,
                               const VnlResample* rs, void* stream);

/* Reset tail for B envs: qpos/qvel/cur_frame(start_frame) are read from `in` (act, ctrl and
 * qacc_warmstart are zero as in mjx.make_data), `out` receives the mjx.forward state, obs,
 * traj and info["termination_error"] (metrics[6]).  Replaces envs/rodent.py:148-176. */
int vnl_reset(const VnlContext* ctx, const void* model, const void* task, int B, const VnlState* in, const VnlState* out,
              const VnlOutputs* outputs, void* stream);

/* Physics only: `nsteps` x mjx.step (forward; euler) with a constant ctrl, no task logic.
 * Replaces PipelineEnv.pipeline_step (envs/rodent.py:181). */
int vnl_pipeline_step(const VnlContext* ctx, const void* model, int B, int nsteps, const VnlState* in, const float* ctrl,
                      const VnlState* out, int32_t* stats, void* stream);

/* Stage dump of one mjx.forward for parity tests: writes the arrays listed in
 * VNL_DUMP_* order into `dump` ([B, vnl_dump_size(model)] floats).  Test hook. */
int vnl_forward_dump(const VnlContext* ctx, const void* model, int B, const VnlState* in, const float* ctrl, float* dump,
                     void* stream);
size_t vnl_dump_size(const void* model_host);

/* Clip preprocessing on the GPU (SURVEY 8 row f4).  Replaces `process_clip` after the pickle load
 * (preprocessing/mjx_preprocess.py:88-105): `extract_features` (set_position -> smooth.kinematics per frame, :109-134) and
 * `compute_velocity_from_kinematics` + the joint-velocity clip (:170-193, :96-99), for `nclips` clips of T frames at once.
 *   qpos             [nclips, T, nq]  raw mocap qpos (free joint first)
 *   qpos_out         [nclips, T, nq]  qpos after kinematics (free-joint quaternion normalised): position | quaternion | joints
 *   body_positions   [nclips, T, nbody, 3], body_quaternions [nclips, T, nbody, 4]   xpos / xquat of every body
 *   qvel_out         [nclips, T, nq-1] velocity | angular_velocity | joints_velocity (joint block clipped to +-max_qvel);
 *                    each clip is padded with its own last frame, as the reference does (last row = 0)
 * The task blob stacks these per clip (VNL_TH_NCLIPS); needs no task blob itself. */
int vnl_process_clip(const VnlContext* ctx, const void* model, int nclips, int T, const float* qpos, float dt, float max_qvel,
                     float* qpos_out, float* body_positions, float* body_quaternions, float* qvel_out, void* stream);

/* Blob validation on the host (magic, version, sizes).  0 = ok. */
int vnl_check_model(const void* model_host, size_t nbytes);
int vnl_check_task(const void* task_host, size_t nbytes);

/* Dynamic shared memory of one CTA for this model, and the number of envs (one warp each) a CTA holds. */
int vnl_step_smem_bytes(const void* model_host);
int vnl_envs_per_cta(const void* model_host);
/* Envs the persistent grid holds at once on the current device (CTAs x envs per CTA): a batch that is a multiple of
 * this runs in whole rounds; host layers cut a step into chunks of this size to overlap result copies with compute. */
int vnl_resident_envs(const void* model_host);

/* Device workspace of the step kernels: the joint-space inertia of every RESIDENT env lives in global memory (L2),
 * laid out in the order the mat-vec lane programs consume it, which is what lets fourteen rodent envs share an SM.
 * The caller allocates vnl_workspace_bytes() bytes on the device (the bound over every launch geometry the library can
 * pick on the current device) and passes them in VnlContext; one workspace serves one stream at a time.  A model that
 * streams its inertia fails with -20 without a workspace and with -21 if the ACTUAL launch geometry of the call (grid x
 * envs per CTA for this B) would index past workspace_bytes. */
size_t vnl_workspace_bytes(const void* model_host);

/* Test hook: (name, float offset, float size) of every array of the per-env shared-memory layout for this model, in the
 * order of make_layout (csrc/vnl_kernels.cu); the last entry "total" carries the slice size as its offset.  Returns the
 * number of entries.  tests/test_layout.py checks that arrays that are live in the same phase never share storage. */
int vnl_debug_layout(const void* model_host, const char** names, int32_t* offsets, int32_t* sizes, int cap);

/* XLA custom-call entry points, STATUS-RETURNING legacy signature (API_VERSION_STATUS_RETURNING = 2):
 *     void f(cudaStream_t stream, void** buffers, const char* opaque, size_t opaque_len, XlaCustomCallStatus* status)
 * Stateless: everything the host needs travels in `opaque` (VnlXlaOpaque: B, the blobs' headers), the workspace is the
 * LAST buffer (declare it as a scratch result of vnl_workspace_bytes() bytes), model and task blobs are ordinary operands
 * at whatever address XLA placed them.  A non-zero return code of the underlying call is reported through
 * XlaCustomCallStatusSetFailure (resolved with dlsym from the hosting process, i.e. jaxlib) -- never silently dropped.
 *   buffers: [model, task, qpos, qvel, act, warm, xpos, xquat, subtree_com, qfrc_actuator, cur_frame, sub_clip_frame, clip_id,
 *             action,
 *             (results) qpos', qvel', act', warm', xpos', xquat', subtree_com', qfrc_actuator', cur_frame', sub_clip_frame',
 *             clip_id', obs, traj, reward, done, metrics, stats, workspace]
 * vnl_xla_reset takes the same list (action is ignored).  The `_rc` forms return the code instead (tests, other hosts). */
typedef struct VnlXlaOpaque {
  int32_t B;        /* envs: product of all leading (vmap) dimensions */
  int32_t version;  /* VNL_XLA_OPAQUE_VERSION */
  uint32_t model_hdr[VNL_DATA_OFF];
  uint32_t task_hdr[VNL_TABLE_OFF];
  uint64_t workspace_bytes;
} VnlXlaOpaque;
#define VNL_XLA_OPAQUE_VERSION 2
#define VNL_XLA_STEP_NBUF 32
void vnl_xla_step(void* stream, void** buffers, const char* opaque, size_t opaque_len, void* status);
void vnl_xla_reset(void* stream, void** buffers, const char* opaque, size_t opaque_len, void* status);
int vnl_xla_step_rc(void* stream, void** buffers, const char* opaque, size_t opaque_len);
int vnl_xla_reset_rc(void* stream, void** buffers, const char* opaque, size_t opaque_len);
/* Fills `opaque` for B envs from a context (host helper for bindings). */
int vnl_xla_make_opaque(const VnlContext* ctx, int B, VnlXlaOpaque* opaque);

/* Measurement helper (bench.py): FFMA-saturating microkernel, flops = blocks * 256 * iters * 32.  `out` needs
 * blocks * 256 floats (never written in practice).  Gives the FP32 roofline denominator of the device. */
int vnl_ffma_probe(int blocks, int iters, float* out, void* stream);

/* vnl_step with one env's per-phase clock64 accumulators written to prof[32] (developer hook, tools/gpu_prof.py). */
int vnl_step_profiled(const VnlContext* ctx, const void* model, const void* task, int B, const VnlState* in, const float* action,
                      const VnlState* out, const VnlOutputs* outputs, void* stream, long long* prof, int block);

const char* vnl_version(void);

#ifdef __cplusplus
}
#endif
#endif /* VNL_B200_H_ */
