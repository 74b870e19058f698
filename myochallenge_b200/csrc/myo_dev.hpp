// Device-side model tables and per-world scratch layout shared by the host packer and the kernels.
#pragma once
#include <cstdint>

#include "../../include/myo_b200.h"

namespace myo {

constexpr int KC = 8;    // max dofs on a body's ancestor chain (myoHand distal phalanx: 3 wrist + 4 finger)
constexpr int KT = 8;    // max dofs a tendon's moment arm touches
constexpr int KS = 16;   // max support of one contact block (chain A xor chain B)
constexpr int LIM_WORDS = 8;    // scratch words per limit record
constexpr int CON_WORDS = 24;   // scratch words per contact record
constexpr int SEG_WORDS = 8;    // table words per tendon segment record
constexpr int SEG_OUT = 9;      // scratch words per tendon segment result: length, KT moment-arm slots
constexpr int ROW_WORDS = 4;    // scratch words per constraint row (one float4)
constexpr int kFastRows = 96;           // constraint rows of the fast layout: 32 limit rows + 4 x 16 contacts
constexpr int kSoloRowsPerLane = 10;    // rows per lane the full-capacity (one world per CTA) kernel keeps in registers

enum { J_FREE = 0, J_BALL = 1, J_SLIDE = 2, J_HINGE = 3 };
enum { G_PLANE = 0, G_SPHERE = 2, G_CAPSULE = 3, G_ELLIPSOID = 4, G_CYLINDER = 5, G_BOX = 6 };
enum { W_PULLEY = 2, W_SITE = 3, W_SPHERE = 4, W_CYLINDER = 5 };
enum { ST_UNSUPPORTED = 1, ST_CON_OVERFLOW = 2, ST_EFC_OVERFLOW = 4, ST_NONFINITE = 8 };
enum { EFC_LIMIT_JOINT = 3, EFC_LIMIT_TENDON = 4, EFC_CONTACT_FRICTIONLESS = 5, EFC_CONTACT_PYRAMIDAL = 6 };

// limit record layout (floats/ints in scratch)
// the support and Jacobian of a limit row are referenced, not copied: the dof indices are a slice of the model's int
// tables (j_dofadr / t_dof, word offset L_IOFF), the values a slice of the world's scratch (word offset L_JOFF: the
// constant 1 kept in o_misc for a joint, the tendon's ten_J row for a tendon) times L_SIGN
enum { L_KIND = 0, L_ID = 1, L_NSUP = 2, L_POS = 3, L_MARGIN = 4, L_SIGN = 5, L_IOFF = 6, L_JOFF = 7 };
// contact record layout
// The contact Jacobian is not stored: its support is the dofs of chain(body A) and chain(body B) past their common
// prefix (C_CP = prefix length | count on the A side << 8; C_NSUP entries in all, A side first) and an entry is
// recomputed from cdof, the contact point and the frame wherever it is needed (contact_entry in myo_phys.cuh).
enum { C_G1 = 0, C_G2 = 1, C_DIM = 2, C_NSUP = 3, C_DIST = 4, C_MARGIN = 5, C_MU = 6, C_ROW0 = 7, C_POS = 8 /*3*/,
       C_FRAME = 11 /*9*/, C_BA = 20, C_BB = 21, C_CP = 22 };
// row record
enum { R_D = 0, R_AREF = 1, R_JAR = 2, R_JP = 3 };

// Model tables live in shared memory: every kernel stages the packed table block (ints, then floats)
// at the start of its dynamic shared memory, and a table is just a word offset into that block.
#if defined(__CUDACC__) || defined(MYO_EMUL)
#ifdef MYO_EMUL
#define MYO_SMEM_WORDS (reinterpret_cast<float*>(emul_smem))
#else
extern __shared__ float4 myo_smem4[];
#define MYO_SMEM_WORDS (reinterpret_cast<float*>(myo_smem4))
#endif
#define MYO_TAB_DI __device__ __forceinline__
struct TabI {
  int off;
  MYO_TAB_DI const int* ptr() const { return reinterpret_cast<const int*>(MYO_SMEM_WORDS) + off; }
  MYO_TAB_DI int operator[](int i) const { return ptr()[i]; }
  MYO_TAB_DI const int* operator+(int i) const { return ptr() + i; }
};
struct TabF {
  int off;
  MYO_TAB_DI const float* ptr() const { return MYO_SMEM_WORDS + off; }
  MYO_TAB_DI float operator[](int i) const { return ptr()[i]; }
  MYO_TAB_DI const float* operator+(int i) const { return ptr() + i; }
};
#else
struct TabI { int off; };
struct TabF { int off; };
#endif

struct DevModel {
  // sizes
  int nq, nv, nu, na, nbody, njnt, ngeom, nsite, ntendon, nwrap, nM, npair, nlevel, ndlevel;
  int nq4, nv4, na4, nu4, nparam, nparam4, nobs, nobs4;
  // observation: task_obs writes the kind's canonical layout (nobs_scr words at o_obs), the caller's buffers take nobs words.
  // With obs_keys the output is gathered from nobs_run runs: obs_run[r] = source word | width << 16 | OBS_RUN_* << 28
  // (nobs_run 0: the canonical layout as it is, nobs == nobs_scr)
  int nobs_scr, nobs_run, obs_run[MYO_MAX_OBS_KEYS];
  int nlim_max, ncon_max, nefc_max;
  int nd;   // dofs [0, nd) couple through the mass matrix; dofs [nd, nv) are simple (diagonal)
  TabI pair_ab;  // unordered support pairs of a contact block (myo_pack.cpp)
  TabI h_roff;   // word offset of row i of the packed lower-triangular Newton Hessian (rows 0..pad4(nv); the last is the rhs)
  int solver_iter;
  float solver_tol, timestep, gravity[3], inv_sqrt_impratio, meaninertia;
  int any_damping, any_tendon_passive, any_joint_spring, any_tendon_limit;
  // body tables
  TabI b_parent, b_root, b_jntadr, b_jntnum, b_dofadr, b_dofnum, b_nchain, b_chain, b_mass_slot, b_pose_slot,
      b_sameframe, lvl_adr, lvl_body, b_subadr, b_sub;
  TabF b_pos, b_mat, b_ipos, b_imat, b_mass, b_inertia, b_invweight0;
  // joints
  TabI j_type, j_qposadr, j_dofadr, j_body, j_limited;
  TabF j_pos, j_axis, j_qpos0, j_range, j_margin, j_solref, j_solimp, j_stiffness, j_qpos_spring;
  // dofs
  TabI d_body, d_parent, d_simple, d_Madr, d_depth, d_jnt, d_prefadr, d_pref, m_rowadr, m_row,
      d_actadr, d_actlist;
  TabF d_armature, d_damping, d_invweight0, d_M0;
  // geoms
  TabI g_type, g_body, g_condim, g_priority, g_size_slot, g_fri_slot;
  TabF g_pos, g_mat, g_size, g_rbound, g_friction, g_solmix, g_solref, g_solimp, g_margin, g_gap;
  // collision pair list (static filters applied on host), geom1.type <= geom2.type
  TabI p_g1, p_g2, p_supported;
  // sites
  TabI s_body, s_pos_slot;
  TabF s_pos;
  // tendons + wraps
  TabI t_limited, t_ndof, t_dof;
  TabI seg_rec, seg_list, t_segadr, t_seg;   // tendon path segments (myo_pack.cpp)
  TabF seg_invdiv;
  int nseg;
  TabF t_range, t_margin, t_solref, t_solimp, t_invweight0, t_stiffness, t_damping, t_lengthspring;
  // actuators
  TabI a_tendon, a_dyntype, a_gaintype, a_biastype, a_ctrllimited, a_forcelimited;
  TabF a_dynprm, a_gainprm, a_biasprm, a_ctrlrange, a_forcerange, a_gear, a_acc0, a_lengthrange;
  // scratch offsets (words) inside one world's shared-memory block
  int o_qpos, o_qvel, o_act, o_ctrl, o_warm, o_xpos, o_xmat, o_xipos, o_cdof, o_cinert, o_cdofdot,
      o_cfrc, o_M, o_tenL, o_tenV, o_tenJ, o_actF, o_bias, o_passive, o_qact, o_smooth, o_qaccs,
      o_qacc, o_qcon, o_actdot, o_grad, o_p, o_Mp, o_Ma, o_H, o_lim, o_con, o_row, o_misc, o_obs, o_wparam,
      o_seg,   // the tendon phase's per-segment results (nseg x SEG_OUT words)
      scratch_words;
  const float* g_tables;     // global copy of the table block
  int tab_words;             // its size in words (multiple of 4); world scratch starts right after it
  TabF init_qpos;   // [nq] state written by reset (MyoSuite init_qpos)
  TabF param0;      // [nparam4] nominal values of the per-world override parameters
  float frame_dt;           // frame_skip * timestep (MyoSuite env.dt)
};

// Model descriptors live in constant memory, one slot per live batch: the (noinline) phases receive the slot index and
// read sizes / table offsets with LDC instead of generic loads through a by-reference kernel parameter
// (round-1 profile: 622 M generic loads in table lookups per 8192-world step).
constexpr int kModelSlots = 16;
#if defined(MYO_EMUL)
static DevModel c_models[kModelSlots];
#define MYO_M const DevModel& m = c_models[mslot];
#elif defined(__CUDACC__)
__constant__ DevModel c_models[kModelSlots];
#define MYO_M const DevModel& m = c_models[mslot];
#endif

// per-batch device pointers
struct BatchPtrs {
  int n_worlds;   // worlds the caller sees
  int n_alloc;    // worlds allocated and stepped (n_worlds rounded up to a multiple of worlds per CTA)
  float *qpos, *qvel, *act, *warm, *time, *wparam, *task_f, *pose_target;
  int *task_i, *status;
  float* dump;   // [n][scratch_words] written by forward / mj_step mode (may be null)
  unsigned long long seed;
  const int* order;   // optional [n_alloc]: slot -> world, worlds grouped by their recent constraint count (null: identity)
  // worlds the fast kernel hands to the full-capacity kernel of the same env step (see myo_kernels.cu): world index | kind << 30
  int* redo_list;     // [n_alloc], -1 = not written yet
  int* redo_count;    // [1]
  // dynamic scheduling of the env step (fast kernel): [0] next group of worlds, [1] groups finished, [2] redo entries taken.
  // CTAs fetch groups until none is left, then serve the redo list with the full-capacity layout, heavy_per_cta worlds at a
  // time in the CTA's own shared memory - the redone worlds ride in the slack of the last wave instead of a pass of their own
  int* sched;
  int heavy_per_cta;
  int* work;          // [n_alloc]: constraint rows of the world's last substep (the grouping key for the next step)
};

enum { TI_ELAPSED = 0, TI_EPISODE = 1, TI_TASK = 2, TI_FLAGS = 3, TI_WORDS = 4 };
enum { TF_ANGLE1 = 0, TF_ANGLE2 = 1, TF_XR = 2, TF_YR = 3, TF_PERIOD = 4, TF_POSDIST = 5, TF_ROTDIST = 6, TF_WORDS = 8 };
// o_misc scratch words
enum { MI_NLIM = 0, MI_NCON = 1, MI_NEFC = 2, MI_ITER = 3, MI_STATUS = 4, MI_ONE = 5 /*float 1*/, MI_WORDS = 8 };

enum { OBS_RUN_COPY = 0, OBS_RUN_TIME = 1 /* the world's time, width 1 */, OBS_RUN_SUM = 2 /* src[i] + src[width + i] */ };

enum StepMode { MODE_ENV_STEP = 0, MODE_MJ_STEP = 1, MODE_FORWARD = 2, MODE_GET_OBS = 3, MODE_RESET = 4, MODE_REDO = 5 };
enum { REDO_STEP = 0, REDO_RESET = 1 };      // kinds of redo-list entries

struct StepArgs {
  int mode, nsub;
  const float* in;        // actions or ctrl [n][nu]
  float* obs;             // [n][nobs]
  float* reward;          // [n]
  uint8_t* done;          // [n]
  uint8_t* truncated;     // [n]
  float* terminal_obs;    // [n][nobs]
  float* info;            // [n][MYO_INFO_TERMS]
  const uint8_t* mask;    // reset mask
};

}  // namespace myo
