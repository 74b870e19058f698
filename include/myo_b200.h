/* myo_b200.h -- C ABI of the B200-native batched myo-simulator (libmyo_b200.so).
 *
 * The reference (amathislab/myochallenge) has no FFI of its own: its hot path crosses two Python
 * seams (SURVEY.md 8b).  Every entry point below names the reference interface it replaces:
 *
 *   myo_model_*      <- mujoco_py.load_model_from_mjb / sim.model.* views that MyoSuite's
 *                       BaseV0.__init__ builds from the `model_path` kwarg
 *                       (/root/reference/src/envs/__init__.py:17,29,44,62) and that
 *                       /root/reference/src/envs/baoding.py:372-389,560-604 read and write.
 *   myo_batch_create <- make_parallel_envs + SubprocVecEnv([...16 thunks])
 *                       (/root/reference/src/main_baoding.py:56-65,74) and the env kwargs of
 *                       /root/reference/src/envs/__init__.py:58-74 (Baoding P2), :137-150 (finger).
 *   myo_batch_reset  <- CustomBaodingP2Env.reset (/root/reference/src/envs/baoding.py:494-647),
 *                       CustomPoseEnv.reset (/root/reference/src/envs/pose.py:53-99),
 *                       MyoSuite 1.2.3 ReachEnvV0.reset, restated from memory ([3P-MEM], SURVEY.md), behind the
 *                       factory names MyoFingerReachFixed / MyoFingerReachRandom
 *                       (/root/reference/src/envs/environment_factory.py:22-61).
 *   myo_batch_step   <- VecEnv.step_async/step_wait -> env.step: BaodingEnvV1.step target update,
 *                       BaseV0.step action remap, Robot.step (frame_skip x mj_step), get_obs,
 *                       get_reward_dict (/root/reference/src/envs/baoding.py:403-467; reach: ReachEnvV0
 *                       get_obs_dict / get_reward_dict [3P-MEM]), TimeLimit and
 *                       the SubprocVecEnv worker's auto-reset.
 *   myo_batch_mj_step / myo_batch_forward <- MjSim.step() / MjSim.forward()
 *                       (/root/reference/src/envs/baoding.py:183,206,625,632 reach them).
 *   myo_batch_set_state / get_state <- MujocoEnv.set_state / sim.data.qpos,qvel,act
 *                       (/root/reference/src/envs/baoding.py:206,632,645).
 *   myo_batch_set_param / get_param <- in-place writes to sim.model.body_mass / geom_friction /
 *                       geom_size / site_pos (/root/reference/src/envs/baoding.py:560-604).
 *   myo_policy_*     <- sb3_contrib RecurrentActorCriticPolicy.forward as constructed by
 *                       /root/reference/src/train/trainer.py:49-64.
 *   myo_running_moments_* / myo_vecnorm_reward <- stable_baselines3 VecNormalize (RunningMeanStd.update,
 *                       step_wait's return/reward handling) wrapped around the envs at
 *                       /root/reference/src/main_baoding.py:75.
 *   myo_gae          <- RecurrentRolloutBuffer.compute_returns_and_advantage, called by RecurrentPPO.learn
 *                       (/root/reference/src/train/trainer.py:67-71).
 *   myo_ppo_*        <- RecurrentPPO.train (sb3-contrib), the policy update half of agent.learn()
 *                       (/root/reference/src/train/trainer.py:67-71; hyper-parameters
 *                       /root/reference/docs/summary.md:86-117): evaluate_actions over sequences, PPO loss,
 *                       backward, clip_grad_norm_, Adam.
 *
 * Conventions: every function returns 0 on success or a negative myo_status; the message for the
 * calling thread's last failure is myo_last_error().  Nothing throws across the boundary.  Handles
 * are opaque and owned by the library.  Pointers named *_dev are CUDA device pointers owned by the
 * caller (e.g. torch tensors); `stream` is a cudaStream_t passed as void* (NULL = default stream).
 * Calls on one handle are not thread-safe; different handles are independent (one per GPU).
 * There is no CPU fallback: without a CUDA device every batch/policy call fails with MYO_E_CUDA.
 */
#ifndef MYO_B200_H
#define MYO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct myo_model myo_model;
typedef struct myo_batch myo_batch;
typedef struct myo_policy myo_policy;
typedef struct myo_ppo myo_ppo;

typedef enum {
  MYO_OK = 0,
  MYO_E_ARG = -1,      /* bad argument */
  MYO_E_IO = -2,       /* file could not be read */
  MYO_E_FORMAT = -3,   /* not a MuJoCo 2.1.0 MJB */
  MYO_E_UNSUPPORTED = -4, /* model uses a feature outside the supported subset */
  MYO_E_CUDA = -5,     /* CUDA runtime error / no device */
  MYO_E_LIMIT = -6     /* model exceeds a compiled-in capacity */
} myo_status;

typedef enum { MYO_TASK_NONE = 0, MYO_TASK_POSE = 1, MYO_TASK_BAODING = 2, MYO_TASK_REORIENT = 3, MYO_TASK_REACH = 4 } myo_task_kind;

/* Baoding `Task` enum values (MyoSuite baoding_v1.Task; 0 = hold, see
 * /root/reference/src/envs/baoding.py:287-294, /root/reference/src/models/classifier.py:116) */
enum { MYO_BAODING_HOLD = 0, MYO_BAODING_CW = 1, MYO_BAODING_CCW = 2 };

/* per-world overridable model parameters (the arrays the reference's reset() writes in place) */
typedef enum {
  MYO_PARAM_BODY_MASS = 0,     /* 1 float  */
  MYO_PARAM_GEOM_SIZE = 1,     /* 3 floats */
  MYO_PARAM_GEOM_FRICTION = 2, /* 3 floats */
  MYO_PARAM_SITE_POS = 3,      /* 3 floats */
  MYO_PARAM_BODY_POS = 4,      /* 3 floats: body_pos (frame in the parent) */
  MYO_PARAM_BODY_MAT = 5       /* 9 floats: rotation matrix of body_quat, row major */
} myo_param_kind;

#define MYO_MAX_OVERRIDE 4
#define MYO_INFO_TERMS 12
#define MYO_MAX_ROT_RANGES 4

/* Task / env configuration: the kwargs of the gym registrations plus the curriculum knobs of
 * CustomBaodingP2Env._setup (/root/reference/src/envs/baoding.py:300-401) and
 * CustomPoseEnv._setup (/root/reference/src/envs/pose.py:7-51). */
typedef struct myo_task_cfg {
  int32_t kind;                 /* myo_task_kind */
  int32_t frame_skip;           /* mj_steps per env step (10; die/pen 5) */
  int32_t max_episode_steps;    /* gym TimeLimit horizon; <=0 disables truncation */
  int32_t normalize_act;        /* BaseV0: ctrl = 1/(1+exp(-5(a-0.5))) for muscle actuators */
  int32_t auto_reset;           /* SubprocVecEnv worker semantics: reset inside step on done */
  int32_t solver_iterations;    /* Newton iteration cap per mj_step (<=0: model's opt.iterations) */
  float solver_tolerance;       /* <=0: model's opt.tolerance */
  /* reward weights, in the order written to info[] (slot 7 always carries the dense reward):
   *  baoding : pos_dist_1 pos_dist_2 act_reg alive sparse solved done dense
   *  pose    : pose bonus penalty act_reg sparse solved done dense
   *  reorient: pos_dist rot_dist act_reg alive sparse solved done dense pos_dist_diff rot_dist_diff
   *  reach   : reach bonus act_reg penalty sparse solved done dense */
  float rwd_weight[MYO_INFO_TERMS];
  /* ---- baoding ---- */
  float drop_th, proximity_th;
  float goal_time_period[2], goal_xrange[2], goal_yrange[2];
  float obj_size_range[2], obj_mass_range[2], obj_friction_change[3];
  int32_t task_choice_random;   /* 1: which_task ~ choice(Task) each reset; 0: fixed_task */
  int32_t fixed_task;           /* used when !task_choice_random (WHICH_TASK = CCW) */
  float overlap_probability, limit_init_angle; /* limit_init_angle <= 0: uniform 0..2pi */
  float noise_fingers;
  float center_pos[2];
  int32_t randomize_physics;    /* 1: sample mass/size/friction per reset (P2); 0: nominal (P1) */
  int32_t ball_body[2], ball_geom[2], ball_site[2], target_site[2];
  int32_t ball_qposadr[2], ball_dofadr[2];
  /* ---- pose ---- */
  float pose_thd, far_th, target_distance;   /* reach: far_th is the whole threshold, ReachEnvV0's far_th x reach_nsite */
  int32_t reset_type;           /* 0 none, 1 init, 2 random, 3 sds */
  int32_t target_type;          /* 0 fixed, 1 generate */
  int32_t n_target_jnt;         /* <=0: target_jnt_value given for all nq */
  int32_t target_jnt_ids[64];
  float target_jnt_range[64][2];
  float target_jnt_value[64];
  /* ---- overrides (filled by the library for baoding; free for other tasks; reach ignores ovr_site and uses its target sites) ---- */
  int32_t n_ovr_body, ovr_body[MYO_MAX_OVERRIDE];
  int32_t n_ovr_geom, ovr_geom[MYO_MAX_OVERRIDE];
  int32_t n_ovr_site, ovr_site[MYO_MAX_OVERRIDE];
  /* ---- rollout glue ---- */
  int32_t clip_actions;         /* 1: clip actions to [-1, 1] first, as RecurrentPPO.collect_rollouts does (np.clip to the
                                   action space) before VecEnv.step; 0: use them as given (plain gym env.step) */
  /* ---- baoding curriculum knobs of CustomBaodingP2Env.reset (/root/reference/src/envs/baoding.py:494-647) ---- */
  int32_t enable_rsi;           /* reference-state initialisation: balls start ON their targets (:606-638) */
  float rsi_probability;
  int32_t balls_overlap;        /* 0: after RSI the start angles are re-drawn uniformly (:634-638) */
  float beta_init_angle[2];     /* (a, b) of np_random.beta; a <= 0: off. Used only with limit_init_angle (:504-520) */
  float beta_ball_size[2], beta_ball_mass[2];   /* (:563-573, :590-600) */
  /* ---- phase-1 env CustomBaodingEnv.reset (/root/reference/src/envs/baoding.py:146-215): start angles 3pi/4 (+ the RSI
   *      phase, drawn whenever enable_rsi), ball placement gated by rsi_probability, then noise on balls / palm / fingers ---- */
  int32_t p1_reset;
  float noise_palm, noise_balls;
  /* ---- die reorientation: CustomReorientEnv._setup / reset (/root/reference/src/envs/reorient.py:58-196) on MyoSuite's
   *      ReorientEnvV0. drop_th and obj_friction_change above are shared with the baoding block. ---- */
  float goal_pos[2], goal_rot[2];          /* ranges of the goal position / Euler-angle offsets */
  float obj_size_change;                   /* die (and target) half sizes +- this much, one draw per reset */
  float pos_th, rot_th;
  int32_t n_goal_rot[3];                   /* goal_rot_x / _y / _z: optional lists of (low, high) ranges, one picked per reset */
  float goal_rot_axis[3][MYO_MAX_ROT_RANGES][2];
  int32_t object_body, goal_body, object_site, goal_site;   /* "Object", "target", "object_o", "target_o" */
  int32_t object_geom0, object_ngeom;      /* geoms of the Object body: the last three scale in all half sizes, earlier ones in size[1] */
  int32_t object_qposadr, object_dofadr;
  float goal_init_pos[3], goal_obj_offset[3];   /* target_o at the initial pose; target_o - object_o there (visualisation offset) */
  int32_t n_ovr_bodypose, ovr_bodypose[MYO_MAX_OVERRIDE];   /* bodies whose body_pos / body_quat are per-world (the goal body) */
  /* ---- pose curriculum knobs of CustomPoseEnv (/root/reference/src/envs/pose.py:55-66, 88-95) ---- */
  float sds_distance;           /* reset_type 3 ("sds"): qpos = (1 - sds_distance) target + sds_distance init_qpos */
  int32_t weight_body;          /* >= 0: body_mass[weight_body] ~ U(weight_range) per reset, geom_size[weight_geom][0] = 0.01 + 2.5 w / 100 */
  int32_t weight_geom;
  float weight_range[2];
  /* ---- reach: MyoSuite ReachEnvV0 (envs/myo/reach_v0.py). Each tip site has a target site ("<tip>_target") whose site_pos
   *      reset() draws uniformly inside (low, high); the targets are per-world MYO_PARAM_SITE_POS overrides. ---- */
  int32_t reach_nsite;                          /* 1 .. MYO_MAX_OVERRIDE (more: MYO_E_LIMIT) */
  int32_t reach_tip_site[MYO_MAX_OVERRIDE], reach_target_site[MYO_MAX_OVERRIDE];
  float reach_range[MYO_MAX_OVERRIDE][2][3];    /* [site][low, high][x, y, z] of the target's site_pos */
  float reach_near_th;                          /* 0.0125 x reach_nsite: bonus below 2 near_th and near_th, solved below near_th */
  int32_t reach_far_steps;                      /* far_th applies from this many elapsed env steps on: ReachEnvV0 compares
                                                   data.time > 2 dt, with time summed in fp64 once per substep (myosuite keeps
                                                   far_th = inf before), so the first such step count is worked out on the host */
} myo_task_cfg;

const char* myo_last_error(void);
const char* myo_version(void);

/* ---- model (host) -------------------------------------------------------------------------- */
int myo_model_load_mjb(const char* path, myo_model** out);
int myo_model_load_mjb_mem(const void* bytes, size_t len, myo_model** out);
void myo_model_free(myo_model* m);
/* integer size by mjModel name ("nq","nv","nu","na","nbody","njnt","ngeom","nsite","ntendon",...) */
int myo_model_size(const myo_model* m, const char* name, int* out);
/* option / statistic by name ("timestep","gravity2","tolerance","iterations","meaninertia",...) */
int myo_model_opt(const myo_model* m, const char* name, double* out);
/* host array by mjModel pointer name. dtype: 0 = float64, 1 = int32, 2 = uint8, 3 = float32, 4 = char.
 * The pointer stays valid until myo_model_free and is writable (sim.model.* semantics): edits made
 * before myo_batch_create are baked into the batch. */
int myo_model_array(myo_model* m, const char* name, void** ptr, int* rows, int* cols, int* dtype);
/* group: "body","jnt"/"joint","geom","site","tendon","actuator" */
int myo_model_name2id(const myo_model* m, const char* group, const char* name);
const char* myo_model_id2name(const myo_model* m, const char* group, int id);
/* fills the baoding id fields of cfg (ball1/ball2 bodies, geoms, sites; target sites) by name */
int myo_task_cfg_default(const myo_model* m, int kind, myo_task_cfg* cfg);
/* Does this model run? MYO_OK, or MYO_E_UNSUPPORTED with EVERY blocking feature listed in `report` (one "- ..." line each;
 * "~ ..." lines are advisory and do not block; report may be NULL) and in myo_last_error(): the answer a user needs for an out-of-band myo_hand_*.mjb
 * (/root/reference/src/envs/__init__.py:17,29,44,62 bind models that are absent from the reference's repository). */
int myo_model_check(const myo_model* m, char* report, size_t report_len);

/* ---- batch (device) ------------------------------------------------------------------------ */
int myo_batch_create(const myo_model* m, int n_worlds, int device, const myo_task_cfg* cfg, uint64_t seed,
                     myo_batch** out);
void myo_batch_destroy(myo_batch* b);
int myo_batch_dims(const myo_batch* b, int* n_worlds, int* nq, int* nv, int* na, int* nu, int* nobs, int* n_param);
/* lanes per world the step kernel uses (8, 16 or 32), and its dynamic shared memory per CTA */
int myo_batch_launch_info(const myo_batch* b, int* lanes_per_world, int* worlds_per_cta, int* smem_bytes,
                          int* regs_per_thread);
/* mask_dev: uint8[n_worlds] or NULL for all worlds. Samples the task's reset distribution on
 * device with a counter-based RNG keyed by (seed, world, episode). obs_dev may be NULL. */
int myo_batch_reset(myo_batch* b, const uint8_t* mask_dev, float* obs_dev, void* stream);
int myo_batch_set_state(myo_batch* b, const float* qpos_dev, const float* qvel_dev, const float* act_dev,
                        const float* time_dev, void* stream);
int myo_batch_get_state(myo_batch* b, float* qpos_dev, float* qvel_dev, float* act_dev, float* time_dev,
                        void* stream);
/* values_dev: float[n_worlds][ncomp] for override slot (kind, id) declared in the task cfg */
int myo_batch_set_param(myo_batch* b, int kind, int id, const float* values_dev, void* stream);
int myo_batch_get_param(myo_batch* b, int kind, int id, float* values_dev, void* stream);
/* Per-world task state - what the reference keeps as attributes of each env object between steps
 * (/root/reference/src/envs/baoding.py:519-557: which_task, ball_{1,2}_starting_angle, x_radius, y_radius, the goal
 * trajectory's time period, counter; /root/reference/src/envs/reorient.py:207-212: pos_dist, rot_dist of the last step).
 *   ti_dev int32[n_worlds][MYO_TASK_STATE_I]: elapsed steps (TimeLimit), episode index (RNG key), task (0 hold, 1 cw, 2 ccw),
 *                                             flags (bit 0: counter = elapsed + 1, the RSI reset's in-reset step)
 *   tf_dev float[n_worlds][MYO_TASK_STATE_F]: start angle 1, start angle 2, x_radius, y_radius, time period, pos_dist, rot_dist, -
 * Either pointer may be NULL. pose_target_dev float[n_worlds][nq]: the pose task's target_jnt_value. */
#define MYO_TASK_STATE_I 4
#define MYO_TASK_STATE_F 8
int myo_batch_get_task_state(myo_batch* b, int32_t* ti_dev, float* tf_dev, float* pose_target_dev, void* stream);
int myo_batch_set_task_state(myo_batch* b, const int32_t* ti_dev, const float* tf_dev, const float* pose_target_dev, void* stream);
/* one env step for every world. actions[n,nu] in [-1,1]; obs[n,nobs]; reward[n]; done[n] (env
 * termination OR time limit, as SB3 sees it); truncated[n] (TimeLimit.truncated);
 * terminal_obs[n,nobs] (written for worlds that finished; may be NULL); info[n,MYO_INFO_TERMS]
 * reward terms + dense (may be NULL). */
int myo_batch_step(myo_batch* b, const float* actions_dev, float* obs_dev, float* reward_dev, uint8_t* done_dev,
                   uint8_t* truncated_dev, float* terminal_obs_dev, float* info_dev, void* stream);
/* raw physics: nsub x mj_step with ctrl[n,nu] applied as data.ctrl (no task logic) */
int myo_batch_mj_step(myo_batch* b, const float* ctrl_dev, int nsub, void* stream);
/* mj_forward at the current state (fills the stage buffers myo_batch_stage_dump reads) */
int myo_batch_forward(myo_batch* b, const float* ctrl_dev, void* stream);
/* current observation without stepping (env.get_obs()) */
int myo_batch_get_obs(myo_batch* b, float* obs_dev, void* stream);

/* per-component parity hooks: copies a stage result of the LAST myo_batch_forward / mj_step
 * substep into out_dev (float or int32 [n_worlds][width]); *width may be queried with out_dev NULL */
typedef enum {
  MYO_STAGE_XPOS = 0,        /* [nbody*3] */
  MYO_STAGE_XMAT = 1,        /* [nbody*9] */
  MYO_STAGE_SITE_XPOS = 2,   /* [nsite*3] */
  MYO_STAGE_TEN_LENGTH = 3,  /* [ntendon] */
  MYO_STAGE_TEN_J = 4,       /* [ntendon*nv] dense */
  MYO_STAGE_QM = 5,          /* [nv*nv] dense mass matrix */
  MYO_STAGE_QFRC_BIAS = 6,   /* [nv] */
  MYO_STAGE_QFRC_PASSIVE = 7,
  MYO_STAGE_QFRC_ACTUATOR = 8,
  MYO_STAGE_ACT_FORCE = 9,   /* [nu] */
  MYO_STAGE_QACC_SMOOTH = 10,
  MYO_STAGE_QACC = 11,
  MYO_STAGE_NCON = 12,       /* int32 [1] */
  MYO_STAGE_CONTACT_GEOMS = 13, /* int32 [ncon_max*2], -1 padded */
  MYO_STAGE_CONTACT_DIST = 14,  /* [ncon_max] */
  MYO_STAGE_NEFC = 15,       /* int32 [1] */
  MYO_STAGE_EFC_TYPE_ID = 16,/* int32 [nefc_max*2] (type,id), -1 padded */
  MYO_STAGE_EFC_J = 17,      /* [nefc_max*nv] dense */
  MYO_STAGE_EFC_AREF = 18,   /* [nefc_max] */
  MYO_STAGE_EFC_D = 19,      /* [nefc_max] */
  MYO_STAGE_EFC_FORCE = 20,  /* [nefc_max] */
  MYO_STAGE_QFRC_CONSTRAINT = 21,
  MYO_STAGE_ACT_DOT = 22,    /* [na] */
  MYO_STAGE_SOLVER_ITER = 23,/* int32 [1] */
  MYO_STAGE_STATUS = 24,     /* int32 [1] bit flags: 1 unsupported pair in range, 2 contact overflow,
                                4 constraint overflow, 8 non-finite state */
  MYO_STAGE_COUNT = 25
} myo_stage;
int myo_batch_stage_dump(myo_batch* b, int stage, void* out_dev, int* width, void* stream);
/* OR of the status flags over all worlds since the last call (host int) */
int myo_batch_status(myo_batch* b, int* flags, void* stream);
/* number of kernel launches issued on behalf of this batch since creation */
int64_t myo_batch_launch_count(const myo_batch* b);

/* Measured FP32 FMA throughput of the device (TFLOP/s, 2 flops per FMA; a few ms): the denominator of bench.py's compute
 * roofline - the world kernel is FP32-issue / latency bound, not HBM bound (DESIGN.md). */
int myo_fp32_fma_peak(int device, double* tflops);

/* ---- recurrent policy forward (sb3-contrib MlpLstmPolicy, separate actor/critic LSTMs) ------ */
typedef struct myo_policy_cfg {
  int32_t obs_dim, act_dim, lstm_hidden;
  int32_t n_pi_layers, pi_layers[4];   /* mlp_extractor policy_net widths (ReLU) */
  int32_t n_vf_layers, vf_layers[4];
  int32_t use_sde;                     /* generalised state-dependent exploration: log_std is [latent_dim][act_dim] (myo_ppo_*;
                                          the rollout side is myo_sde_*; myo_policy_forward itself only produces the mean) */
} myo_policy_cfg;
int myo_policy_create(const myo_policy_cfg* cfg, int max_batch, int device, myo_policy** out);
void myo_policy_destroy(myo_policy* p);
/* name follows the SB3 state-dict key (e.g. "lstm_actor.weight_ih_l0", "action_net.bias", "log_std");
 * data_dev: fp32 device tensor in torch layout */
int myo_policy_set_weight(myo_policy* p, const char* name, const float* data_dev, int64_t numel, void* stream);
/* obs[n,obs_dim] (already normalised unless myo_policy_set_obs_norm is active); h/c: [2][n][H] (0 = actor,
 * 1 = critic), updated in place; episode_start[n] (uint8 0/1, SB3's bool `_last_episode_starts`; the `done`
 * array of myo_batch_step can be passed as is) zeroes the state first; noise[n,act_dim] ~ N(0,1) or NULL for the
 * deterministic mean; outputs: actions[n,act_dim] (unclipped), values[n], logp[n]. */
int myo_policy_forward(myo_policy* p, int n, const float* obs_dev, float* h_dev, float* c_dev,
                       const uint8_t* episode_start_dev, const float* noise_dev, float* actions_dev,
                       float* values_dev, float* logp_dev, void* stream);
/* VecNormalize.normalize_obs fused into the policy's input load (/root/reference/src/main_eval.py:65-67,
 * /root/reference/src/main_baoding.py:75): obs <- clip((obs - mean) / sqrt(var + epsilon), +-clip_obs).
 * mean_dev / var_dev: float[obs_dim] device pointers; NULL switches normalisation off. */
int myo_policy_set_obs_norm(myo_policy* p, const float* mean_dev, const float* var_dev, float epsilon, float clip_obs,
                            void* stream);
/* seed != 0: when noise_dev is NULL, myo_policy_forward samples the Gaussian action noise in-kernel from a
 * counter-based stream keyed by (seed, world, forward-call counter); seed 0 restores the deterministic mean. */
int myo_policy_seed(myo_policy* p, uint64_t seed);
/* 0 (default): bf16 operands, fp32 accumulation on the tensor cores (tcgen05) - the rollout path. 1: plain fp32 arithmetic
 * (library SGEMMs + elementwise kernels), the precision sb3-contrib's torch policy runs at: for evaluating trained reference
 * checkpoints (/root/reference/src/main_eval.py:60-120) without the bf16 rounding of the action mean. Same arguments, same
 * sampling stream. */
int myo_policy_set_precision(myo_policy* p, int precision);
int64_t myo_policy_launch_count(const myo_policy* p);
/* latent_dev: float[max_batch][latent_dim] (latent_dim = last mlp_extractor policy width) that every following
 * myo_policy_forward fills with latent_pi, the input of action_net; NULL stops it. Without policy MLP layers latent_pi is
 * the actor's new hidden state h[0] and nothing is written. */
int myo_policy_set_latent_out(myo_policy* p, float* latent_dev);
/* Generalised state-dependent exploration (SB3 StateDependentNoiseDistribution; `use_sde=True` in the reference's winning
 * runs, /root/reference/docs/summary.md:86-117). log_std: float[latent_dim][act_dim].
 * myo_sde_reset_noise  <- reset_noise / sample_weights: one exploration matrix per world, noise_mat[n][latent_dim][act_dim]
 *                         (bf16 bits) = exp(log_std) * N(0,1), and std2[latent_dim][act_dim] = exp(2 log_std); counter-based
 *                         draws keyed by (seed, world, epoch).
 * myo_sde_sample       <- get_noise + log_prob: actions (holding the mean on entry) += latent . noise_mat[w];
 *                         logp = sum_k log N(noise_k; 0, latent^2 . std2 + 1e-6). */
int myo_sde_reset_noise(uint16_t* noise_mat_dev, float* std2_dev, const float* log_std_dev, int n, int latent_dim, int act_dim,
                        uint64_t seed, uint32_t epoch, void* stream);
int myo_sde_sample(const float* latent_dev, int latent_ld, const uint16_t* noise_mat_dev, const float* std2_dev, float* actions_dev,
                   float* logp_dev, int n, int latent_dim, int act_dim, void* stream);

/* ---- rollout side: VecNormalize running moments, reward scaling, GAE (SURVEY.md 8a rows a14, a17) ------------ */
/* Running moments as SB3's RunningMeanStd keeps them, on the device in fp64: state_dev = mean[d], var[d], count
 * (2 d + 1 doubles; initialise to 0, 1, epsilon as RunningMeanStd.__init__ does).
 * myo_running_moments_update folds the batch x_dev[n][d] (fp32, row-major) into the state exactly as
 * RunningMeanStd.update does (batch mean / population variance, Chan merge). scratch_dev: at least
 * myo_running_moments_scratch(n, d) doubles. mean_f_dev / var_f_dev (optional, float[d]) receive fp32 copies of the new
 * moments, in the form myo_policy_set_obs_norm takes (call it again after an update: it caches 1 / sqrt(var + eps)). */
int myo_running_moments_scratch(int n, int d);
int myo_running_moments_update(double* state_dev, const float* x_dev, int n, int d, double* scratch_dev, float* mean_f_dev,
                               float* var_f_dev, void* stream);
int myo_running_moments_export(const double* state_dev, int d, float* mean_f_dev, float* var_f_dev, void* stream);
/* VecNormalize.step_wait's reward path for one step of n worlds: returns = returns * gamma + reward; (training)
 * ret_rms.update(returns); out = clip(reward / sqrt(ret_rms.var + epsilon), +-clip_reward) (norm_reward) else reward;
 * returns[done] = 0. ret_state_dev: the 3 doubles mean, var, count of ret_rms; returns_dev: double[n];
 * scratch_dev: myo_running_moments_scratch(n, 1) doubles. gamma / epsilon / clip_reward are doubles because SB3 applies
 * them as Python floats to its fp64 return accumulator. */
int myo_vecnorm_reward(double* ret_state_dev, double* returns_dev, const float* reward_dev, const uint8_t* done_dev,
                       float* out_reward_dev, int n, double gamma, double epsilon, double clip_reward, int training,
                       int norm_reward, double* scratch_dev, void* stream);
/* Generalised advantage estimation over a rollout stored step-major ([n_steps][n], SB3's buffer layout):
 *   delta_t = r_t + gamma V_{t+1} (1 - start_{t+1}) - V_t,  A_t = delta_t + gamma lambda (1 - start_{t+1}) A_{t+1},
 * with V_T = last_values and start_T = last_dones; returns = advantages + values. */
int myo_gae(const float* rewards_dev, const float* values_dev, const uint8_t* episode_starts_dev,
            const float* last_values_dev, const uint8_t* last_dones_dev, int n_steps, int n, float gamma, float gae_lambda,
            float* advantages_dev, float* returns_dev, void* stream);

/* VecNormalize.normalize_obs as a stand-alone pass (what the rollout buffer stores: the observation the policy saw):
 * out[n][d] = clip((obs - mean) / sqrt(var + epsilon), +-clip_obs); mean_f / var_f as myo_running_moments_* export them. */
int myo_normalize_obs(const float* obs_dev, const float* mean_f_dev, const float* var_f_dev, float epsilon, float clip_obs,
                      float* out_dev, int n, int d, void* stream);

/* ---- PPO update of the recurrent policy (SURVEY.md 8a row a18) ------------------------------------------------ */
typedef struct myo_ppo_hyper {
  float clip_range;              /* PPO clip on the probability ratio */
  float clip_range_vf;           /* <= 0: no value clipping (SB3 default None) */
  float ent_coef, vf_coef;
  int32_t normalize_advantage;   /* per-minibatch (adv - mean) / (std + 1e-8), torch's unbiased std */
} myo_ppo_hyper;
/* precision: 0 = fp32 GEMMs (parity tests), 1 = bf16 operands with fp32 accumulation (as the rollout kernel computes).
 * max_steps x max_worlds bounds a minibatch (whole sequences of max_worlds worlds). */
int myo_ppo_create(const myo_policy_cfg* cfg, int max_steps, int max_worlds, int precision, int device, myo_ppo** out);
void myo_ppo_destroy(myo_ppo* p);
/* All parameters live in ONE flat fp32 vector owned by the caller (so do the gradient and the Adam moments, same
 * length): myo_ppo_param_count floats; a tensor named by its SB3 state-dict key sits at myo_ppo_param_offset. */
int64_t myo_ppo_param_count(const myo_ppo* p);
int myo_ppo_param_offset(const myo_ppo* p, const char* name, int64_t* offset, int64_t* numel);
/* Loss and gradient of one minibatch = the full n_steps sequences of the n_worlds worlds world_idx_dev[] names, read
 * from the step-major rollout buffers ([n_steps][n_envs][.]): obs (as the policy saw them, i.e. normalised), actions
 * (unclipped samples), episode_starts, old values / log-probs, advantages, returns; h0 / c0: [2][n_envs][H] LSTM
 * states the rollout started from (0 = actor, 1 = critic). Writes the flat gradient (every element) and
 * stats_dev[8] = policy_loss, value_loss, entropy_loss, approx_kl, clip_fraction, loss, adv_mean, adv_std. */
int myo_ppo_minibatch_grad(myo_ppo* p, const float* params_dev, int n_steps, int n_envs, const int32_t* world_idx_dev, int n_worlds,
                           const float* obs_dev, const float* actions_dev, const uint8_t* episode_starts_dev,
                           const float* old_values_dev, const float* old_logp_dev, const float* advantages_dev,
                           const float* returns_dev, const float* h0_dev, const float* c0_dev, const myo_ppo_hyper* hyper,
                           float* grad_dev, float* stats_dev, void* stream);
/* g = grad * grad_scale (1 / world_size after a summing all-reduce); clip_grad_norm_(g, max_grad_norm) (<= 0: off);
 * torch.optim.Adam step number `step` (1-based) on the flat vectors. grad_norm_dev (optional): the norm before clipping. */
int myo_ppo_adam_step(myo_ppo* p, float* params_dev, const float* grad_dev, float* exp_avg_dev, float* exp_avg_sq_dev, int step,
                      float lr, float beta1, float beta2, float eps, float max_grad_norm, float grad_scale, float* grad_norm_dev,
                      void* stream);
int64_t myo_ppo_launch_count(const myo_ppo* p);

#ifdef __cplusplus
}
#endif
#endif /* MYO_B200_H */
