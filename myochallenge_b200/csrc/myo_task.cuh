// Task layer fused around the physics substeps: what the reference does in Python per env.step.
//   baoding: BaodingEnvV1.step target update + CustomBaodingP2Env.get_reward_dict / reset
//            (/root/reference/src/envs/baoding.py:403-467, 494-647), obs layout pinned by
//            /root/reference/src/envs/baoding.py:186-190,627-631 (SURVEY.md 8a row a11)
//   pose   : CustomPoseEnv.reset / get_target_pose (/root/reference/src/envs/pose.py:53-113) on
//            MyoSuite PoseEnvV0 obs / reward keys
//   reach  : MyoSuite 1.2.3 ReachEnvV0 get_obs_dict / get_reward_dict / generate_target_pose + reset, restated from memory
//            ([3P-MEM], SURVEY.md) behind MyoFingerReachFixed / MyoFingerReachRandom (/root/reference/src/envs/environment_factory.py)
//   all    : BaseV0.step muscle action remap, gym TimeLimit, SubprocVecEnv worker auto-reset.
#pragma once
#include "myo_phys.cuh"

namespace myo {

template <int G, int V>
MYO_PHASE void copy_words(Ctx<G, V> c, float* dst, const float* src, int n4) {   // n4: multiple of 4 words
  const float4* s4 = reinterpret_cast<const float4*>(src);
  float4* d4 = reinterpret_cast<float4*>(dst);
  for (int i = c.lane; i < n4 / 4; i += G) d4[i] = s4[i];
}

template <int G, int V>
MYO_PHASE void load_world(int mslot, Ctx<G, V> c, const BatchPtrs& b, int w) {
  MYO_M
  copy_words<G>(c, SF(o_qpos), b.qpos + (size_t)w * m.nq4, m.nq4);
  copy_words<G>(c, SF(o_qvel), b.qvel + (size_t)w * m.nv4, m.nv4);
  copy_words<G>(c, SF(o_warm), b.warm + (size_t)w * m.nv4, m.nv4);
  if (m.na) copy_words<G>(c, SF(o_act), b.act + (size_t)w * m.na4, m.na4);
  copy_words<G>(c, SF(o_wparam), b.wparam + (size_t)w * m.nparam4, m.nparam4);
  if (c.lane == 0) SF(o_misc)[MI_ONE] = 1.f;
  c.tile.sync();
}
template <int G, int V>
MYO_PHASE void store_world(int mslot, Ctx<G, V> c, const BatchPtrs& b, int w, bool params) {
  MYO_M
  c.tile.sync();
  copy_words<G>(c, b.qpos + (size_t)w * m.nq4, SF(o_qpos), m.nq4);
  copy_words<G>(c, b.qvel + (size_t)w * m.nv4, SF(o_qvel), m.nv4);
  copy_words<G>(c, b.warm + (size_t)w * m.nv4, SF(o_warm), m.nv4);
  if (m.na) copy_words<G>(c, b.act + (size_t)w * m.na4, SF(o_act), m.na4);
  if (params) copy_words<G>(c, b.wparam + (size_t)w * m.nparam4, SF(o_wparam), m.nparam4);
}

// BaseV0.step: muscle actuators with normalize_act get ctrl = 1/(1+exp(-5(a-0.5))); other actuators
// are de-normalised linearly into ctrlrange (MyoSuite Robot.normalize_actions).
template <int G, int V>
MYO_PHASE void task_action(int mslot, const myo_task_cfg& t, Ctx<G, V> c, const float* a) {      // a == nullptr: the zero action
  MYO_M
  float* ctrl = SF(o_ctrl);
  for (int i = c.lane; i < m.nu; i += G) {
    float u = a ? a[i] : 0.f;
    if (t.clip_actions) u = clipf(u, -1.f, 1.f);
    if (t.normalize_act) {
      if (m.a_dyntype[i] == 3) u = 1.f / (1.f + expf(-5.f * (u - 0.5f)));
      else {
        const float lo = (m.g_tables + m.a_ctrlrange.off)[2 * i], hi = (m.g_tables + m.a_ctrlrange.off)[2 * i + 1];
        u = 0.5f * (lo + hi) + clipf(u, -1.f, 1.f) * 0.5f * (hi - lo);
      }
    }
    ctrl[i] = u;
  }
}

// BaodingEnvV1.step: target sites follow goal[counter] = sign*2*pi*counter*dt/period (a6, a7)
template <int G, int V>
MYO_PHASE void baoding_targets(int mslot, const myo_task_cfg& t, Ctx<G, V> c, const int* ti, const float* tf) {
  MYO_M
  if (c.lane == 0) {
    const int task = ti[TI_TASK], counter = ti[TI_ELAPSED] + (ti[TI_FLAGS] & 1);   // bit 0: RSI's in-reset step already advanced self.counter
    // BaodingEnvV1.step moves the target sites only for the two rotation tasks; in a hold episode site_pos keeps what
    // the world's previous episode left there (model state is not reset), SURVEY.md row a7
    const float sign = task == MYO_BAODING_CW ? -1.f : 1.f;
    if (task == MYO_BAODING_CW || task == MYO_BAODING_CCW) {
    const float ang = sign * 2.f * kPi * ((float)counter * m.frame_dt / tf[TF_PERIOD]);
#pragma unroll
    for (int k = 0; k < 2; k++) {
      const float th = ang + tf[TF_ANGLE1 + k];
      float sn, cs;
      sincosf(th, &sn, &cs);
      const int slot = m.s_pos_slot[t.target_site[k]];
      if (slot >= 0) {
        c.wpp(m)[slot] = tf[TF_XR] * cs + t.center_pos[0];
        c.wpp(m)[slot + 1] = tf[TF_YR] * sn + t.center_pos[1];
      }
    }
    }
  }
  c.tile.sync();
}

// observation vector into scratch o_obs (kinematics must be current)
template <int G, int V>
MYO_PHASE void task_obs(int mslot, const myo_task_cfg& t, Ctx<G, V> c, const float* pose_target) {
  MYO_M
  float* obs = SF(o_obs);
  const float* qpos = SF(o_qpos); const float* qvel = SF(o_qvel); const float* act = SF(o_act);
  if (t.kind == MYO_TASK_BAODING) {
    const int nh = m.nq - 14;
    for (int i = c.lane; i < nh; i += G) obs[i] = qpos[i];
    for (int i = c.lane; i < m.na; i += G) obs[nh + 24 + i] = act[i];
    for (int k = c.lane; k < 2; k += G) {
      float o[3], g[3];
      site_world(m, c.sp(), c.wpp(m), t.ball_site[k], o);
      site_world(m, c.sp(), c.wpp(m), t.target_site[k], g);
      const int da = t.ball_dofadr[k];
#pragma unroll
      for (int e = 0; e < 3; e++) {
        obs[nh + 6 * k + e] = o[e];                          // object{k}_pos
        obs[nh + 6 * k + 3 + e] = qvel[da + e] * m.frame_dt;   // object{k}_velp
        obs[nh + 12 + 3 * k + e] = g[e];                     // target{k}_pos
        obs[nh + 18 + 3 * k + e] = g[e] - o[e];              // target{k}_err
      }
    }
  } else if (t.kind == MYO_TASK_POSE) {
    for (int i = c.lane; i < m.nq; i += G) { obs[i] = qpos[i]; obs[m.nq + m.nv + i] = pose_target[i] - qpos[i]; }
    for (int i = c.lane; i < m.nv; i += G) obs[m.nq + i] = qvel[i] * m.frame_dt;
    for (int i = c.lane; i < m.na; i += G) obs[2 * m.nq + m.nv + i] = act[i];
  } else if (t.kind == MYO_TASK_REORIENT) {
    // ReorientEnvV0.get_obs_dict: hand_qpos | hand_qvel * dt | obj_pos | goal_pos | pos_err | obj_rot | goal_rot | rot_err | act
    const int nh = m.nq - 7, nhv = m.nv - 6, o0 = nh + nhv;
    for (int i = c.lane; i < nh; i += G) obs[i] = qpos[i];
    for (int i = c.lane; i < nhv; i += G) obs[nh + i] = qvel[i] * m.frame_dt;
    for (int i = c.lane; i < m.na; i += G) obs[o0 + 18 + i] = act[i];
    if (c.lane == 0) {
      float po[3], pg[3], eo[3], eg[3];
      site_world(m, c.sp(), c.wpp(m), t.object_site, po);
      site_world(m, c.sp(), c.wpp(m), t.goal_site, pg);
      mat2euler(eo, SF(o_xmat) + 9 * m.s_body[t.object_site]);      // the sites share their bodies' frames (checked on the host)
      mat2euler(eg, SF(o_xmat) + 9 * m.s_body[t.goal_site]);
#pragma unroll
      for (int e = 0; e < 3; e++) {
        obs[o0 + e] = po[e]; obs[o0 + 3 + e] = pg[e]; obs[o0 + 6 + e] = pg[e] - po[e] - t.goal_obj_offset[e];
        obs[o0 + 9 + e] = eo[e]; obs[o0 + 12 + e] = eg[e]; obs[o0 + 15 + e] = eg[e] - eo[e];
      }
    }
  } else if (t.kind == MYO_TASK_REACH) {
    // ReachEnvV0.get_obs_dict: qpos | qvel * dt | tip_pos | reach_err = target_pos - tip_pos | act, sites in target_reach_range order
    const int o0 = m.nq + m.nv, ns = t.reach_nsite;
    for (int i = c.lane; i < m.nq; i += G) obs[i] = qpos[i];
    for (int i = c.lane; i < m.nv; i += G) obs[m.nq + i] = qvel[i] * m.frame_dt;
    for (int i = c.lane; i < m.na; i += G) obs[o0 + 6 * ns + i] = act[i];
    for (int k = c.lane; k < ns; k += G) {
      float p[3], g[3];
      site_world(m, c.sp(), c.wpp(m), t.reach_tip_site[k], p);
      site_world(m, c.sp(), c.wpp(m), t.reach_target_site[k], g);
#pragma unroll
      for (int e = 0; e < 3; e++) { obs[o0 + 3 * k + e] = p[e]; obs[o0 + 3 * ns + 3 * k + e] = g[e] - p[e]; }
    }
  } else {
    for (int i = c.lane; i < m.nq; i += G) obs[i] = qpos[i];
    for (int i = c.lane; i < m.nv; i += G) obs[m.nq + i] = qvel[i];
    for (int i = c.lane; i < m.na; i += G) obs[m.nq + m.nv + i] = act[i];
  }
  c.tile.sync();
}

// ReachEnvV0.get_reward_dict from the observation in scratch: one distance over all 3 n entries of reach_err. ReachEnvV0 applies
// far_th only once data.time > 2 dt; `elapsed` (env steps since the reset, this one included) stands in for the time.
template <int G, int V>
MYO_PHASE void reach_reward(int mslot, const myo_task_cfg& t, Ctx<G, V> c, int elapsed, float* info, float* reward, bool* done) {
  MYO_M
  const float* obs = SF(o_obs); const float* act = SF(o_act);
  float a2 = 0.f;
  for (int i = c.lane; i < m.na; i += G) a2 += act[i] * act[i];
  a2 = tile_sum<G>(c, a2);
  const float act_mag = m.na ? sqrtf(a2) / (float)m.na : 0.f;
  const float* err = obs + m.nq + m.nv + 3 * t.reach_nsite;
  float e2 = 0.f;
  for (int i = 0; i < 3 * t.reach_nsite; i++) e2 += err[i] * err[i];
  const float d = sqrtf(e2), near = t.reach_near_th;
  const bool far = elapsed >= t.reach_far_steps && d > t.far_th;
  float term[MYO_INFO_TERMS];
#pragma unroll
  for (int k = 0; k < MYO_INFO_TERMS; k++) term[k] = 0.f;
  term[0] = -d; term[1] = (d < 2.f * near ? 1.f : 0.f) + (d < near ? 1.f : 0.f); term[2] = -act_mag;
  term[3] = far ? -1.f : 0.f; term[4] = -d; term[5] = d < near ? 1.f : 0.f; term[6] = far ? 1.f : 0.f;
  float dense = 0.f;
#pragma unroll
  for (int k = 0; k < MYO_INFO_TERMS; k++) if (k != 7) dense += t.rwd_weight[k] * term[k];
  term[7] = dense;
#pragma unroll
  for (int k = 0; k < MYO_INFO_TERMS; k++) info[k] = term[k];
  *reward = dense; *done = far;
}

// reward terms + dense reward + termination from the observation in scratch. info: MYO_INFO_TERMS floats. elapsed: env steps
// since the reset, this one included.
template <int G, int V>
MYO_PHASE void task_reward(int mslot, const myo_task_cfg& t, Ctx<G, V> c, float* tf, int elapsed, float* info, float* reward, bool* done) {
  MYO_M
  if (t.kind == MYO_TASK_REACH) { reach_reward<G>(mslot, t, c, elapsed, info, reward, done); return; }
  const float* obs = SF(o_obs); const float* act = SF(o_act);
  float a2 = 0.f;
  for (int i = c.lane; i < m.na; i += G) a2 += act[i] * act[i];
  a2 = tile_sum<G>(c, a2);
  const float act_mag = m.na ? sqrtf(a2) / (float)m.na : 0.f;
  float term[MYO_INFO_TERMS];
#pragma unroll
  for (int k = 0; k < MYO_INFO_TERMS; k++) term[k] = 0.f;
  bool dn = false;
  if (t.kind == MYO_TASK_BAODING) {
    const int nh = m.nq - 14;
    const float* e1 = obs + nh + 18; const float* e2 = obs + nh + 21;
    const float d1 = norm3(e1), d2 = norm3(e2);
    const bool fall = obs[nh + 2] < t.drop_th || obs[nh + 8] < t.drop_th;
    term[0] = -d1; term[1] = -d2; term[2] = -act_mag; term[3] = fall ? 0.f : 1.f; term[4] = -(d1 + d2);
    term[5] = (d1 < t.proximity_th && d2 < t.proximity_th && !fall) ? 1.f : 0.f;
    term[6] = fall ? 1.f : 0.f;
    dn = fall;
  } else if (t.kind == MYO_TASK_POSE) {
    float e2 = 0.f;
    for (int i = c.lane; i < m.nq; i += G) { const float e = obs[m.nq + m.nv + i]; e2 += e * e; }
    const float dist = sqrtf(tile_sum<G>(c, e2));
    term[0] = -dist;
    term[1] = (dist < t.pose_thd ? 1.f : 0.f) + (dist < 1.5f * t.pose_thd ? 1.f : 0.f);
    term[2] = dist > t.far_th ? -1.f : 0.f;
    term[3] = -act_mag; term[4] = -dist; term[5] = dist < t.pose_thd ? 1.f : 0.f;
    term[6] = dist > t.far_th ? 1.f : 0.f;
    dn = dist > t.far_th;
  } else if (t.kind == MYO_TASK_REORIENT) {
    // CustomReorientEnv.get_reward_dict (/root/reference/src/envs/reorient.py:11-56): distances, their decrease since the last
    // step (self.pos_dist / self.rot_dist, refreshed in step() and reset()), drop = pos_dist > drop_th
    const int o0 = (m.nq - 7) + (m.nv - 6);
    const float pd = norm3(obs + o0 + 6), rd = norm3(obs + o0 + 15);
    const bool drop = pd > t.drop_th;
    term[0] = -pd; term[1] = -rd; term[2] = -act_mag; term[3] = drop ? 0.f : 1.f; term[4] = -rd - 10.f * pd;
    term[5] = (pd < t.pos_th && rd < t.rot_th && !drop) ? 1.f : 0.f;
    term[6] = drop ? 1.f : 0.f;
    term[8] = tf[TF_POSDIST] - pd; term[9] = tf[TF_ROTDIST] - rd;
    dn = drop;
    c.tile.sync();
    if (c.lane == 0) { tf[TF_POSDIST] = pd; tf[TF_ROTDIST] = rd; }      // step(): self.pos_dist / self.rot_dist <- this step's
  }
  float dense = 0.f;
#pragma unroll
  for (int k = 0; k < MYO_INFO_TERMS; k++) if (k != 7) dense += t.rwd_weight[k] * term[k];
  term[7] = dense;
#pragma unroll
  for (int k = 0; k < MYO_INFO_TERMS; k++) info[k] = term[k];
  *reward = dense; *done = dn;
}

// does this task's reset run physics (the reference's RSI branch calls self.step(zeros) inside reset())? Such resets are only
// performed by the one-world-per-CTA kernel (SOLO), which may call the substep phases conditionally.
inline __host__ __device__ bool reset_needs_physics(const myo_task_cfg& t) { return t.kind == MYO_TASK_BAODING && t.enable_rsi != 0; }

// env.reset(): sample the task's reset distribution with a counter-based RNG keyed by
// (seed, world, episode) and write the initial state into scratch.
template <int G, int RMAX, bool SOLO, int V>
MYO_PHASE void task_reset(int mslot, const myo_task_cfg& t, Ctx<G, V> c, const BatchPtrs& b, int w, int* ti,
                           float* tf, float* pose_target) {
  MYO_M
  float* qpos = SF(o_qpos);
  const int episode = ti[TI_EPISODE] + 1;
  float nf_th = 0.f, nf_fl = 0.f;      // phase-2 finger noise (lane 0), applied after the RSI branch as the reference orders it
  c.tile.sync();
  if (!(t.kind == MYO_TASK_POSE && t.reset_type == 0)) {   // reset_type "none" keeps the last state
    for (int i = c.lane; i < m.nq; i += G) qpos[i] = m.init_qpos[i];
    for (int i = c.lane; i < m.nv; i += G) { SF(o_qvel)[i] = 0.f; SF(o_warm)[i] = 0.f; }
    for (int i = c.lane; i < m.na; i += G) SF(o_act)[i] = 0.f;
  }
  c.tile.sync();
  if (c.lane == 0) {
    Philox rng;
    rng.init(b.seed, (uint32_t)w, (uint32_t)episode);
    ti[TI_EPISODE] = episode; ti[TI_ELAPSED] = 0;
    if (t.kind == MYO_TASK_BAODING && t.p1_reset) {
      // CustomBaodingEnv.reset (phase 1, /root/reference/src/envs/baoding.py:146-215)
      ti[TI_TASK] = t.task_choice_random ? min(2, (int)(rng.uniform() * 3.f)) : t.fixed_task;      // sample_task
      const float phase = t.enable_rsi ? rng.uniform(-kPi, kPi) : 0.f;
      tf[TF_ANGLE1] = 0.75f * kPi + phase; tf[TF_ANGLE2] = -0.25f * kPi + phase;
      tf[TF_XR] = rng.uniform(t.goal_xrange[0], t.goal_xrange[1]);
      tf[TF_YR] = rng.uniform(t.goal_yrange[0], t.goal_yrange[1]);
      tf[TF_PERIOD] = rng.uniform(t.goal_time_period[0], t.goal_time_period[1]);
      ti[TI_FLAGS] = 0;
      if (t.enable_rsi && rng.uniform() < t.rsi_probability) {      // self.step(zeros) + balls onto the targets (closed form, see below)
        ti[TI_FLAGS] = 1;
        if (ti[TI_TASK] == MYO_BAODING_CW || ti[TI_TASK] == MYO_BAODING_CCW) {
#pragma unroll
          for (int k = 0; k < 2; k++) {
            float sn, cs;
            sincosf(tf[TF_ANGLE1 + k], &sn, &cs);
            const int slot = m.s_pos_slot[t.target_site[k]];
            if (slot >= 0) { c.wpp(m)[slot] = tf[TF_XR] * cs + t.center_pos[0]; c.wpp(m)[slot + 1] = tf[TF_YR] * sn + t.center_pos[1]; }
          }
        }
      }
    } else if (t.kind == MYO_TASK_BAODING) {
      float a1;
      if (t.task_choice_random) {
        ti[TI_TASK] = min(2, (int)(rng.uniform() * 3.f));
        const float u = rng.uniform();
        if (u < t.overlap_probability) a1 = 0.75f * kPi;
        else if (t.limit_init_angle > 0.f) {
          float phase = rng.uniform(-t.limit_init_angle, t.limit_init_angle);
          if (t.beta_init_angle[0] > 0.f) phase = rng.beta(t.beta_init_angle[0], t.beta_init_angle[1]) * 2.f * kPi - kPi;
          a1 = 0.75f * kPi + phase;
        }
        else a1 = rng.uniform(0.f, 2.f * kPi);
      } else {
        // task_choice "fixed": the start angles are drawn ONCE per env object, in _setup (:326-331), and reset() never touches
        // them again: one draw per world, the same in every episode
        ti[TI_TASK] = t.fixed_task;
        Philox once;
        once.init(b.seed ^ 0xD1B54A32D192ED03ull, (uint32_t)w, 0u);
        a1 = (once.uniform() < t.overlap_probability) ? 0.75f * kPi : 0.25f * kPi;
      }
      tf[TF_ANGLE1] = a1; tf[TF_ANGLE2] = a1 - kPi;
      tf[TF_XR] = rng.uniform(t.goal_xrange[0], t.goal_xrange[1]);
      tf[TF_YR] = rng.uniform(t.goal_yrange[0], t.goal_yrange[1]);
      tf[TF_PERIOD] = rng.uniform(t.goal_time_period[0], t.goal_time_period[1]);
      if (t.randomize_physics) {
#pragma unroll
        for (int k = 0; k < 2; k++) {
          const int ms = m.b_mass_slot[t.ball_body[k]];
          if (ms >= 0) c.wpp(m)[ms] = rng.uniform(t.obj_mass_range[0], t.obj_mass_range[1]);
        }
        if (t.beta_ball_mass[0] > 0.f) {
#pragma unroll
          for (int k = 0; k < 2; k++) {
            const int ms = m.b_mass_slot[t.ball_body[k]];
            const float v = rng.beta(t.beta_ball_mass[0], t.beta_ball_mass[1]) * (t.obj_mass_range[1] - t.obj_mass_range[0]) + t.obj_mass_range[0];
            if (ms >= 0) c.wpp(m)[ms] = v;
          }
        }
#pragma unroll
        for (int k = 0; k < 2; k++) {
          const int fs = m.g_fri_slot[t.ball_geom[k]];
          for (int e = 0; e < 3; e++) {
            const float nominal = m.g_friction[3 * t.ball_geom[0] + e];
            const float v = rng.uniform(nominal - t.obj_friction_change[e], nominal + t.obj_friction_change[e]);
            if (fs >= 0) c.wpp(m)[fs + e] = v;
          }
        }
#pragma unroll
        for (int k = 0; k < 2; k++) {
          const int ss = m.g_size_slot[t.ball_geom[k]];
          const float v = rng.uniform(t.obj_size_range[0], t.obj_size_range[1]);
          if (ss >= 0) { c.wpp(m)[ss] = v; c.wpp(m)[ss + 1] = v; c.wpp(m)[ss + 2] = v; }
        }
        if (t.beta_ball_size[0] > 0.f) {
#pragma unroll
          for (int k = 0; k < 2; k++) {
            const int ss = m.g_size_slot[t.ball_geom[k]];
            const float v = rng.beta(t.beta_ball_size[0], t.beta_ball_size[1]) * (t.obj_size_range[1] - t.obj_size_range[0]) + t.obj_size_range[0];
            if (ss >= 0) { c.wpp(m)[ss] = v; c.wpp(m)[ss + 1] = v; c.wpp(m)[ss + 2] = v; }
          }
        }
      }
      // RSI (/root/reference/src/envs/baoding.py:606-638): new start angles, one env.step(zeros) on the freshly reset env,
      // then the balls are put on the targets' world xy as that step's observation shows them, and set_state(qpos, qvel)
      // restores the hand pose and zero velocities (activations, time and the warm start keep what the step left). The
      // targets ride on the palm, which sags a little during the step, so the step is really run (below, SOLO kernel).
      ti[TI_FLAGS] = 0;
      if (t.enable_rsi && rng.uniform() < t.rsi_probability) {
        ti[TI_FLAGS] = 1;
        const float phase = rng.uniform(-kPi, kPi);
        a1 = 0.75f * kPi + phase;
        tf[TF_ANGLE1] = a1; tf[TF_ANGLE2] = -0.25f * kPi + phase;
        if (ti[TI_TASK] == MYO_BAODING_CW || ti[TI_TASK] == MYO_BAODING_CCW) {
#pragma unroll
          for (int k = 0; k < 2; k++) {          // goal[0] = 0: the targets sit at the start angles
            float sn, cs;
            sincosf(tf[TF_ANGLE1 + k], &sn, &cs);
            const int slot = m.s_pos_slot[t.target_site[k]];
            if (slot >= 0) { c.wpp(m)[slot] = tf[TF_XR] * cs + t.center_pos[0]; c.wpp(m)[slot + 1] = tf[TF_YR] * sn + t.center_pos[1]; }
          }
        }
        if (!t.balls_overlap) { tf[TF_ANGLE1] = rng.uniform(0.f, 2.f * kPi); tf[TF_ANGLE2] = tf[TF_ANGLE1] - kPi; }
      }
      if (t.noise_fingers > 0.f && m.nq - 14 >= 23) {   // _add_noise_to_finger_positions: one draw per group
        nf_th = rng.uniform(-kPi / 18.f * t.noise_fingers, kPi / 18.f * t.noise_fingers);
        nf_fl = rng.uniform(0.f, kPi / 6.f * t.noise_fingers);
      }
    } else if (t.kind == MYO_TASK_REORIENT) {
      // CustomReorientEnv.reset (/root/reference/src/envs/reorient.py:127-178): goal position, goal orientation (set_orientation,
      // :180-205), die friction, one size offset for die and target. The RSI branch only edits body_pos / body_quat of the
      // free-jointed die, which MuJoCo's kinematics never reads (a free body's pose is its qpos): it changes nothing.
      const int ps = m.b_pose_slot[t.goal_body];
      if (ps >= 0) {
        for (int e = 0; e < 3; e++) c.wpp(m)[ps + e] = t.goal_init_pos[e] + rng.uniform(t.goal_pos[0], t.goal_pos[1]);
        float lo[3], hi[3];
        for (int ax = 0; ax < 3; ax++) {      // the three range choices first, then the three angles (the reference's draw order)
          lo[ax] = t.goal_rot[0]; hi[ax] = t.goal_rot[1];
          if (t.n_goal_rot[ax] > 0) {
            const int k = min(t.n_goal_rot[ax] - 1, (int)(rng.uniform() * (float)t.n_goal_rot[ax]));
            lo[ax] = t.goal_rot_axis[ax][k][0]; hi[ax] = t.goal_rot_axis[ax][k][1];
          }
        }
        float eul[3], q[4], R[9];
        for (int ax = 0; ax < 3; ax++) eul[ax] = rng.uniform(lo[ax], hi[ax]);
        euler2quat(q, eul);
        quat2mat(R, q);
        for (int e = 0; e < 9; e++) c.wpp(m)[ps + 3 + e] = R[e];
      }
      for (int k = 0; k < t.object_ngeom; k++) {
        const int g = t.object_geom0 + k, fs = m.g_fri_slot[g];
        for (int e = 0; e < 3; e++) {
          const float nominal = m.g_friction[3 * g + e];
          const float v = rng.uniform(nominal - t.obj_friction_change[e], nominal + t.obj_friction_change[e]);
          if (fs >= 0) c.wpp(m)[fs + e] = v;
        }
      }
      const float del = rng.uniform(-t.obj_size_change, t.obj_size_change);
      for (int k = 0; k < t.object_ngeom; k++) {
        const int g = t.object_geom0 + k, ss = m.g_size_slot[g];
        if (ss < 0) continue;
        const bool slab = k >= t.object_ngeom - 3;       // the last three geoms grow in every half size, earlier ones in size[1]
        for (int e = 0; e < 3; e++) c.wpp(m)[ss + e] = m.g_size[3 * g + e] + ((slab || e == 1) ? del : 0.f);
      }
    } else if (t.kind == MYO_TASK_POSE) {
      if (t.weight_body >= 0) {      // CustomPoseEnv.reset: a new weight, and the size of its first geom with it (pose.py:55-66)
        const float wgt = rng.uniform(t.weight_range[0], t.weight_range[1]);
        const int ms = m.b_mass_slot[t.weight_body], ss = t.weight_geom >= 0 ? m.g_size_slot[t.weight_geom] : -1;
        if (ms >= 0) c.wpp(m)[ms] = wgt;
        if (ss >= 0) c.wpp(m)[ss] = 0.01f + 2.5f * wgt / 100.f;
      }
      // update_target: sample target_jnt_value inside target_jnt_range, then get_target_pose scales the
      // distance from init_qpos by target_distance
      for (int i = 0; i < m.nq; i++) pose_target[i] = (t.n_target_jnt > 0) ? 0.f : t.target_jnt_value[i];
      if (t.n_target_jnt > 0) {
        for (int k = 0; k < t.n_target_jnt; k++) {
          const float lo = t.target_jnt_range[k][0], hi = t.target_jnt_range[k][1];
          const float v = (t.target_type == 1) ? rng.uniform(lo, hi) : 0.5f * (lo + hi);
          pose_target[m.j_qposadr[t.target_jnt_ids[k]]] = v;
        }
      }
      for (int i = 0; i < m.nq; i++) pose_target[i] = m.init_qpos[i] + t.target_distance * (pose_target[i] - m.init_qpos[i]);
      if (t.reset_type == 3) {   // "sds": start between the target and the initial pose (pose.py:88-95)
        for (int i = 0; i < m.nq; i++) qpos[i] = (1.f - t.sds_distance) * pose_target[i] + t.sds_distance * m.init_qpos[i];
      }
      if (t.reset_type == 2) {   // "random": uniform inside jnt_range for every joint
        for (int j = 0; j < m.njnt; j++)
          if (m.j_type[j] == J_HINGE || m.j_type[j] == J_SLIDE)
            qpos[m.j_qposadr[j]] = rng.uniform(m.j_range[2 * j], m.j_range[2 * j + 1]);
      }
    } else if (t.kind == MYO_TASK_REACH) {
      // ReachEnvV0.generate_target_pose: site_pos[<tip>_target] = np_random.uniform(low, high), x y z of each site in turn
      for (int k = 0; k < t.reach_nsite; k++) {
        const int slot = m.s_pos_slot[t.reach_target_site[k]];
        for (int e = 0; e < 3; e++) {
          const float v = rng.uniform(t.reach_range[k][0][e], t.reach_range[k][1][e]);
          if (slot >= 0) c.wpp(m)[slot + e] = v;
        }
      }
    }
  }
  c.tile.sync();
  if constexpr (SOLO) {
    if (t.kind == MYO_TASK_BAODING && t.enable_rsi && (ti[TI_FLAGS] & 1)) {
      // self.step(np.zeros(nu)): the target sites already sit at goal[0] + the RSI angles (rotation tasks), the zero action
      // goes through BaseV0.step's remap, Robot.step runs frame_skip substeps, get_obs -> sim.forward
      task_action<G>(mslot, t, c, nullptr);
      c.tile.sync();
      int st = 0;
      for (int sub = 0; sub < t.frame_skip; sub++) mj_step_dev<G, RMAX, false>(mslot, c, &st, true);
      phase_tree_forward<G>(mslot, c, false);
      float g[2][3];
#pragma unroll
      for (int k = 0; k < 2; k++) site_world(m, c.sp(), c.wpp(m), t.target_site[k], g[k]);
      c.tile.sync();
      // qpos = init_qpos.copy(); qpos[23, 24] = obs[35, 36]; qpos[30, 31] = obs[38, 39]; set_state(qpos, init_qvel) (:627-632)
      for (int i = c.lane; i < m.nq; i += G) qpos[i] = m.init_qpos[i];
      for (int i = c.lane; i < m.nv; i += G) SF(o_qvel)[i] = 0.f;
      c.tile.sync();
      if (c.lane == 0) {
#pragma unroll
        for (int k = 0; k < 2; k++) { qpos[t.ball_qposadr[k]] = g[k][0]; qpos[t.ball_qposadr[k] + 1] = g[k][1]; }
      }
      c.tile.sync();
    }
  }
  if (t.kind == MYO_TASK_BAODING && !t.p1_reset && t.noise_fingers > 0.f && m.nq - 14 >= 23) {
    if (c.lane == 0) {
      qpos[4] = nf_th; qpos[5] = nf_th; qpos[6] = nf_th;
      const int idx[12] = {7, 9, 10, 11, 13, 14, 15, 17, 18, 19, 21, 22};
#pragma unroll
      for (int k = 0; k < 12; k++) qpos[idx[k]] = nf_fl;
    }
    c.tile.sync();
  }
  if (t.kind == MYO_TASK_BAODING && t.p1_reset && (t.noise_balls > 0.f || t.noise_palm > 0.f || t.noise_fingers > 0.f) && m.nq - 14 >= 23) {
    if (c.lane == 0) {     // phase-1 noise, applied after the RSI ball placement as the reference orders it (:196-210)
      Philox rng;
      rng.init(b.seed ^ 0x9E3779B97F4A7C15ull, (uint32_t)w, (uint32_t)ti[TI_EPISODE]);
      if (t.noise_balls > 0.f)
        for (int k = 0; k < 2; k++) for (int e = 0; e < 3; e++) qpos[t.ball_qposadr[k] + e] += rng.uniform(-t.noise_balls, t.noise_balls);
      if (t.noise_palm > 0.f) {       // _add_noise_to_palm_position
        qpos[0] = rng.uniform(-0.5f * kPi, -0.5f * kPi + kPi / 18.f * t.noise_palm);
        qpos[1] = rng.uniform(-kPi / 18.f * t.noise_palm, kPi / 18.f * t.noise_palm);
        qpos[2] = rng.uniform(-kPi / 18.f * t.noise_palm, kPi / 18.f * t.noise_palm);
      }
      if (t.noise_fingers > 0.f) {    // phase-1 _add_noise_to_finger_positions: thumb 3..6, flexions, abductions - one draw per group
        const float th = rng.uniform(-kPi / 18.f * t.noise_fingers, kPi / 18.f * t.noise_fingers);
        qpos[3] = th; qpos[4] = th; qpos[5] = th; qpos[6] = th;
        const float fl = rng.uniform(0.f, kPi / 6.f * t.noise_fingers);
        const int idx[12] = {7, 9, 10, 11, 13, 14, 15, 17, 18, 19, 21, 22};
#pragma unroll
        for (int k = 0; k < 12; k++) qpos[idx[k]] = fl;
        const float ab = rng.uniform(-kPi / 36.f * t.noise_fingers, kPi / 36.f * t.noise_fingers);
        qpos[8] = ab; qpos[12] = ab; qpos[16] = ab; qpos[20] = ab;
      }
    }
    c.tile.sync();
  }
  if (t.kind == MYO_TASK_REORIENT) {      // reset(): self.pos_dist / self.rot_dist from the reset observation (reorient.py:176-177)
    phase_tree_forward<G>(mslot, c, false);
    task_obs<G>(mslot, t, c, pose_target);
    if (c.lane == 0) {
      const int o0 = (m.nq - 7) + (m.nv - 6);
      tf[TF_POSDIST] = norm3(SF(o_obs) + o0 + 6); tf[TF_ROTDIST] = norm3(SF(o_obs) + o0 + 15);
    }
    c.tile.sync();
  }
}

}  // namespace myo
