// Physics phases of one mj_step for one world held in shared memory, executed by a tile of G lanes.
// Each phase states the MuJoCo 2.1.0 stage it reproduces (SURVEY.md 8a rows a10.1-a10.9); the
// reference reaches them through env.step -> Robot.step -> sim.step
// (/root/reference/src/envs/baoding.py:183,625; /root/reference/src/envs/pose.py:102).
#pragma once
#include <cooperative_groups.h>

#include "myo_dev.hpp"
#include "myo_math.cuh"

namespace myo {
namespace cg = cooperative_groups;

// V: code variant. The full-capacity passes instantiate every phase with V = 1, i.e. as separate functions, so that the register
// conventions ptxas derives for the fast path's phases are not widened by the deeper call graph of those passes (measured:
// sharing the functions cost the fast path 5 %).
template <int G, int V = 0>
struct Ctx {
  cg::thread_block_tile<G> tile;
  int lane;
  int soff;          // word offset of this world's scratch inside the CTA's dynamic shared memory
  __device__ Ctx(cg::thread_block_tile<G> t) : tile(t), lane(t.thread_rank()), soff(0) {}
  // Scratch pointers are always re-derived from the __shared__ base, never carried as pointers: the compiler then
  // knows the address space inside the (noinline) phases and emits LDS/STS with 32-bit addresses instead of
  // generic LD/ST + memory descriptors (round-1 profile: 739 M generic loads, 1054 M R2UR per 8192-world step).
  MYO_DI float* sp() const { return MYO_SMEM_WORDS + soff; }
  MYO_DI float* wpp(const DevModel& m) const { return MYO_SMEM_WORDS + soff + m.o_wparam; }   // per-world override parameters
};

// cold model table (global memory only, see Builder::Fcold in myo_pack.cpp)
#define GT(field) (m.g_tables + m.field.off)
#define SF(field) (MYO_SMEM_WORDS + c.soff + m.field)
#define SI(field) (reinterpret_cast<int*>(MYO_SMEM_WORDS + c.soff + m.field))
#define SO(off) (MYO_SMEM_WORDS + c.soff + (off))   // scratch word offset -> pointer (noinline phases take offsets, not pointers)

// optional per-phase cycle counters (development builds: -DMYO_PROFILE)
#ifdef MYO_PROFILE
__device__ unsigned long long g_prof[16];
#define MYO_PH_BEGIN long long ph_t0 = clock64();
#define MYO_PH_RESTART ph_t0 = clock64();
#define MYO_PH(i) { long long ph_t = clock64(); if (c.lane == 0) atomicAdd(&g_prof[i], (unsigned long long)(ph_t - ph_t0)); ph_t0 = clock64(); }
#else
#define MYO_PH_BEGIN
#define MYO_PH_RESTART
#define MYO_PH(i)
#endif

template <int G, int V> MYO_DI float tile_sum(const Ctx<G, V> c, float v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += c.tile.shfl_xor(v, o);
  return v;
}
template <int G, int V> MYO_DI float tile_max(const Ctx<G, V> c, float v) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v = fmaxf(v, c.tile.shfl_xor(v, o));
  return v;
}

// support index / Jacobian value e of a limit record (see L_IOFF / L_JOFF in myo_dev.hpp); s = the world's scratch
MYO_DI int lim_idx(const int* li, int e) { return reinterpret_cast<const int*>(MYO_SMEM_WORDS)[li[L_IOFF] + e]; }
MYO_DI float lim_J(const float* s, const float* lr, const int* li, int e) { return lr[L_SIGN] * s[li[L_JOFF] + e]; }

// Entry e of a contact's Jacobian block (see C_CP in myo_dev.hpp): the dof and the three basis rows (normal, tangent 1,
// tangent 2) = +-frame . (lin_d + ang_d x (pos - tree reference)), - on the body-A side. s = the world's scratch.
MYO_DI int contact_entry(const DevModel& m, const float* s, const float* cr, const int* ci, int e, float* jn, float* jt1, float* jt2) {
  const int cp = ci[C_CP] & 255, na = ci[C_CP] >> 8;
  const bool onb = e >= na;
  const int body = onb ? ci[C_BB] : ci[C_BA];
  const int d = m.b_chain[body * KC + cp + (onb ? e - na : e)];
  const float sgn = onb ? 1.f : -1.f;
  float off[3], t[3];
  sub3(off, cr + C_POS, s + m.o_xipos + 3 * m.b_root[body]);
  const float* cd = s + m.o_cdof + 6 * d;
  cross3(t, cd, off);
  const float v[3] = {cd[3] + t[0], cd[4] + t[1], cd[5] + t[2]};
  *jn = sgn * dot3(cr + C_FRAME, v);
  *jt1 = sgn * dot3(cr + C_FRAME + 3, v);
  *jt2 = sgn * dot3(cr + C_FRAME + 6, v);
  return d;
}

// ------------------------------------------------------------------------------------------------
// a10.1 kinematics + comPos (+ comVel + RNE forward when dyn).
// Reference point of every kinematic tree = xipos of its root body (MuJoCo uses the subtree COM;
// the dynamics are invariant to that choice and a nearby point keeps fp32 cross products small).
// Split so that only a short composition sits on the serial level-by-level path:
//   A  (all bodies at once)  pose of the body in its PARENT's frame from qpos (Rodrigues per hinge, no quaternions);
//                            hinge axis | anchor and slide axis in the parent's frame, parked in the dof's cdof slot
//   B  (level by level)      world pose = parent's world pose o local pose (27 + 9 FMA per body)
//   C  (all at once)         xipos, then cdof about the tree reference, cinert
//   D  (level by level, dyn) cvel, cdof_dot, cacc (mj_comVel / mj_rne forward), cfrc
MYO_DI void rodrigues(float* R, const float* a, float ang) {
  float sn, cs;
  sincosf(ang, &sn, &cs);
  const float t = 1.f - cs;
  R[0] = cs + t * a[0] * a[0];        R[1] = t * a[0] * a[1] - sn * a[2]; R[2] = t * a[0] * a[2] + sn * a[1];
  R[3] = t * a[0] * a[1] + sn * a[2]; R[4] = cs + t * a[1] * a[1];        R[5] = t * a[1] * a[2] - sn * a[0];
  R[6] = t * a[0] * a[2] - sn * a[1]; R[7] = t * a[1] * a[2] + sn * a[0]; R[8] = cs + t * a[2] * a[2];
}

template <int G, int V>
MYO_PHASE void body_local_pose(int mslot, Ctx<G, V> c, int b) {
  MYO_M
  const float* qpos = SF(o_qpos);
  float* cdof = SF(o_cdof);
  const int jadr = m.b_jntadr[b], jnum = m.b_jntnum[b];
  float R[9], pos[3];
  if (jnum == 1 && m.j_type[jadr] == J_FREE) {
    const int qa = m.j_qposadr[jadr];
    float q[4] = {qpos[qa + 3], qpos[qa + 4], qpos[qa + 5], qpos[qa + 6]};
    pos[0] = qpos[qa]; pos[1] = qpos[qa + 1]; pos[2] = qpos[qa + 2];
    normalize4(q);
    quat2mat(R, q);
  } else {
    const int ps = m.b_pose_slot[b];      // per-world body_pos / body_quat (the reorient goal body)
    if (ps >= 0) {
      cpy3(pos, c.wpp(m) + ps);
#pragma unroll
      for (int k = 0; k < 9; k++) R[k] = c.wpp(m)[ps + 3 + k];
    } else {
#pragma unroll
      for (int k = 0; k < 9; k++) R[k] = m.b_mat[9 * b + k];
      cpy3(pos, m.b_pos + 3 * b);
    }
    for (int j = jadr; j < jadr + jnum; j++) {
      const int qa = m.j_qposadr[j], da = m.j_dofadr[j];
      const float dq = qpos[qa] - m.j_qpos0[j];
      float ax[3];
      mulmatvec3(ax, R, m.j_axis + 3 * j);
      if (m.j_type[j] == J_SLIDE) {
        pos[0] += ax[0] * dq; pos[1] += ax[1] * dq; pos[2] += ax[2] * dq;
        cdof[6 * da] = ax[0]; cdof[6 * da + 1] = ax[1]; cdof[6 * da + 2] = ax[2];
      } else {
        float anchor[3], Rj[9], vec[3];
        mulmatvec3(anchor, R, m.j_pos + 3 * j);
        add3(anchor, anchor, pos);
        rodrigues(Rj, m.j_axis + 3 * j, dq);
        mulmat3(R, R, Rj);
        mulmatvec3(vec, R, m.j_pos + 3 * j);
        sub3(pos, anchor, vec);
        cdof[6 * da] = ax[0]; cdof[6 * da + 1] = ax[1]; cdof[6 * da + 2] = ax[2];
        cdof[6 * da + 3] = anchor[0]; cdof[6 * da + 4] = anchor[1]; cdof[6 * da + 5] = anchor[2];
      }
    }
  }
  float* xp = SF(o_xpos) + 3 * b;
  float* xm = SF(o_xmat) + 9 * b;
  cpy3(xp, pos);
#pragma unroll
  for (int k = 0; k < 9; k++) xm[k] = R[k];
}

template <int G, int V>
MYO_PHASE void phase_tree_forward(int mslot, Ctx<G, V> c, bool dyn) {
  MYO_M
  if (c.lane == 0) {
    float* xp = SF(o_xpos); float* xm = SF(o_xmat); float* xi = SF(o_xipos);
    xp[0] = xp[1] = xp[2] = 0.f; xi[0] = xi[1] = xi[2] = 0.f;
#pragma unroll
    for (int k = 0; k < 9; k++) xm[k] = (k % 4 == 0) ? 1.f : 0.f;
    if (dyn) {
      float* cf = SF(o_cfrc); float* ci = SF(o_cinert);
#pragma unroll
      for (int k = 0; k < 6; k++) cf[k] = 0.f;
#pragma unroll
      for (int k = 0; k < 10; k++) ci[k] = 0.f;
    }
  }
  // A: poses in the parent's frame
  for (int b = 1 + c.lane; b < m.nbody; b += G) body_local_pose<G>(mslot, c, b);
  c.tile.sync();
  // B: compose down the tree (children of the world are already in world coordinates)
  for (int L = 1; L < m.nlevel; L++) {
    for (int i = m.lvl_adr[L] + c.lane; i < m.lvl_adr[L + 1]; i += G) {
      const int b = m.lvl_body[i], pid = m.b_parent[b];
      float* xp = SF(o_xpos) + 3 * b; float* xm = SF(o_xmat) + 9 * b;
      const float* pR = SF(o_xmat) + 9 * pid;
      float v[3];
      mulmatvec3(v, pR, xp);
      add3(xp, v, SF(o_xpos) + 3 * pid);
      mulmat3(xm, pR, xm);
    }
    c.tile.sync();
  }
  // C: inertial frame origins, then cdof about the tree reference and cinert
  for (int b = 1 + c.lane; b < m.nbody; b += G) {
    float ip[3];
    mulmatvec3(ip, SF(o_xmat) + 9 * b, m.b_ipos + 3 * b);
    add3(SF(o_xipos) + 3 * b, ip, SF(o_xpos) + 3 * b);
  }
  c.tile.sync();
  float* cdof = SF(o_cdof);
  for (int j = c.lane; j < m.njnt; j += G) {
    const int b = m.j_body[j], pid = m.b_parent[b], da = m.j_dofadr[j], jt = m.j_type[j];
    const float* cref = SF(o_xipos) + 3 * m.b_root[b];
    if (jt == J_FREE) {
      const float* R = SF(o_xmat) + 9 * b;
      float off[3];
      sub3(off, cref, SF(o_xpos) + 3 * b);
#pragma unroll
      for (int k = 0; k < 3; k++) {
        float* t = cdof + 6 * (da + k);
        t[0] = t[1] = t[2] = 0.f; t[3] = (k == 0); t[4] = (k == 1); t[5] = (k == 2);
        float* r = cdof + 6 * (da + 3 + k);
        float ax[3] = {R[k], R[3 + k], R[6 + k]};
        cpy3(r, ax);
        cross3(r + 3, ax, off);
      }
    } else {
      const float* pR = SF(o_xmat) + 9 * pid;
      float* t = cdof + 6 * da;
      float ax[3];
      mulmatvec3(ax, pR, t);
      if (jt == J_SLIDE) { t[0] = t[1] = t[2] = 0.f; cpy3(t + 3, ax); }
      else {
        float anchor[3], off[3];
        mulmatvec3(anchor, pR, t + 3);
        add3(anchor, anchor, SF(o_xpos) + 3 * pid);
        sub3(off, cref, anchor);
        cpy3(t, ax);
        cross3(t + 3, ax, off);
      }
    }
  }
  if (!dyn) { c.tile.sync(); return; }
  for (int b = 1 + c.lane; b < m.nbody; b += G) {
    float off[3], mass = m.b_mass[b];
    const int slot = m.b_mass_slot[b];
    if (slot >= 0) mass = c.wpp(m)[slot];
    sub3(off, SF(o_xipos) + 3 * b, SF(o_xipos) + 3 * m.b_root[b]);
    float* ci = SF(o_cinert) + 10 * b;
    const float* R = SF(o_xmat) + 9 * b;
    if (m.b_sameframe[b]) inert_com(ci, m.b_inertia + 3 * b, R, off, mass);
    else {
      float Ri[9];
      mulmat3(Ri, R, m.b_imat + 9 * b);
      inert_com(ci, m.b_inertia + 3 * b, Ri, off, mass);
    }
  }
  c.tile.sync();
  // D: mj_comVel + mj_rne forward (flg_acc = 0) without a sweep down the tree. All cdof share their tree's reference
  // point, so a body's spatial velocity is the plain sum over its dof chain, and cdof_dot_i = (motion of the dofs that
  // precede i: host list d_pref) x cdof_i needs no parent result either: a lane per dof, then a lane per body.
  const float* qvel = SF(o_qvel);
  float* cdd = SF(o_cdofdot);
  for (int i = c.lane; i < m.nv; i += G) {
    float v[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, t[6];
    for (int k = m.d_prefadr[i]; k < m.d_prefadr[i + 1]; k++) {
      const int d = m.d_pref[k];
      const float w = qvel[d];
#pragma unroll
      for (int e = 0; e < 6; e++) v[e] += cdof[6 * d + e] * w;
    }
    cross_motion(t, v, cdof + 6 * i);
#pragma unroll
    for (int e = 0; e < 6; e++) cdd[6 * i + e] = t[e];
  }
  c.tile.sync();
  for (int b = 1 + c.lane; b < m.nbody; b += G) {
    float cv[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    float ca[6] = {0.f, 0.f, 0.f, -m.gravity[0], -m.gravity[1], -m.gravity[2]};
    for (int k = 0; k < m.b_nchain[b]; k++) {
      const int d = m.b_chain[b * KC + k];
      const float w = qvel[d];
#pragma unroll
      for (int e = 0; e < 6; e++) { cv[e] += cdof[6 * d + e] * w; ca[e] += cdd[6 * d + e] * w; }
    }
    const float* ci = SF(o_cinert) + 10 * b;
    float f[6], t[6], t1[6];
    mul_inert_vec(f, ci, ca);
    mul_inert_vec(t, ci, cv);
    cross_force(t1, cv, t);
    float* of = SF(o_cfrc) + 6 * b;
#pragma unroll
    for (int k = 0; k < 6; k++) of[k] = f[k] + t1[k];
  }
  c.tile.sync();
}

// a10.4 mj_crb + mj_rne backward + qfrc_bias, a lane per dof and no sweep up the tree: the lane adds the composite
// inertia and the force of its body's subtree itself (host list b_sub), then forms its mass-matrix row in MuJoCo's
// sparse dof_Madr layout (row i: i, parent(i), ...) and qfrc_bias_i = cdof_i . (subtree force).
template <int G, int V>
MYO_PHASE void phase_mass_bias(int mslot, Ctx<G, V> c) {
  MYO_M
  const float* cdof = SF(o_cdof); const float* cin = SF(o_cinert); const float* cf = SF(o_cfrc);
  float* M = SF(o_M); float* bias = SF(o_bias);
  for (int i = c.lane; i < m.nv; i += G) {
    const int body = m.d_body[i];
    const bool simple = m.d_simple[i] != 0;
    float crb[10], fs[6];
#pragma unroll
    for (int e = 0; e < 10; e++) crb[e] = 0.f;
#pragma unroll
    for (int e = 0; e < 6; e++) fs[e] = 0.f;
    for (int k = m.b_subadr[body]; k < m.b_subadr[body + 1]; k++) {
      const int b = m.b_sub[k];
      if (!simple) {
#pragma unroll
        for (int e = 0; e < 10; e++) crb[e] += cin[10 * b + e];
      }
#pragma unroll
      for (int e = 0; e < 6; e++) fs[e] += cf[6 * b + e];
    }
    float s = 0.f;
#pragma unroll
    for (int e = 0; e < 6; e++) s += cdof[6 * i + e] * fs[e];
    bias[i] = s;
    int adr = m.d_Madr[i];
    if (simple) {   // mj_crb: simple dofs take the stored dof_M0, off-diagonals stay zero
      M[adr] = m.d_M0[i];
      for (int q = 1; q <= m.d_depth[i]; q++) M[adr + q] = 0.f;
      continue;
    }
    float buf[6];
    mul_inert_vec(buf, crb, cdof + 6 * i);
    int j = i;
    bool first = true;
    while (j >= 0) {
      float v = 0.f;
#pragma unroll
      for (int e = 0; e < 6; e++) v += cdof[6 * j + e] * buf[e];
      if (first) { v += m.d_armature[i]; first = false; }
      M[adr++] = v;
      j = m.d_parent[j];
    }
  }
  c.tile.sync();
}

// y = M x (mj_mulM): a lane per row over the host-built list of the row's nonzeros (column | qM index << 8)
template <int G, int V>
MYO_PHASE void mul_M(int mslot, Ctx<G, V> c, int oM, int ox, int oy, bool sync = true) {
  MYO_M
  const float* M = SO(oM); const float* x = SO(ox); float* y = SO(oy);
  for (int i = c.lane; i < m.nv; i += G) {
    float v0 = 0.f, v1 = 0.f;
    int k = m.m_rowadr[i];
    const int k1 = m.m_rowadr[i + 1];
    for (; k + 1 < k1; k += 2) {
      const int e0 = m.m_row[k], e1 = m.m_row[k + 1];
      v0 += M[e0 >> 8] * x[e0 & 255];
      v1 += M[e1 >> 8] * x[e1 & 255];
    }
    if (k < k1) { const int e0 = m.m_row[k]; v0 += M[e0 >> 8] * x[e0 & 255]; }
    y[i] = v0 + v1;
  }
  if (sync) c.tile.sync();
}

// Helpers that take pointers to the caller's small arrays (points, frames, coefficient sets): as noinline functions those arrays
// live in local memory and every call stores and reloads them (round-2 profile: 240 local loads + 90 local stores per world
// and substep, 1.85 of 32 bytes used per sector). Inlined, they stay in registers.

// ------------------------------------------------------------------------------------------------
// a10.2 tendon length + moment arms (mj_tendon + mju_wrap), one lane per tendon.
MYO_DI void site_world(const DevModel& m, const float* s, const float* wp, int sid, float* out) {
  const int b = m.s_body[sid];
  const int slot = m.s_pos_slot[sid];
  float lp[3];
  if (slot >= 0) { lp[0] = wp[slot]; lp[1] = wp[slot + 1]; lp[2] = wp[slot + 2]; }
  else cpy3(lp, m.s_pos + 3 * sid);
  mulmatvec3(out, s + m.o_xmat + 9 * b, lp);
  add3(out, out, s + m.o_xpos + 3 * b);
}
MYO_DI bool seg_intersect(const float* p1, const float* p2, const float* p3, const float* p4) {
  const float det = (p4[1] - p3[1]) * (p2[0] - p1[0]) - (p4[0] - p3[0]) * (p2[1] - p1[1]);
  if (fabsf(det) < kMinVal) return false;
  const float a = ((p4[0] - p3[0]) * (p1[1] - p3[1]) - (p4[1] - p3[1]) * (p1[0] - p3[0])) / det;
  const float b = ((p2[0] - p1[0]) * (p1[1] - p3[1]) - (p2[1] - p1[1]) * (p1[0] - p3[0])) / det;
  return a >= 0.f && a <= 1.f && b >= 0.f && b <= 1.f;
}
// 2-D wrap around a circle (MuJoCo wrap_circle). Arc angle via atan2(|cross|, dot): same value as
// MuJoCo's acos(dot) but well conditioned in fp32 for small arcs.
MYO_DI float wrap_circle(float* pnt, const float* d, const float* sd, float rad) {
  const float sqlen0 = d[0] * d[0] + d[1] * d[1], sqlen1 = d[2] * d[2] + d[3] * d[3], sqrad = rad * rad;
  const float dif[2] = {d[2] - d[0], d[3] - d[1]};
  const float dd = dif[0] * dif[0] + dif[1] * dif[1];
  if (sqlen0 < sqrad || sqlen1 < sqrad || rad < kMinVal) return -1.f;
  if (dd < kMinVal) return -1.f;
  float a = clipf(-(dif[0] * d[0] + dif[1] * d[1]) / dd, 0.f, 1.f);
  const float tmp[2] = {a * dif[0] + d[0], a * dif[1] + d[1]};
  if (tmp[0] * tmp[0] + tmp[1] * tmp[1] > sqrad && (!sd || sd[0] * tmp[0] + sd[1] * tmp[1] >= 0.f)) return -1.f;
  const float sqrt0 = sqrtf(sqlen0 - sqrad), sqrt1 = sqrtf(sqlen1 - sqrad);
  float sol[2][4], good[2];
#pragma unroll
  for (int i = 0; i < 2; i++) {
    const float sgn = (i == 0) ? 1.f : -1.f;
    sol[i][0] = (d[0] * sqrad + sgn * rad * d[1] * sqrt0) / sqlen0;
    sol[i][1] = (d[1] * sqrad - sgn * rad * d[0] * sqrt0) / sqlen0;
    sol[i][2] = (d[2] * sqrad - sgn * rad * d[3] * sqrt1) / sqlen1;
    sol[i][3] = (d[3] * sqrad + sgn * rad * d[2] * sqrt1) / sqlen1;
    if (sd) {
      float t[2] = {sol[i][0] + sol[i][2], sol[i][1] + sol[i][3]};
      const float n = sqrtf(t[0] * t[0] + t[1] * t[1]);
      if (n < kMinVal) { t[0] = 1.f; t[1] = 0.f; } else { t[0] /= n; t[1] /= n; }
      good[i] = t[0] * sd[0] + t[1] * sd[1];
    } else {
      const float t[2] = {sol[i][0] - sol[i][2], sol[i][1] - sol[i][3]};
      good[i] = -(t[0] * t[0] + t[1] * t[1]);
    }
    if (seg_intersect(d, sol[i], d + 2, sol[i] + 2)) good[i] = -10000.f;
  }
  const int i = (good[0] > good[1]) ? 0 : 1;
  const float* sl = (i == 0) ? sol[0] : sol[1];
  pnt[0] = sl[0]; pnt[1] = sl[1]; pnt[2] = sl[2]; pnt[3] = sl[3];
  if (seg_intersect(d, pnt, d + 2, pnt + 2)) return -1.f;
  const float dt = pnt[0] * pnt[2] + pnt[1] * pnt[3];
  const float cr = pnt[1] * pnt[2] - pnt[0] * pnt[3];
  float angle = atan2f(fabsf(cr), dt);
  // a grazing contact has cr ~ 0 with a rounding-noise sign; the reflex branch (arc > pi) is only
  // taken when the sign is resolved, otherwise a zero-length arc would flip to a full 2*pi turn
  if (fabsf(cr) > 1e-5f * sqrad && ((cr > 0.f && i) || (cr < 0.f && !i))) angle = 2.f * kPi - angle;
  return rad * angle;
}
// returns curved length (>= 0) and two world points in wpnt[0..5]; -1 no wrap; -2 unsupported (inside wrap)
MYO_DI float wrap_geom(float* wpnt, const float* x0, const float* x1, const float* gpos, const float* gmat, float radius,
                       int type, const float* side) {
  float p0[3], p1[3], dif[3], axis0[3], axis1[3], normal[3];
  sub3(dif, x0, gpos); mulmatTvec3(p0, gmat, dif);
  sub3(dif, x1, gpos); mulmatTvec3(p1, gmat, dif);
  if (norm3(p0) < kMinVal || norm3(p1) < kMinVal) return -1.f;
  if (type == W_SPHERE) {
    cpy3(axis0, p0); normalize3(axis0);
    cross3(normal, p0, p1);
    if (norm3(normal) < kMinVal) {
      int im = 0;
      if (fabsf(axis0[1]) > fabsf(axis0[im])) im = 1;
      if (fabsf(axis0[2]) > fabsf(axis0[im])) im = 2;
      float a1[3] = {1.f, 1.f, 1.f};
      a1[im] = 0.f;
      cross3(normal, axis0, a1);
    }
    normalize3(normal);
    cross3(axis1, normal, axis0); normalize3(axis1);
  } else {
    axis0[0] = 1.f; axis0[1] = 0.f; axis0[2] = 0.f; axis1[0] = 0.f; axis1[1] = 1.f; axis1[2] = 0.f;
  }
  const float dd[4] = {dot3(p0, axis0), dot3(p0, axis1), dot3(p1, axis0), dot3(p1, axis1)};
  float sd[2];
  const float* sdp = nullptr;
  if (side) {
    float sv[3];
    sub3(dif, side, gpos); mulmatTvec3(sv, gmat, dif);
    const float in_norm = (type == W_SPHERE) ? norm3(sv) : sqrtf(sv[0] * sv[0] + sv[1] * sv[1]);
    if (in_norm < radius) return -2.f;
    sd[0] = dot3(sv, axis0); sd[1] = dot3(sv, axis1);
    const float n = sqrtf(sd[0] * sd[0] + sd[1] * sd[1]);
    if (n < kMinVal) { sd[0] = 1.f; sd[1] = 0.f; } else { sd[0] /= n; sd[1] /= n; }
    sd[0] *= radius; sd[1] *= radius;
    sdp = sd;
  }
  float pnt[4];
  float wlen = wrap_circle(pnt, dd, sdp, radius);
  if (wlen < 0.f) return -1.f;
  float res[6];
#pragma unroll
  for (int k = 0; k < 3; k++) {
    res[k] = axis0[k] * pnt[0] + axis1[k] * pnt[1];
    res[3 + k] = axis0[k] * pnt[2] + axis1[k] * pnt[3];
  }
  if (type == W_CYLINDER) {
    const float L0 = sqrtf((p0[0] - res[0]) * (p0[0] - res[0]) + (p0[1] - res[1]) * (p0[1] - res[1]));
    const float L1 = sqrtf((p1[0] - res[3]) * (p1[0] - res[3]) + (p1[1] - res[4]) * (p1[1] - res[4]));
    res[2] = p0[2] + (p1[2] - p0[2]) * L0 / (L0 + wlen + L1);
    res[5] = p0[2] + (p1[2] - p0[2]) * (L0 + wlen) / (L0 + wlen + L1);
    const float h = fabsf(res[5] - res[2]);
    wlen = sqrtf(wlen * wlen + h * h);
  }
  mulmatvec3(wpnt, gmat, res); add3(wpnt, wpnt, gpos);
  mulmatvec3(wpnt + 3, gmat, res + 3); add3(wpnt + 3, wpnt + 3, gpos);
  return wlen;
}
MYO_DI int common_prefix(const DevModel& m, int ba, int bb) {
  if (m.b_root[ba] != m.b_root[bb]) return 0;
  const int na = m.b_nchain[ba], nb = m.b_nchain[bb];
  int cp = 0;
  while (cp < na && cp < nb && m.b_chain[ba * KC + cp] == m.b_chain[bb * KC + cp]) cp++;
  return cp;
}
// Moment-arm contributions of the straight piece pa -> pb (points fixed to two bodies) to its tendon:
//   d|pb - pa| / dq_d = +-dir . (lin_d + ang_d x off) = +-(lin_d . dir + ang_d . (off x dir)),  cdof_d = (ang_d; lin_d)
// for the dofs on either body's chain past their common prefix (- on the pa side, + on the pb side). The dof list of the
// (body, body) pair is precomputed (myo_pack.cpp seg_list): header n | rootA << 8 | rootB << 20, entries
// dof | slot << 8 | end << 16, slot = position in the tendon's dof list = position in the segment's result row.
MYO_DI void segment_moment(int mslot, int soff, int list, const float* pa, const float* pb, float inv_div, float* out) {
  MYO_M
  if (list < 0) return;
  const float* s = MYO_SMEM_WORDS + soff;
  const int* L = m.seg_list + list;
  const int head = L[0], n = head & 255;
  float dir[3], oa[3], ob[3], ta[3], tb[3];
  sub3(dir, pb, pa);
  normalize3(dir);
  sub3(oa, pa, s + m.o_xipos + 3 * ((head >> 8) & 4095));
  sub3(ob, pb, s + m.o_xipos + 3 * ((head >> 20) & 4095));
  cross3(ta, oa, dir);
  cross3(tb, ob, dir);
  const float* cdof = s + m.o_cdof;
  auto term = [&](int e) {
    const float* cd = cdof + 6 * (e & 255);
    const bool end = (e >> 16) & 1;
    const float* t = end ? tb : ta;
    const float v = cd[0] * t[0] + cd[1] * t[1] + cd[2] * t[2] + cd[3] * dir[0] + cd[4] * dir[1] + cd[5] * dir[2];
    return end ? v * inv_div : -v * inv_div;
  };
  // two entries at a time, loads before stores: the entries of one list are distinct dofs, hence distinct slots of `out`
  int k = 1;
  for (; k + 1 <= n; k += 2) {
    const int e0 = L[k], e1 = L[k + 1];
    float* o0 = out + 1 + ((e0 >> 8) & 255);
    float* o1 = out + 1 + ((e1 >> 8) & 255);
    const float a0 = *o0, a1 = *o1;
    const float v0 = term(e0), v1 = term(e1);
    *o0 = a0 + v0;
    *o1 = a1 + v1;
  }
  if (k <= n) { const int e = L[k]; out[1 + ((e >> 8) & 255)] += term(e); }
}

// One lane per path segment (results to scratch: length and moment-arm slots), then one lane per tendon adds its
// segments in path order: ten_length, ten_J (KT slots over the tendon's dof list) and ten_velocity = J . qvel.
// The per-segment results live in words the Newton Hessian and the records of the constraint phases use later
// (myo_pack.cpp: o_seg).
template <int G, int V>
MYO_PHASE void phase_tendon(int mslot, Ctx<G, V> c, int* status) {
  MYO_M
  float* res = SF(o_seg);
  for (int sg = c.lane; sg < m.nseg; sg += G) {
    const int* rec = m.seg_rec + sg * SEG_WORDS;
    const int type = rec[0] >> 16, id0 = rec[1], id1 = rec[2], g = rec[3], side = rec[4];
    const float inv_div = m.seg_invdiv[sg];
    float* out = res + sg * SEG_OUT;
#pragma unroll
    for (int e = 0; e < SEG_OUT; e++) out[e] = 0.f;
    float x0[3], x1[3];
    site_world(m, c.sp(), c.wpp(m), id0, x0);
    site_world(m, c.sp(), c.wpp(m), id1, x1);
    float wlen = -1.f, wp2[6];
    if (g >= 0) {
      const int bw = m.g_body[g];
      float gpos[3], gmat[9];
      mulmatvec3(gpos, SF(o_xmat) + 9 * bw, m.g_pos + 3 * g);
      add3(gpos, gpos, SF(o_xpos) + 3 * bw);
      mulmat3(gmat, SF(o_xmat) + 9 * bw, m.g_mat + 9 * g);
      float sp[3];
      if (side >= 0) site_world(m, c.sp(), c.wpp(m), side, sp);
      float radius = m.g_size[3 * g];
      if (m.g_size_slot[g] >= 0) radius = c.wpp(m)[m.g_size_slot[g]];
      wlen = wrap_geom(wp2, x0, x1, gpos, gmat, radius, type, side >= 0 ? sp : nullptr);
      if (wlen == -2.f) { *status |= ST_UNSUPPORTED; wlen = -1.f; }
    }
    if (wlen < 0.f) {
      float d[3];
      sub3(d, x1, x0);
      out[0] = norm3(d) * inv_div;
      segment_moment(mslot, c.soff, rec[5], x0, x1, inv_div, out);
    } else {
      float d0[3], d1[3];
      sub3(d0, wp2, x0); sub3(d1, x1, wp2 + 3);
      out[0] = (norm3(d0) + wlen + norm3(d1)) * inv_div;
      segment_moment(mslot, c.soff, rec[6], x0, wp2, inv_div, out);
      segment_moment(mslot, c.soff, rec[7], wp2 + 3, x1, inv_div, out);
    }
  }
  c.tile.sync();
  const float* qvel = SF(o_qvel);
  for (int t = c.lane; t < m.ntendon; t += G) {
    const int ntd = m.t_ndof[t];
    const int* tdof = m.t_dof + t * KT;
    float J[KT];
#pragma unroll
    for (int e = 0; e < KT; e++) J[e] = 0.f;
    float len = 0.f;
    for (int k = m.t_segadr[t]; k < m.t_segadr[t + 1]; k++) {
      const float* r = res + m.t_seg[k] * SEG_OUT;
      len += r[0];
#pragma unroll
      for (int e = 0; e < KT; e++) J[e] += r[1 + e];
    }
    float vel = 0.f;
    float* Jo = SF(o_tenJ) + t * KT;
#pragma unroll
    for (int e = 0; e < KT; e++) { Jo[e] = J[e]; if (e < ntd) vel += J[e] * qvel[tdof[e]]; }
    SF(o_tenL)[t] = len;
    SF(o_tenV)[t] = vel;
  }
  c.tile.sync();
}

// ------------------------------------------------------------------------------------------------
// a10.7 muscle model (mju_muscleGain / Bias / Dynamics), passive forces, actuator forces
MYO_DI float muscle_FL(float L, float lmin, float lmax) {
  if (L < lmin || L > lmax) return 0.f;
  const float a = 0.5f * (lmin + 1.f), b = 0.5f * (1.f + lmax);
  float x;
  if (L <= a) { x = (L - lmin) / fmaxf(kMinVal, a - lmin); return 0.5f * x * x; }
  if (L <= 1.f) { x = (1.f - L) / fmaxf(kMinVal, 1.f - a); return 1.f - 0.5f * x * x; }
  if (L <= b) { x = (L - 1.f) / fmaxf(kMinVal, b - 1.f); return 1.f - 0.5f * x * x; }
  x = (lmax - L) / fmaxf(kMinVal, lmax - b);
  return 0.5f * x * x;
}
template <int G, int V>
MYO_PHASE void phase_actuation(int mslot, Ctx<G, V> c) {
  MYO_M
  const float* ctrl = SF(o_ctrl); const float* act = SF(o_act);
  for (int i = c.lane; i < m.nu; i += G) {
    const int t = m.a_tendon[i];
    const float gear = GT(a_gear)[i];
    const float len = gear * SF(o_tenL)[t], vel = gear * SF(o_tenV)[t];
    float u = ctrl[i];
    if (m.a_ctrllimited[i]) u = clipf(u, GT(a_ctrlrange)[2 * i], GT(a_ctrlrange)[2 * i + 1]);
    const int ai = i - (m.nu - m.na);
    const float* dp = GT(a_dynprm) + 3 * i;
    const float* gp = GT(a_gainprm) + 9 * i;
    const float* bp = GT(a_biasprm) + 9 * i;
    const float lr0 = GT(a_lengthrange)[2 * i], lr1 = GT(a_lengthrange)[2 * i + 1], acc0 = GT(a_acc0)[i];
    const int dyn = m.a_dyntype[i];
    float a_cur = (ai >= 0 && dyn != 0) ? act[ai] : 0.f;
    if (dyn == 3) {          // muscle
      const float uc = clipf(u, 0.f, 1.f), ac = clipf(a_cur, 0.f, 1.f);
      const float tau = (uc > a_cur) ? dp[0] * (0.5f + 1.5f * ac) : dp[1] / (0.5f + 1.5f * ac);
      SF(o_actdot)[ai] = (uc - a_cur) / fmaxf(kMinVal, tau);
    } else if (dyn == 1) SF(o_actdot)[ai] = u;                                   // integrator
    else if (dyn == 2) SF(o_actdot)[ai] = (u - a_cur) / fmaxf(kMinVal, dp[0]);     // filter
    float gain, bias = 0.f;
    if (m.a_gaintype[i] == 1) {
      float F0 = gp[2];
      if (F0 < 0.f) F0 = gp[3] / fmaxf(kMinVal, acc0);
      const float L0 = (lr1 - lr0) / fmaxf(kMinVal, gp[1] - gp[0]);
      const float L = gp[0] + (len - lr0) / fmaxf(kMinVal, L0);
      const float Vn = vel / fmaxf(kMinVal, L0 * gp[6]);
      const float FL = muscle_FL(L, gp[4], gp[5]);
      const float y = gp[8] - 1.f;
      float FV;
      if (Vn <= -1.f) FV = 0.f;
      else if (Vn <= 0.f) FV = (Vn + 1.f) * (Vn + 1.f);
      else if (Vn <= y) FV = gp[8] - (y - Vn) * (y - Vn) / fmaxf(kMinVal, y);
      else FV = gp[8];
      gain = -F0 * FL * FV;
    } else gain = gp[0];
    if (m.a_biastype[i] == 1) bias = bp[0] + bp[1] * len + bp[2] * vel;
    else if (m.a_biastype[i] == 2) {
      float F0 = bp[2];
      if (F0 < 0.f) F0 = bp[3] / fmaxf(kMinVal, acc0);
      const float L0 = (lr1 - lr0) / fmaxf(kMinVal, bp[1] - bp[0]);
      const float L = bp[0] + (len - lr0) / fmaxf(kMinVal, L0);
      const float b = 0.5f * (1.f + bp[5]);
      if (L <= 1.f) bias = 0.f;
      else if (L <= b) { const float x = (L - 1.f) / fmaxf(kMinVal, b - 1.f); bias = -F0 * bp[7] * 0.5f * x * x; }
      else { const float x = (L - b) / fmaxf(kMinVal, b - 1.f); bias = -F0 * bp[7] * (0.5f + x); }
    }
    float force = (dyn == 0 ? gain * u : gain * a_cur) + bias;
    if (m.a_forcelimited[i]) force = clipf(force, GT(a_forcerange)[2 * i], GT(a_forcerange)[2 * i + 1]);
    SF(o_actF)[i] = force;
  }
  c.tile.sync();
  // qfrc_actuator = moment' * force and mj_passive, gathered per dof in a fixed order
  const float* qpos = SF(o_qpos); const float* qvel = SF(o_qvel);
  for (int d = c.lane; d < m.nv; d += G) {
    float s = 0.f;
    for (int k = m.d_actadr[d]; k < m.d_actadr[d + 1]; k++) {
      const int code = m.d_actlist[k];
      const int a = code >> 8, slot = code & 255;
      s += GT(a_gear)[a] * SF(o_tenJ)[m.a_tendon[a] * KT + slot] * SF(o_actF)[a];
    }
    SF(o_qact)[d] = s;
    float p = -m.d_damping[d] * qvel[d];
    if (m.any_joint_spring) {
      const int j = m.d_jnt[d];
      const int jt = m.j_type[j];
      if ((jt == J_HINGE || jt == J_SLIDE) && m.j_stiffness[j] != 0.f) {
        const int qa = m.j_qposadr[j];
        p -= m.j_stiffness[j] * (qpos[qa] - m.j_qpos_spring[j]);
      }
    }
    if (m.any_tendon_passive) {
      for (int t = 0; t < m.ntendon; t++) {
        const float k = m.t_stiffness[t], bd = m.t_damping[t];
        if (k == 0.f && bd == 0.f) continue;
        const float frc = -k * (SF(o_tenL)[t] - m.t_lengthspring[t]) - bd * SF(o_tenV)[t];
        for (int e = 0; e < m.t_ndof[t]; e++) if (m.t_dof[t * KT + e] == d) p += SF(o_tenJ)[t * KT + e] * frc;
      }
    }
    SF(o_passive)[d] = p;
    SF(o_smooth)[d] = p - SF(o_bias)[d] + s;
    SF(o_qaccs)[d] = SF(o_smooth)[d];
  }
  c.tile.sync();
}

// ------------------------------------------------------------------------------------------------
// a10.5 collision: static candidate pair list, bounding-sphere cull with the *model's* rbound (stale
// after size randomisation, as in the reference), primitive narrow phase with per-world sizes.
MYO_DI void geom_world_pos(const DevModel& m, const float* s, int g, float* out) {
  const int b = m.g_body[g];
  mulmatvec3(out, s + m.o_xmat + 9 * b, m.g_pos + 3 * g);
  add3(out, out, s + m.o_xpos + 3 * b);
}
MYO_DI void geom_world_zaxis(const DevModel& m, const float* s, int g, float* out) {
  const float lz[3] = {m.g_mat[9 * g + 2], m.g_mat[9 * g + 5], m.g_mat[9 * g + 8]};
  mulmatvec3(out, s + m.o_xmat + 9 * m.g_body[g], lz);
}
MYO_DI void make_frame(float* f) {
  normalize3(f);
  f[3] = 0.f; f[4] = 0.f; f[5] = 0.f;
  if (f[1] < 0.5f && f[1] > -0.5f) f[4] = 1.f; else f[5] = 1.f;
  const float t = dot3(f, f + 3);
  f[3] -= t * f[0]; f[4] -= t * f[1]; f[5] -= t * f[2];
  normalize3(f + 3);
  cross3(f + 6, f, f + 3);
}
MYO_DI bool sphere_sphere(float margin, const float* p1, float r1, const float* p2, float r2, float* dist, float* pos, float* nrm) {
  float dif[3];
  sub3(dif, p2, p1);
  const float cd2 = dot3(dif, dif), mind = margin + r1 + r2;
  if (cd2 > mind * mind) return false;
  const float n = normalize3(dif);
  *dist = n - r1 - r2;
  cpy3(nrm, dif);
  const float k = r1 + 0.5f * (*dist);
  pos[0] = p1[0] + dif[0] * k; pos[1] = p1[1] + dif[1] * k; pos[2] = p1[2] + dif[2] * k;
  return true;
}

// ---- capsule - box: own closest-point collider (NOT MuJoCo's mjc_CapsuleBox; see oracle/myo_oracle.c capsule_box, the same
// algorithm in fp64). Capsule core segment p(t) = c + t d, |t| <= h, in the box frame; f(t) = sum_i max(0, |c_i + t d_i| - s_i)^2
// is convex piecewise quadratic: walk the sorted breakpoints of its piecewise-linear derivative.
MYO_DI float seg_box_dfdt(const float* c, const float* d, const float* s, float t) {
  float g = 0.f;
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const float x = c[i] + t * d[i], e = fabsf(x) - s[i];
    if (e > 0.f) g += 2.f * e * (x > 0.f ? d[i] : -d[i]);
  }
  return g;
}
MYO_DI float seg_box_closest_t(const float* c, const float* d, float h, const float* s) {
  float bp[8];
  int nb = 0;
  bp[nb++] = -h;
#pragma unroll
  for (int i = 0; i < 3; i++)
    if (fabsf(d[i]) > 1e-12f) {
#pragma unroll
      for (int sg = -1; sg <= 1; sg += 2) {
        const float t = ((float)sg * s[i] - c[i]) / d[i];
        if (t > -h && t < h) bp[nb++] = t;
      }
    }
  bp[nb++] = h;
  for (int i = 1; i < nb; i++) { const float v = bp[i]; int j = i - 1; while (j >= 0 && bp[j] > v) { bp[j + 1] = bp[j]; j--; } bp[j + 1] = v; }
  float g[8];
  int lo = -1, hi = nb;
  for (int k = 0; k < nb; k++) g[k] = seg_box_dfdt(c, d, s, bp[k]);
  for (int k = 0; k < nb; k++) if (g[k] < 0.f) lo = k;
  for (int k = nb - 1; k >= 0; k--) if (g[k] > 0.f) hi = k;
  if (hi == 0) return bp[0];
  if (lo == nb - 1) return bp[nb - 1];
  if (hi == lo + 1) return bp[lo] + (bp[hi] - bp[lo]) * (-g[lo]) / (g[hi] - g[lo]);
  return 0.5f * (bp[lo + 1] + bp[hi - 1]);
}
// one contact between the capsule's point p (box frame) and the box: dist, position and normal (capsule -> box) in the box frame
MYO_DI bool capsule_box_point(const float* p, const float* s, float r, float margin, float* dist, float* pos_b, float* nrm_b) {
  float q[3], f = 0.f;
#pragma unroll
  for (int i = 0; i < 3; i++) { q[i] = clipf(p[i], -s[i], s[i]); f += (p[i] - q[i]) * (p[i] - q[i]); }
  const float dd = sqrtf(f);
  if (dd > r + margin) return false;
  if (dd > 1e-10f) {
#pragma unroll
    for (int i = 0; i < 3; i++) nrm_b[i] = (q[i] - p[i]) / dd;
    *dist = dd - r;
  } else {      // core segment inside the box: leave through the nearest face
    int ax = 0;
    float best = 3.0e38f;
#pragma unroll
    for (int i = 0; i < 3; i++) { const float dep = s[i] - fabsf(p[i]); if (dep < best) { best = dep; ax = i; } }
    nrm_b[0] = nrm_b[1] = nrm_b[2] = 0.f;
    nrm_b[ax] = p[ax] > 0.f ? -1.f : 1.f;
    *dist = -best - r;
  }
#pragma unroll
  for (int i = 0; i < 3; i++) pos_b[i] = p[i] + nrm_b[i] * (r + 0.5f * (*dist));
  return true;
}
// contact number `sub` (0 or 1) of capsule (pc, axis, r, h) vs box (pb, Rb, s): both end points within reach -> one contact per end
// point, else a single contact at the closest point of the core segment
MYO_PHASE bool capsule_box(int sub, float margin, const float* pc, const float* axis, float r, float h, const float* pb, const float* Rb,
                            const float* s, float* dist, float* pos, float* nrm) {
  float dif[3], c[3], d[3];
  sub3(dif, pc, pb); mulmatTvec3(c, Rb, dif); mulmatTvec3(d, Rb, axis);
  // conservative early out (never drops a contact): the segment's extent along each box axis against the face plus reach
#pragma unroll
  for (int i = 0; i < 3; i++) if (fabsf(c[i]) - fabsf(d[i]) * h > s[i] + r + margin) return false;
  float pe[2][3], de[2], pb2[2][3], nb2[2][3];
  bool he[2];
#pragma unroll
  for (int e = 0; e < 2; e++) {
    const float t = e ? h : -h;
#pragma unroll
    for (int i = 0; i < 3; i++) pe[e][i] = c[i] + t * d[i];
    he[e] = capsule_box_point(pe[e], s, r, margin, &de[e], pb2[e], nb2[e]);
  }
  float posb[3], nrmb[3];
  if (he[0] && he[1]) {
    *dist = de[sub];
    cpy3(posb, pb2[sub]); cpy3(nrmb, nb2[sub]);
  } else {
    if (sub) return false;
    const float t = seg_box_closest_t(c, d, h, s);
    float p[3] = {c[0] + t * d[0], c[1] + t * d[1], c[2] + t * d[2]};
    if (!capsule_box_point(p, s, r, margin, dist, posb, nrmb)) return false;
  }
  mulmatvec3(pos, Rb, posb); add3(pos, pos, pb);
  mulmatvec3(nrm, Rb, nrmb);
  return true;
}

template <int G, int V>
MYO_PHASE void phase_collision(int mslot, Ctx<G, V> c, int* status) {
  MYO_M
  int* misc = SI(o_misc);
  int ncon = 0;
  for (int base = 0; base < m.npair; base += G) {
    const int p = base + c.lane;
    bool hit = false;
    float dist = 0.f, pos[3] = {0, 0, 0}, nrm[3] = {1, 0, 0};
    int g1 = 0, g2 = 0;
    if (p < m.npair) {
      g1 = m.p_g1[p]; g2 = m.p_g2[p];
      const float margin = fmaxf(m.g_margin[g1], m.g_margin[g2]);
      float p1[3], p2[3];
      geom_world_pos(m, c.sp(), g1, p1);
      geom_world_pos(m, c.sp(), g2, p2);
      const float rb1 = m.g_rbound[g1], rb2 = m.g_rbound[g2];
      bool pass = true;
      const int t1 = m.g_type[g1], t2 = m.g_type[g2];
      float z1[3] = {0.f, 0.f, 1.f};
      if (rb1 > 0.f && rb2 > 0.f) {
        float d[3];
        sub3(d, p1, p2);
        const float bound = rb1 + rb2 + margin;
        pass = dot3(d, d) <= bound * bound;
      } else if (t1 == G_PLANE && rb2 > 0.f) {
        geom_world_zaxis(m, c.sp(), g1, z1);
        float d[3];
        sub3(d, p2, p1);
        pass = dot3(d, z1) <= margin + rb2;
      }
      if (pass) {
        if (!m.p_supported[p]) *status |= ST_UNSUPPORTED;
        else {
          float s1 = m.g_size[3 * g1], s2 = m.g_size[3 * g2];
          if (m.g_size_slot[g1] >= 0) s1 = c.wpp(m)[m.g_size_slot[g1]];
          if (m.g_size_slot[g2] >= 0) s2 = c.wpp(m)[m.g_size_slot[g2]];
          if (t1 == G_SPHERE && t2 == G_SPHERE) hit = sphere_sphere(margin, p1, s1, p2, s2, &dist, pos, nrm);
          else if (t1 == G_CAPSULE && t2 == G_BOX) {
            float ax[3], Rb[9], sz[3];
            geom_world_zaxis(m, c.sp(), g1, ax);
            mulmat3(Rb, SF(o_xmat) + 9 * m.g_body[g2], m.g_mat + 9 * g2);
            float half = m.g_size[3 * g1 + 1];
            if (m.g_size_slot[g1] >= 0) half = c.wpp(m)[m.g_size_slot[g1] + 1];
#pragma unroll
            for (int e = 0; e < 3; e++) sz[e] = (m.g_size_slot[g2] >= 0) ? c.wpp(m)[m.g_size_slot[g2] + e] : m.g_size[3 * g2 + e];
            // (own output variables: handing &dist / pos / nrm to the noinline collider would park them in local memory for
            // every pair type)
            float bd, bp3[3], bn3[3];
            hit = capsule_box(m.p_supported[p] - 1, margin, p1, ax, s1, half, p2, Rb, sz, &bd, bp3, bn3);
            if (hit) { dist = bd; cpy3(pos, bp3); cpy3(nrm, bn3); }
          }
          else if (t1 == G_SPHERE && t2 == G_CAPSULE) {
            float ax[3], v[3];
            geom_world_zaxis(m, c.sp(), g2, ax);
            sub3(v, p1, p2);
            float half = m.g_size[3 * g2 + 1];
            if (m.g_size_slot[g2] >= 0) half = c.wpp(m)[m.g_size_slot[g2] + 1];
            const float x = clipf(dot3(ax, v), -half, half);
            v[0] = p2[0] + ax[0] * x; v[1] = p2[1] + ax[1] * x; v[2] = p2[2] + ax[2] * x;
            hit = sphere_sphere(margin, p1, s1, v, s2, &dist, pos, nrm);
          } else {  // plane - sphere
            float d[3];
            sub3(d, p2, p1);
            const float cd = dot3(d, z1);
            if (cd <= margin + s2) {
              hit = true;
              dist = cd - s2;
              cpy3(nrm, z1);
              const float k = -0.5f * dist - s2;
              pos[0] = p2[0] + z1[0] * k; pos[1] = p2[1] + z1[1] * k; pos[2] = p2[2] + z1[2] * k;
            }
          }
          if (hit && dist >= margin) hit = false;
        }
      }
    }
    const unsigned ball = c.tile.ballot(hit);
    if (hit) {
      const int slot = ncon + __popc(ball & ((1u << c.lane) - 1u));
      if (slot < m.ncon_max) {
        float* cr = SF(o_con) + slot * CON_WORDS;
        int* ci = reinterpret_cast<int*>(cr);
        ci[C_G1] = g1; ci[C_G2] = g2;
        cr[C_DIST] = dist;
        cpy3(cr + C_POS, pos);
        cpy3(cr + C_FRAME, nrm);
      } else *status |= ST_CON_OVERFLOW;
    }
    ncon += __popc(ball);
  }
  if (ncon > m.ncon_max) ncon = m.ncon_max;
  if (c.lane == 0) misc[MI_NCON] = ncon;
  c.tile.sync();
}

// impedance, regularisation and reference-acceleration coefficients of one row (mj_makeImpedance)
MYO_DI void row_params(int mslot, const float* solref, const float* solimp, float pos, float margin, float diag,
                   float* R, float* K, float* B, float* imp) {
  MYO_M
  const float s0 = clipf(solimp[0], 0.0001f, 0.9999f), s1 = clipf(solimp[1], 0.0001f, 0.9999f);
  const float s2 = fmaxf(0.f, solimp[2]), s3 = clipf(solimp[3], 0.0001f, 0.9999f), s4 = fmaxf(1.f, solimp[4]);
  float im;
  if (s0 == s1 || s2 <= kMinVal) im = 0.5f * (s0 + s1);
  else {
    const float x = fabsf((pos - margin) / s2);
    if (x >= 1.f) im = s1;
    else if (x <= 0.f) im = s0;
    else {
      float y;
      if (s4 == 1.f) y = x;
      else if (x <= s3) y = (s4 == 2.f) ? x * x / s3 : powf(x, s4) / powf(s3, s4 - 1.f);
      else y = (s4 == 2.f) ? 1.f - (1.f - x) * (1.f - x) / (1.f - s3) : 1.f - powf(1.f - x, s4) / powf(1.f - s3, s4 - 1.f);
      im = s0 + y * (s1 - s0);
    }
  }
  *imp = im;
  *R = fmaxf(kMinVal, (1.f - im) * diag / im);
  if (solref[0] > 0.f) {
    const float tc = fmaxf(solref[0], 2.f * m.timestep), dr = solref[1];
    *K = 1.f / fmaxf(kMinVal, s1 * s1 * tc * tc * dr * dr);
    *B = 2.f / fmaxf(kMinVal, s1 * tc);
  } else {
    *K = -solref[0] / fmaxf(kMinVal, s1 * s1);
    *B = -solref[1] / fmaxf(kMinVal, s1);
  }
}

// a10.6 constraint assembly. Limits first (joints then tendons, MuJoCo order), then contacts with
// 2*(condim-1) pyramid rows each. Rows keep (D, aref); Jacobians stay factored per block:
// a limit has one basis vector over <= KT dofs, a contact has (normal, tangent1, tangent2) over
// the <= KS dofs in chain(body1) xor chain(body2).
template <int G, int V>
MYO_PHASE void phase_constraints(int mslot, Ctx<G, V> c, int* status) {
  MYO_M
  int* misc = SI(o_misc);
  const float* qpos = SF(o_qpos); const float* qvel = SF(o_qvel);
  int nlim = 0;
  // joint limits: row order joint-major, lower side before upper side
  for (int base = 0; base < m.njnt; base += G) {
    const int j = base + c.lane;
    bool lo = false, hi = false;
    float dlo = 0.f, dhi = 0.f, margin = 0.f;
    if (j < m.njnt && m.j_limited[j] && (m.j_type[j] == J_HINGE || m.j_type[j] == J_SLIDE)) {
      const float v = qpos[m.j_qposadr[j]];
      margin = m.j_margin[j];
      dlo = v - m.j_range[2 * j]; dhi = m.j_range[2 * j + 1] - v;
      lo = dlo < margin; hi = dhi < margin;
    }
    const unsigned blo = c.tile.ballot(lo), bhi = c.tile.ballot(hi);
    const unsigned lt = (1u << c.lane) - 1u;
    int slot = nlim + __popc(blo & lt) + __popc(bhi & lt);
    if (lo) {
      if (slot < m.nlim_max) {
        float* r = SF(o_lim) + slot * LIM_WORDS; int* ri = reinterpret_cast<int*>(r);
        ri[L_KIND] = EFC_LIMIT_JOINT; ri[L_ID] = j; ri[L_NSUP] = 1; r[L_POS] = dlo; r[L_MARGIN] = margin;
        r[L_SIGN] = 1.f; ri[L_IOFF] = m.j_dofadr.off + j; ri[L_JOFF] = m.o_misc + MI_ONE;
      } else *status |= ST_EFC_OVERFLOW;
      slot++;
    }
    if (hi) {
      if (slot < m.nlim_max) {
        float* r = SF(o_lim) + slot * LIM_WORDS; int* ri = reinterpret_cast<int*>(r);
        ri[L_KIND] = EFC_LIMIT_JOINT; ri[L_ID] = j; ri[L_NSUP] = 1; r[L_POS] = dhi; r[L_MARGIN] = margin;
        r[L_SIGN] = -1.f; ri[L_IOFF] = m.j_dofadr.off + j; ri[L_JOFF] = m.o_misc + MI_ONE;
      } else *status |= ST_EFC_OVERFLOW;
    }
    nlim += __popc(blo) + __popc(bhi);
  }
  for (int base = 0; base < m.ntendon; base += G) {
    const int t = base + c.lane;
    bool lo = false, hi = false;
    float dlo = 0.f, dhi = 0.f, margin = 0.f;
    if (t < m.ntendon && m.t_limited[t]) {
      const float v = SF(o_tenL)[t];
      margin = m.t_margin[t];
      dlo = v - m.t_range[2 * t]; dhi = m.t_range[2 * t + 1] - v;
      lo = dlo < margin; hi = dhi < margin;
    }
    const unsigned blo = c.tile.ballot(lo), bhi = c.tile.ballot(hi);
    const unsigned lt = (1u << c.lane) - 1u;
    int slot = nlim + __popc(blo & lt) + __popc(bhi & lt);
    for (int side = 0; side < 2; side++) {
      if (!(side ? hi : lo)) continue;
      if (slot < m.nlim_max) {
        float* r = SF(o_lim) + slot * LIM_WORDS; int* ri = reinterpret_cast<int*>(r);
        ri[L_KIND] = EFC_LIMIT_TENDON; ri[L_ID] = t; ri[L_NSUP] = m.t_ndof[t];
        r[L_POS] = side ? dhi : dlo; r[L_MARGIN] = margin;
        r[L_SIGN] = side ? -1.f : 1.f; ri[L_IOFF] = m.t_dof.off + t * KT; ri[L_JOFF] = m.o_tenJ + t * KT;
      } else *status |= ST_EFC_OVERFLOW;
      slot++;
    }
    nlim += __popc(blo) + __popc(bhi);
  }
  if (nlim > m.nlim_max) nlim = m.nlim_max;
  const int ncon = misc[MI_NCON];
  c.tile.sync();

  // limit rows: parameters + reference acceleration
  float* rows = SF(o_row);
  for (int r = c.lane; r < nlim; r += G) {
    const float* lr = SF(o_lim) + r * LIM_WORDS; const int* li = reinterpret_cast<const int*>(lr);
    const int id = li[L_ID];
    float R, K, B, imp, vel = 0.f;
    if (li[L_KIND] == EFC_LIMIT_JOINT) {
      row_params(mslot, m.j_solref + 2 * id, m.j_solimp + 5 * id, lr[L_POS], lr[L_MARGIN], m.d_invweight0[m.j_dofadr[id]], &R, &K, &B, &imp);
      vel = lr[L_SIGN] * qvel[m.j_dofadr[id]];
    } else {
      row_params(mslot, m.t_solref + 2 * id, m.t_solimp + 5 * id, lr[L_POS], lr[L_MARGIN], m.t_invweight0[id], &R, &K, &B, &imp);
      for (int e = 0; e < li[L_NSUP]; e++) vel += lim_J(c.sp(), lr, li, e) * qvel[lim_idx(li, e)];
    }
    float* row = rows + r * ROW_WORDS;
    row[R_D] = 1.f / R;
    row[R_AREF] = -B * vel - K * imp * (lr[L_POS] - lr[L_MARGIN]);
  }
  // contacts: mixing (mj_contactParam), frame, support, rows. A lane per contact; the row index comes from an exclusive
  // scan of the row counts inside the tile (fixed contact order), then the same lane fills its rows.
  int nrow_con = 0, nrow_valid = 0;
  for (int base = 0; base < ncon; base += G) {
    const int k = base + c.lane;
    int nr = 0, dim = 0;
    float mu = 0.f, D = 0.f, Bc = 0.f, ref = 0.f, vn = 0.f, vt1 = 0.f, vt2 = 0.f;
    if (k < ncon) {
      float* cr = SF(o_con) + k * CON_WORDS; int* ci = reinterpret_cast<int*>(cr);
      const int g1 = ci[C_G1], g2 = ci[C_G2];
      float fri[3], solref[2], solimp[5];
      float f1[3], f2[3];
#pragma unroll
      for (int e = 0; e < 3; e++) {
        f1[e] = (m.g_fri_slot[g1] >= 0) ? c.wpp(m)[m.g_fri_slot[g1] + e] : m.g_friction[3 * g1 + e];
        f2[e] = (m.g_fri_slot[g2] >= 0) ? c.wpp(m)[m.g_fri_slot[g2] + e] : m.g_friction[3 * g2 + e];
      }
      const int pr1 = m.g_priority[g1], pr2 = m.g_priority[g2];
      if (pr1 != pr2) {
        const int g = pr1 > pr2 ? g1 : g2;
        dim = m.g_condim[g];
        solref[0] = m.g_solref[2 * g]; solref[1] = m.g_solref[2 * g + 1];
#pragma unroll
        for (int e = 0; e < 5; e++) solimp[e] = m.g_solimp[5 * g + e];
#pragma unroll
        for (int e = 0; e < 3; e++) fri[e] = pr1 > pr2 ? f1[e] : f2[e];
      } else {
        dim = max(m.g_condim[g1], m.g_condim[g2]);
        const float sm1 = m.g_solmix[g1], sm2 = m.g_solmix[g2];
        float mix;
        if (sm1 >= kMinVal && sm2 >= kMinVal) mix = sm1 / (sm1 + sm2);
        else if (sm1 < kMinVal && sm2 < kMinVal) mix = 0.5f;
        else mix = (sm1 < kMinVal) ? 0.f : 1.f;
        const float* r1 = m.g_solref + 2 * g1; const float* r2 = m.g_solref + 2 * g2;
        if (r1[0] > 0.f && r2[0] > 0.f) { solref[0] = mix * r1[0] + (1.f - mix) * r2[0]; solref[1] = mix * r1[1] + (1.f - mix) * r2[1]; }
        else { solref[0] = fminf(r1[0], r2[0]); solref[1] = fminf(r1[1], r2[1]); }
#pragma unroll
        for (int e = 0; e < 5; e++) solimp[e] = mix * m.g_solimp[5 * g1 + e] + (1.f - mix) * m.g_solimp[5 * g2 + e];
#pragma unroll
        for (int e = 0; e < 3; e++) fri[e] = fmaxf(f1[e], f2[e]);
      }
      const float margin = fmaxf(m.g_margin[g1], m.g_margin[g2]) - fmaxf(m.g_gap[g1], m.g_gap[g2]);
      mu = fri[0];
      ci[C_DIM] = dim; cr[C_MARGIN] = margin; cr[C_MU] = mu;
      float fr[9];
      cpy3(fr, cr + C_FRAME);
      make_frame(fr);
#pragma unroll
      for (int e = 0; e < 9; e++) cr[C_FRAME + e] = fr[e];
      const int ba = m.g_body[g1], bb = m.g_body[g2];
      ci[C_BA] = ba; ci[C_BB] = bb;
      const int cp = common_prefix(m, ba, bb);
      const int na = max(m.b_nchain[ba] - cp, 0), nb = max(m.b_nchain[bb] - cp, 0);
      int ns = na + nb;
      if (ns > KS || cp > 255) { *status |= ST_UNSUPPORTED; ns = 0; }
      ci[C_CP] = cp | (na << 8);
      ci[C_NSUP] = ns;
      // relative velocity of the contact point in the contact frame
      for (int e = 0; e < ns; e++) {
        float jn, jt1, jt2;
        const int dof = contact_entry(m, c.sp(), cr, ci, e, &jn, &jt1, &jt2);
        const float w = qvel[dof];
        vn += jn * w; vt1 += jt1 * w; vt2 += jt2 * w;
      }
      const float dist = cr[C_DIST];
      if (dist < margin) {
        if (dim == 1) nr = 1;
        else if (dim == 3) nr = 4;
        else *status |= ST_UNSUPPORTED;
      }
      const float tran = m.b_invweight0[2 * ba] + m.b_invweight0[2 * bb];
      float R, K, imp;
      // diagApprox of the first row: tran + mu^2 * tran (pyramidal) or tran (frictionless)
      row_params(mslot, solref, solimp, dist, margin, dim == 1 ? tran : tran + mu * mu * tran, &R, &K, &Bc, &imp);
      if (dim == 3) { const float mu_r = mu * m.inv_sqrt_impratio; R = 2.f * mu_r * mu_r * R; }
      D = 1.f / R; ref = -K * imp * (dist - margin);
    }
    // exclusive scan of row counts inside the tile (fixed contact order)
    int incl = nr;
#pragma unroll
    for (int o = 1; o < G; o <<= 1) { const int t = c.tile.shfl_up(incl, o); if (c.lane >= o) incl += t; }
    const int excl = incl - nr;
    const int total = c.tile.shfl(incl, G - 1);
    if (k < ncon) {
      int* ci = SI(o_con) + k * CON_WORDS;
      const int row0 = nlim + nrow_con + excl;
      if (nr && row0 + nr > m.nefc_max) { *status |= ST_EFC_OVERFLOW; nr = 0; }
      ci[C_ROW0] = nr ? row0 : -1;
      for (int q = 0; q < nr; q++) {
        float vel = vn;
        if (dim == 3) vel += ((q & 1) ? -mu : mu) * ((q < 2) ? vt1 : vt2);
        float* row = rows + (row0 + q) * ROW_WORDS;
        row[R_D] = D;
        row[R_AREF] = -Bc * vel + ref;
      }
    }
    int valid = nr;   // rows are dropped only at the tail, so valid rows stay contiguous
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) valid += c.tile.shfl_xor(valid, o);
    nrow_valid += valid;
    nrow_con += total;
  }
  const int nefc = nlim + nrow_valid;
  if (c.lane == 0) { misc[MI_NLIM] = nlim; misc[MI_NEFC] = nefc; }
  c.tile.sync();
}

// ------------------------------------------------------------------------------------------------
// row helper: J_r . x for every row -> rows[r][field]; optionally subtract aref (jar = J a - aref)
template <int G, int V>
MYO_PHASE void rows_dot(int mslot, Ctx<G, V> c, int ox, int field, bool sub_aref, bool sync = true) {
  MYO_M
  const float* x = SO(ox);
  const int* misc = SI(o_misc);
  const int nlim = misc[MI_NLIM], ncon = misc[MI_NCON];
  float* rows = SF(o_row);
  for (int r = c.lane; r < nlim; r += G) {
    const float* lr = SF(o_lim) + r * LIM_WORDS; const int* li = reinterpret_cast<const int*>(lr);
    float v = 0.f;
    for (int e = 0; e < li[L_NSUP]; e++) v += lim_J(c.sp(), lr, li, e) * x[lim_idx(li, e)];
    float* row = rows + r * ROW_WORDS;
    row[field] = sub_aref ? v - row[R_AREF] : v;
  }
  // contacts: E lanes per contact, each taking every E-th support entry, partial sums combined by shuffles
  constexpr int E = G >= KS ? KS : G;
  const int sub = c.lane % E;
  for (int base = 0; base < ncon; base += G / E) {
    const int k = base + c.lane / E;
    const bool on = k < ncon;
    const float* cr = SF(o_con) + (on ? k : 0) * CON_WORDS; const int* ci = reinterpret_cast<const int*>(cr);
    const int row0 = on ? ci[C_ROW0] : -1;
    float vn = 0.f, vt1 = 0.f, vt2 = 0.f;
    if (row0 >= 0)
      for (int e = sub; e < ci[C_NSUP]; e += E) {
        float jn, jt1, jt2;
        const int dof = contact_entry(m, c.sp(), cr, ci, e, &jn, &jt1, &jt2);
        const float w = x[dof];
        vn += jn * w; vt1 += jt1 * w; vt2 += jt2 * w;
      }
#pragma unroll
    for (int o = E / 2; o > 0; o >>= 1) { vn += c.tile.shfl_xor(vn, o); vt1 += c.tile.shfl_xor(vt1, o); vt2 += c.tile.shfl_xor(vt2, o); }
    if (row0 >= 0 && sub == 0) {
      const float mu = cr[C_MU];
      const int nr = ci[C_DIM] == 1 ? 1 : 4;
      for (int q = 0; q < nr; q++) {
        float v = vn;
        if (nr == 4) v += ((q & 1) ? -mu : mu) * ((q < 2) ? vt1 : vt2);
        float* row = rows + (row0 + q) * ROW_WORDS;
        row[field] = sub_aref ? v - row[R_AREF] : v;
      }
    }
  }
  if (sync) c.tile.sync();
}

// Joint-limit rows touch one dof each and come joint-major (lower side, then upper side), so a lane per row can apply
// them without write conflicts: the lane of a joint's first row also applies the second row if both sides are present.
// fn(r) -> contribution weight of row r; apply(dof, sign * weight)
template <int G, int V, class W, class A>
MYO_DI void for_joint_limit_rows(const DevModel& m, const Ctx<G, V> c, int nlim, W weight, A apply) {
  for (int r = c.lane; r < nlim; r += G) {
    const float* lr = MYO_SMEM_WORDS + c.soff + m.o_lim + r * LIM_WORDS; const int* li = reinterpret_cast<const int*>(lr);
    if (li[L_KIND] != EFC_LIMIT_JOINT) continue;
    if (r > 0 && li[L_KIND - LIM_WORDS] == EFC_LIMIT_JOINT && li[L_ID - LIM_WORDS] == li[L_ID]) continue;
    float v = lr[L_SIGN] * weight(r);
    if (r + 1 < nlim && li[L_KIND + LIM_WORDS] == EFC_LIMIT_JOINT && li[L_ID + LIM_WORDS] == li[L_ID]) v += lr[L_SIGN + LIM_WORDS] * weight(r + 1);
    apply(lim_idx(li, 0), v);
  }
}

// out[dof] += sum_r J_r[dof] * w_r  with w_r = (jar_r < 0 ? -D_r jar_r : 0) * scale  (forces)
// joint-limit rows in parallel (above); tendon-limit rows and contacts one after the other, lanes across the block's
// support: no atomics, fixed order.
template <int G, int V>
MYO_PHASE void rows_JT_force(int mslot, Ctx<G, V> c, int oout, float scale) {
  MYO_M
  float* out = SO(oout);
  const int* misc = SI(o_misc);
  const int nlim = misc[MI_NLIM], ncon = misc[MI_NCON];
  const float* rows = SF(o_row);
  for_joint_limit_rows<G>(m, c, nlim,
      [&](int r) { const float* row = rows + r * ROW_WORDS; return row[R_JAR] < 0.f ? -row[R_D] * row[R_JAR] * scale : 0.f; },
      [&](int dof, float v) { out[dof] += v; });
  c.tile.sync();
  if (m.any_tendon_limit)
    for (int r = 0; r < nlim; r++) {
      const float* lr = SF(o_lim) + r * LIM_WORDS; const int* li = reinterpret_cast<const int*>(lr);
      if (li[L_KIND] == EFC_LIMIT_JOINT) continue;
      const float* row = rows + r * ROW_WORDS;
      const float f = row[R_JAR] < 0.f ? -row[R_D] * row[R_JAR] * scale : 0.f;
      if (f != 0.f) for (int e = c.lane; e < li[L_NSUP]; e += G) out[lim_idx(li, e)] += lim_J(c.sp(), lr, li, e) * f;
      c.tile.sync();
    }
  if constexpr (G >= 2 * KS) {
    // two contacts per pass, half a tile each (support <= KS): the Jacobian entries - the expensive part - are computed for both at
    // once; the two halves then add one after the other (their supports overlap on the dofs of a shared body)
    const int hf = c.lane / KS, sub = c.lane % KS;
    for (int k0 = 0; k0 < ncon; k0 += 2) {
      const int k = k0 + hf;
      const bool has = k < ncon;
      const float* cr = SF(o_con) + (has ? k : k0) * CON_WORDS; const int* ci = reinterpret_cast<const int*>(cr);
      const int row0 = has ? ci[C_ROW0] : -1;
      float fn = 0.f, ft1 = 0.f, ft2 = 0.f;
      if (row0 >= 0) {
        const int nr = ci[C_DIM] == 1 ? 1 : 4;
        const float mu = cr[C_MU];
        for (int q = 0; q < nr; q++) {
          const float* row = rows + (row0 + q) * ROW_WORDS;
          const float f = row[R_JAR] < 0.f ? -row[R_D] * row[R_JAR] * scale : 0.f;
          fn += f;
          if (nr == 4) { const float t = ((q & 1) ? -mu : mu) * f; if (q < 2) ft1 += t; else ft2 += t; }
        }
      }
      const bool on = fn != 0.f && sub < ci[C_NSUP];
      float v = 0.f;
      int dof = 0;
      if (on) {
        float jn, jt1, jt2;
        dof = contact_entry(m, c.sp(), cr, ci, sub, &jn, &jt1, &jt2);
        v = jn * fn + jt1 * ft1 + jt2 * ft2;
      }
      if (on && hf == 0) out[dof] += v;
      c.tile.sync();
      if (on && hf == 1) out[dof] += v;
      c.tile.sync();
    }
  } else
  if constexpr (G >= KS && G > 1) {
    // support <= KS <= G: lane e holds entry e; the entries of contact k + 1 are computed under the update of contact k (see newton_system)
    auto load_entry = [&](int k, float& e_jn, float& e_jt1, float& e_jt2, int& e_dof) {
      e_jn = 0.f; e_jt1 = 0.f; e_jt2 = 0.f; e_dof = 0;
      if (k < ncon) {
        const float* cr = SF(o_con) + k * CON_WORDS; const int* ci = reinterpret_cast<const int*>(cr);
        if (ci[C_ROW0] >= 0 && c.lane < ci[C_NSUP]) e_dof = contact_entry(m, c.sp(), cr, ci, c.lane, &e_jn, &e_jt1, &e_jt2);
      }
    };
    float jn, jt1, jt2;
    int dof;
    load_entry(0, jn, jt1, jt2, dof);
    for (int k = 0; k < ncon; k++) {
      float njn, njt1, njt2;
      int ndof;
      load_entry(k + 1, njn, njt1, njt2, ndof);
      const float* cr = SF(o_con) + k * CON_WORDS; const int* ci = reinterpret_cast<const int*>(cr);
      const int row0 = ci[C_ROW0];
      if (row0 >= 0) {
        const int nr = ci[C_DIM] == 1 ? 1 : 4;
        const float mu = cr[C_MU];
        float fn = 0.f, ft1 = 0.f, ft2 = 0.f;
        for (int q = 0; q < nr; q++) {
          const float* row = rows + (row0 + q) * ROW_WORDS;
          const float f = row[R_JAR] < 0.f ? -row[R_D] * row[R_JAR] * scale : 0.f;
          fn += f;
          if (nr == 4) { const float t = ((q & 1) ? -mu : mu) * f; if (q < 2) ft1 += t; else ft2 += t; }
        }
        if (fn != 0.f) {
          if (c.lane < ci[C_NSUP]) out[dof] += jn * fn + jt1 * ft1 + jt2 * ft2;
          c.tile.sync();
        }
      }
      jn = njn; jt1 = njt1; jt2 = njt2; dof = ndof;
    }
  } else
  for (int k = 0; k < ncon; k++) {
    const float* cr = SF(o_con) + k * CON_WORDS; const int* ci = reinterpret_cast<const int*>(cr);
    const int row0 = ci[C_ROW0];
    if (row0 < 0) continue;
    const int nr = ci[C_DIM] == 1 ? 1 : 4;
    const float mu = cr[C_MU];
    float fn = 0.f, ft1 = 0.f, ft2 = 0.f;
    for (int q = 0; q < nr; q++) {
      const float* row = rows + (row0 + q) * ROW_WORDS;
      const float f = row[R_JAR] < 0.f ? -row[R_D] * row[R_JAR] * scale : 0.f;
      fn += f;
      if (nr == 4) { const float t = ((q & 1) ? -mu : mu) * f; if (q < 2) ft1 += t; else ft2 += t; }
    }
    for (int e = c.lane; e < ci[C_NSUP]; e += G) {
      float jn, jt1, jt2;
      const int dof = contact_entry(m, c.sp(), cr, ci, e, &jn, &jt1, &jt2);
      out[dof] += jn * fn + jt1 * ft1 + jt2 * ft2;
    }
    c.tile.sync();
  }
}

// Dense Newton system in scratch: lower triangle of H by rows, row i starting at word m.h_roff[i] (float4 aligned; four
// rows share a length that is an odd number of float4s, so a lane per row reads float4s with few bank conflicts);
// rows nv..n4-1 pad to a multiple of four (identity), row n4 holds the right-hand side.
//   grad = M a - f_smooth - J' f(jar)          (f_r = -D_r jar_r on active rows: jar_r < 0)
//   H    = M + sum_{active rows} D_r J_r' J_r,  right-hand side = -grad
// One walk over the constraint blocks feeds both: joint-limit rows lane-parallel (disjoint dofs), tendon-limit rows and
// contacts one after the other, lanes across the block's support / support pairs (no atomics, fixed order).
template <int G, int V>
MYO_PHASE void newton_system(int mslot, Ctx<G, V> c) {
  MYO_M
  float* H = SF(o_H); const float* M = SF(o_M); float* grad = SF(o_grad);
  const float* Ma = SF(o_Ma); const float* fs = SF(o_smooth);
  const int nv = m.nv;
  const int* roff = m.h_roff.ptr();
  const int n4 = (nv + 3) & ~3;
  for (int i = nv + c.lane; i < n4; i += G) {       // identity padding rows up to a multiple of four
    for (int k = 0; k <= i; k++) H[roff[i] + k] = (k == i) ? 1.f : 0.f;
  }
  // a lane owns a row: clear it, then drop the row's mass-matrix entries (i, ancestors of i) into it
  for (int i = c.lane; i < nv; i += G) {
    grad[i] = Ma[i] - fs[i];
    float* Hi = H + roff[i];
    float4* row4 = reinterpret_cast<float4*>(Hi);
    for (int k = 0; k <= i / 4; k++) row4[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    int adr = m.d_Madr[i], j = i;
    while (j >= 0) { Hi[j] = M[adr++]; j = m.d_parent[j]; }
  }
  c.tile.sync();
  const int* misc = SI(o_misc);
  const int nlim = misc[MI_NLIM], ncon = misc[MI_NCON];
  const float* rows = SF(o_row);
  // joint limits: J = +-1 on one dof: H_dd += D, grad_d -= sign * f = sign * D * jar
  for_joint_limit_rows<G>(m, c, nlim,
      [&](int r) { const float* row = rows + r * ROW_WORDS; const float* lr = SF(o_lim) + r * LIM_WORDS;
                   return row[R_JAR] < 0.f ? row[R_D] * lr[L_SIGN] : 0.f; },     // sign * (sign * D) = D
      [&](int dof, float v) { H[roff[dof] + dof] += v; });
  for_joint_limit_rows<G>(m, c, nlim,
      [&](int r) { const float* row = rows + r * ROW_WORDS; return row[R_JAR] < 0.f ? row[R_D] * row[R_JAR] : 0.f; },
      [&](int dof, float v) { grad[dof] += v; });
  c.tile.sync();
  if (m.any_tendon_limit)
    for (int r = 0; r < nlim; r++) {
      const float* lr = SF(o_lim) + r * LIM_WORDS; const int* li = reinterpret_cast<const int*>(lr);
      if (li[L_KIND] == EFC_LIMIT_JOINT) continue;
      const float* row = rows + r * ROW_WORDS;
      if (row[R_JAR] < 0.f) {
        const int ns = li[L_NSUP];
        const float D = row[R_D], nf = D * row[R_JAR];     // -f
        for (int e = c.lane; e < ns; e += G) grad[lim_idx(li, e)] += lim_J(c.sp(), lr, li, e) * nf;
        for (int e = c.lane; e < ns * ns; e += G) {
          const int a = e / ns, b = e - a * ns;
          const int ia = lim_idx(li, a), ib = lim_idx(li, b);
          if (ia >= ib) H[roff[ia] + ib] += D * lim_J(c.sp(), lr, li, a) * lim_J(c.sp(), lr, li, b);
        }
      }
      c.tile.sync();
    }
  if constexpr (G >= 2 * KS) {
    // Two contacts per pass: half h of the tile holds the Jacobian entries of contact k0 + h (support <= KS), computed for both at
    // once and - software-pipelined by hand - one pass ahead of the pair updates that consume them by shuffle; two batches of pairs
    // are in flight at a time (loads, arithmetic, stores: the pairs of one contact are distinct entries of H). With 3.5 warps per
    // scheduler the kernel lives on the independent instructions each warp brings itself.
    const int hf = c.lane / KS, sub = c.lane % KS;
    auto load_entry = [&](int k0, float& e_jn, float& e_jt1, float& e_jt2, int& e_dof) {
      e_jn = 0.f; e_jt1 = 0.f; e_jt2 = 0.f; e_dof = 0;
      const int k = k0 + hf;
      if (k < ncon) {
        const float* cr = SF(o_con) + k * CON_WORDS; const int* ci = reinterpret_cast<const int*>(cr);
        if (ci[C_ROW0] >= 0 && sub < ci[C_NSUP]) e_dof = contact_entry(m, c.sp(), cr, ci, sub, &e_jn, &e_jt1, &e_jt2);
      }
    };
    float jn, jt1, jt2;
    int dof;
    load_entry(0, jn, jt1, jt2, dof);
    for (int k0 = 0; k0 < ncon; k0 += 2) {
      float njn, njt1, njt2;
      int ndof;
      load_entry(k0 + 2, njn, njt1, njt2, ndof);
      for (int h = 0; h < 2 && k0 + h < ncon; h++) {
        const float* cr = SF(o_con) + (k0 + h) * CON_WORDS; const int* ci = reinterpret_cast<const int*>(cr);
        const int row0 = ci[C_ROW0];
        if (row0 < 0) continue;
        const int nr = ci[C_DIM] == 1 ? 1 : 4, ns = ci[C_NSUP];
        const float mu = cr[C_MU];
        // W = sum_active D c c', c = (1, +-mu, 0) / (1, 0, +-mu); (gn, g1, g2) = -(force in the contact frame)
        float w00 = 0.f, w01 = 0.f, w02 = 0.f, w11 = 0.f, w22 = 0.f, gn = 0.f, g1 = 0.f, g2 = 0.f;
        for (int q = 0; q < nr; q++) {
          const float4 row = *reinterpret_cast<const float4*>(rows + (row0 + q) * ROW_WORDS);     // D, aref, jar, jp
          if (row.z < 0.f) {
            const float D = row.x, nf = D * row.z;
            w00 += D; gn += nf;
            if (nr == 4) {
              const float s = (q & 1) ? -mu : mu;
              if (q < 2) { w01 += D * s; w11 += D * s * s; g1 += nf * s; } else { w02 += D * s; w22 += D * s * s; g2 += nf * s; }
            }
          }
        }
        if (w00 == 0.f) continue;
        const int base = h * KS;
        if (hf == h && sub < ns) grad[dof] += jn * gn + jt1 * g1 + jt2 * g2;
        // (W J) of the lane's own entry once, so that a pair costs three products: (W J_a) . J_b
        const float un = w00 * jn + w01 * jt1 + w02 * jt2, ut = w01 * jn + w11 * jt1, uu = w02 * jn + w22 * jt2;
        // every unordered pair (a >= b) of the support once: e = a (a + 1) / 2 + b
        const int npair = ns * (ns + 1) / 2;
        for (int e0 = 0; e0 < npair; e0 += 2 * G) {
          const int eA = e0 + c.lane, eB = e0 + G + c.lane;
          const bool onA = eA < npair, onB = eB < npair;
          const int abA = m.pair_ab[onA ? eA : 0], abB = m.pair_ab[onB ? eB : 0];
          const int aA = base + (abA & 255), bA = base + (abA >> 8), aB = base + (abB & 255), bB = base + (abB >> 8);
          const int iaA = c.tile.shfl(dof, aA), ibA = c.tile.shfl(dof, bA), iaB = c.tile.shfl(dof, aB), ibB = c.tile.shfl(dof, bB);
          const float naA = c.tile.shfl(un, aA), taA = c.tile.shfl(ut, aA), uaA = c.tile.shfl(uu, aA);
          const float nbA = c.tile.shfl(jn, bA), tbA = c.tile.shfl(jt1, bA), ubA = c.tile.shfl(jt2, bA);
          const float naB = c.tile.shfl(un, aB), taB = c.tile.shfl(ut, aB), uaB = c.tile.shfl(uu, aB);
          const float nbB = c.tile.shfl(jn, bB), tbB = c.tile.shfl(jt1, bB), ubB = c.tile.shfl(jt2, bB);
          float* hA = H + roff[max(iaA, ibA)] + min(iaA, ibA);
          float* hB = H + roff[max(iaB, ibB)] + min(iaB, ibB);
          const float oA = onA ? *hA : 0.f, oB = onB ? *hB : 0.f;
          const float vA = naA * nbA + taA * tbA + uaA * ubA;
          const float vB = naB * nbB + taB * tbB + uaB * ubB;
          if (onA) *hA = oA + vA;
          if (onB) *hB = oB + vB;
        }
        c.tile.sync();
      }
      jn = njn; jt1 = njt1; jt2 = njt2; dof = ndof;
    }
  } else
  if constexpr (G >= KS && G > 1) {
    // A contact block fits the tile (support <= KS <= G): lane e holds entry e and pairs fetch both entries by shuffle. The walk is
    // software-pipelined by hand - the entries of contact k + 1 (a chain of dependent shared-memory loads) are computed before
    // the pairs of contact k are applied, and two batches of pairs are in flight at a time (loads, arithmetic, stores: the pairs
    // of one contact are distinct entries of H) - because with 3.5 warps per scheduler the kernel lives on the independent
    // instructions each warp brings itself.
    auto load_entry = [&](int k, float& e_jn, float& e_jt1, float& e_jt2, int& e_dof) {
      e_jn = 0.f; e_jt1 = 0.f; e_jt2 = 0.f; e_dof = 0;
      if (k < ncon) {
        const float* cr = SF(o_con) + k * CON_WORDS; const int* ci = reinterpret_cast<const int*>(cr);
        if (ci[C_ROW0] >= 0 && c.lane < ci[C_NSUP]) e_dof = contact_entry(m, c.sp(), cr, ci, c.lane, &e_jn, &e_jt1, &e_jt2);
      }
    };
    float jn, jt1, jt2;
    int dof;
    load_entry(0, jn, jt1, jt2, dof);
    for (int k = 0; k < ncon; k++) {
      float njn, njt1, njt2;
      int ndof;
      load_entry(k + 1, njn, njt1, njt2, ndof);
      const float* cr = SF(o_con) + k * CON_WORDS; const int* ci = reinterpret_cast<const int*>(cr);
      const int row0 = ci[C_ROW0];
      if (row0 >= 0) {
        const int nr = ci[C_DIM] == 1 ? 1 : 4, ns = ci[C_NSUP];
        const float mu = cr[C_MU];
        // W = sum_active D c c', c = (1, +-mu, 0) / (1, 0, +-mu); (gn, g1, g2) = -(force in the contact frame)
        float w00 = 0.f, w01 = 0.f, w02 = 0.f, w11 = 0.f, w22 = 0.f, gn = 0.f, g1 = 0.f, g2 = 0.f;
        for (int q = 0; q < nr; q++) {
          const float4 row = *reinterpret_cast<const float4*>(rows + (row0 + q) * ROW_WORDS);     // D, aref, jar, jp
          if (row.z < 0.f) {
            const float D = row.x, nf = D * row.z;
            w00 += D; gn += nf;
            if (nr == 4) {
              const float s = (q & 1) ? -mu : mu;
              if (q < 2) { w01 += D * s; w11 += D * s * s; g1 += nf * s; } else { w02 += D * s; w22 += D * s * s; g2 += nf * s; }
            }
          }
        }
        if (w00 != 0.f) {
          if (c.lane < ns) grad[dof] += jn * gn + jt1 * g1 + jt2 * g2;
          // every unordered pair (a >= b) of the support once: e = a (a + 1) / 2 + b
          const int npair = ns * (ns + 1) / 2;
          for (int e0 = 0; e0 < npair; e0 += 2 * G) {
            const int eA = e0 + c.lane, eB = e0 + G + c.lane;
            const bool onA = eA < npair, onB = eB < npair;
            const int abA = m.pair_ab[onA ? eA : 0], abB = m.pair_ab[onB ? eB : 0];
            const int aA = abA & 255, bA = abA >> 8, aB = abB & 255, bB = abB >> 8;
            const int iaA = c.tile.shfl(dof, aA), ibA = c.tile.shfl(dof, bA), iaB = c.tile.shfl(dof, aB), ibB = c.tile.shfl(dof, bB);
            const float naA = c.tile.shfl(jn, aA), taA = c.tile.shfl(jt1, aA), uaA = c.tile.shfl(jt2, aA);
            const float nbA = c.tile.shfl(jn, bA), tbA = c.tile.shfl(jt1, bA), ubA = c.tile.shfl(jt2, bA);
            const float naB = c.tile.shfl(jn, aB), taB = c.tile.shfl(jt1, aB), uaB = c.tile.shfl(jt2, aB);
            const float nbB = c.tile.shfl(jn, bB), tbB = c.tile.shfl(jt1, bB), ubB = c.tile.shfl(jt2, bB);
            float* hA = H + roff[max(iaA, ibA)] + min(iaA, ibA);
            float* hB = H + roff[max(iaB, ibB)] + min(iaB, ibB);
            const float oA = onA ? *hA : 0.f, oB = onB ? *hB : 0.f;
            const float vA = w00 * naA * nbA + w01 * (naA * tbA + taA * nbA) + w02 * (naA * ubA + uaA * nbA) + w11 * taA * tbA + w22 * uaA * ubA;
            const float vB = w00 * naB * nbB + w01 * (naB * tbB + taB * nbB) + w02 * (naB * ubB + uaB * nbB) + w11 * taB * tbB + w22 * uaB * ubB;
            if (onA) *hA = oA + vA;
            if (onB) *hB = oB + vB;
          }
          c.tile.sync();
        }
      }
      jn = njn; jt1 = njt1; jt2 = njt2; dof = ndof;
    }
  } else
  for (int k = 0; k < ncon; k++) {
    const float* cr = SF(o_con) + k * CON_WORDS; const int* ci = reinterpret_cast<const int*>(cr);
    const int row0 = ci[C_ROW0];
    if (row0 < 0) continue;
    const int nr = ci[C_DIM] == 1 ? 1 : 4, ns = ci[C_NSUP];
    const float mu = cr[C_MU];
    // W = sum_active D c c', c = (1, +-mu, 0) / (1, 0, +-mu); (gn, g1, g2) = -(force in the contact frame)
    float w00 = 0.f, w01 = 0.f, w02 = 0.f, w11 = 0.f, w22 = 0.f, gn = 0.f, g1 = 0.f, g2 = 0.f;
    for (int q = 0; q < nr; q++) {
      const float4 row = *reinterpret_cast<const float4*>(rows + (row0 + q) * ROW_WORDS);     // D, aref, jar, jp
      if (row.z < 0.f) {
        const float D = row.x, nf = D * row.z;
        w00 += D; gn += nf;
        if (nr == 4) {
          const float s = (q & 1) ? -mu : mu;
          if (q < 2) { w01 += D * s; w11 += D * s * s; g1 += nf * s; } else { w02 += D * s; w22 += D * s * s; g2 += nf * s; }
        }
      }
    }
    if (w00 != 0.f) {
      // lane e holds entry e of the block and pairs fetch both entries by shuffle (when the block fits the tile;
      // narrower development tiles and the single-lane host emulation recompute the two entries instead)
      const bool by_shfl = G > 1 && ns <= G;
      float jn = 0.f, jt1 = 0.f, jt2 = 0.f;
      int dof = 0;
      if (by_shfl) {
        if (c.lane < ns) { dof = contact_entry(m, c.sp(), cr, ci, c.lane, &jn, &jt1, &jt2); grad[dof] += jn * gn + jt1 * g1 + jt2 * g2; }
      } else {
        for (int e = c.lane; e < ns; e += G) { const int d = contact_entry(m, c.sp(), cr, ci, e, &jn, &jt1, &jt2); grad[d] += jn * gn + jt1 * g1 + jt2 * g2; }
      }
      // every unordered pair (a >= b) of the support once: e = a (a + 1) / 2 + b
      const int npair = ns * (ns + 1) / 2;
      for (int e0 = 0; e0 < npair; e0 += G) {
        const int e = e0 + c.lane;
        const int ab = m.pair_ab[e < npair ? e : 0];
        const int a = ab & 255, b = ab >> 8;
        int ia, ib;
        float na, ta, ua, nb, tb, ub;
        if (by_shfl) {
          ia = c.tile.shfl(dof, a); na = c.tile.shfl(jn, a); ta = c.tile.shfl(jt1, a); ua = c.tile.shfl(jt2, a);
          ib = c.tile.shfl(dof, b); nb = c.tile.shfl(jn, b); tb = c.tile.shfl(jt1, b); ub = c.tile.shfl(jt2, b);
        } else {
          ia = contact_entry(m, c.sp(), cr, ci, a, &na, &ta, &ua);
          ib = contact_entry(m, c.sp(), cr, ci, b, &nb, &tb, &ub);
        }
        if (e < npair)
          H[roff[max(ia, ib)] + min(ia, ib)] += w00 * na * nb + w01 * (na * tb + ta * nb) + w02 * (na * ub + ua * nb) + w11 * ta * tb + w22 * ua * ub;
      }
    }
    c.tile.sync();
  }
  for (int k = c.lane; k < n4; k += G) H[roff[n4] + k] = k < nv ? -grad[k] : 0.f;
  c.tile.sync();
}

// In-place dense Cholesky H = L L', left-looking by blocks of four columns, a lane per row. For a block the lane
// accumulates four dot products of its row against the four pivot rows (float4 loads, 16 independent FMA chains), the
// 4 x 4 diagonal block is gathered with shuffles and factored redundantly in registers, and the lane finishes its four
// entries with a register triangular solve: one tile barrier per four columns. The forward substitution is fused in:
// the right-hand-side row n4 is carried through like one more matrix row and ends as y = L^-1 rhs. Diagonal slots keep
// 1 / L_jj. n4 = n rounded up to 4 (rows n..n4-1 are identity rows written by build_hessian).
// Then the back substitution L' x = y, column oriented, with y held in registers (lane i owns y_i, y_{i+G}, ...)
// and each finished x_j broadcast by a shuffle; x goes to scratch at ox.
template <int G, int V>
MYO_PHASE void chol_factor_solve(int mslot, Ctx<G, V> c, int oH, int ox, int n) {
  MYO_M
  float* H = SO(oH); float* x = SO(ox);
  const int* roff = m.h_roff.ptr();
  const int n4 = (n + 3) & ~3;
  if constexpr (G < 4) {   // single-lane host emulation (tests/emul): same storage convention, unblocked
    for (int j = 0; j < n4; j++) {
      float inv = 0.f;
      for (int i = j; i <= n4; i++) {
        float s = H[roff[i] + j];
        for (int k = 0; k < j; k++) s -= H[roff[i] + k] * H[roff[j] + k];
        if (i == j) { inv = 1.f / sqrtf(fmaxf(s, kMinVal)); H[roff[i] + j] = inv; } else H[roff[i] + j] = s * inv;
      }
    }
  } else
  for (int J = 0; J < n4; J += 4) {
    const float* P0 = H + roff[J];     // pivot rows J..J+3
    const float* P1 = H + roff[J + 1]; const float* P2 = H + roff[J + 2]; const float* P3 = H + roff[J + 3];
    float l10 = 0.f, l20 = 0.f, l21 = 0.f, l30 = 0.f, l31 = 0.f, l32 = 0.f, inv0 = 0.f, inv1 = 0.f, inv2 = 0.f, inv3 = 0.f;
    // Late blocks have few rows left (n4 + 1 - J) and the longest dot products: when the rows fit half a tile, two lanes share a
    // row - lane and lane + G/2 each take half of the column chunks, one shuffle adds the halves - so the idle lanes shorten the
    // longest dependent stretch of the factorisation (the result differs from the one-lane sum in the last bits only).
    const bool split = G >= 8 && J >= 8 && n4 + 1 - J <= G / 2;
    for (int i0 = J; i0 <= n4; i0 += G) {
      const int hlf = split ? c.lane / (G / 2) : 0;
      const int i = i0 + (split ? c.lane % (G / 2) : c.lane);
      const bool on = i <= n4;
      float* Li = H + roff[on ? i : J];
      float4 acc = *reinterpret_cast<const float4*>(Li + J);
      int k0 = 0, k1 = J;
      if (split) {
        const int mid = ((J / 4 + 1) / 2) * 4;
        if (hlf) { k0 = mid; acc = make_float4(0.f, 0.f, 0.f, 0.f); } else k1 = mid;
      }
      for (int k = k0; k < k1; k += 4) {
        const float4 a = *reinterpret_cast<const float4*>(Li + k);
        const float4 b0 = *reinterpret_cast<const float4*>(P0 + k);
        const float4 b1 = *reinterpret_cast<const float4*>(P1 + k);
        const float4 b2 = *reinterpret_cast<const float4*>(P2 + k);
        const float4 b3 = *reinterpret_cast<const float4*>(P3 + k);
        acc.x -= a.x * b0.x; acc.x -= a.y * b0.y; acc.x -= a.z * b0.z; acc.x -= a.w * b0.w;
        acc.y -= a.x * b1.x; acc.y -= a.y * b1.y; acc.y -= a.z * b1.z; acc.y -= a.w * b1.w;
        acc.z -= a.x * b2.x; acc.z -= a.y * b2.y; acc.z -= a.z * b2.z; acc.z -= a.w * b2.w;
        acc.w -= a.x * b3.x; acc.w -= a.y * b3.y; acc.w -= a.z * b3.z; acc.w -= a.w * b3.w;
      }
      if (split) {
        acc.x += c.tile.shfl_xor(acc.x, G / 2); acc.y += c.tile.shfl_xor(acc.y, G / 2);
        acc.z += c.tile.shfl_xor(acc.z, G / 2); acc.w += c.tile.shfl_xor(acc.w, G / 2);
      }
      if (i0 == J) {   // first pass: lanes 0..3 hold the diagonal block
        const float d00 = c.tile.shfl(acc.x, 0);
        const float d10 = c.tile.shfl(acc.x, 1 % G), d11 = c.tile.shfl(acc.y, 1 % G);
        const float d20 = c.tile.shfl(acc.x, 2 % G), d21 = c.tile.shfl(acc.y, 2 % G), d22 = c.tile.shfl(acc.z, 2 % G);
        const float d30 = c.tile.shfl(acc.x, 3 % G), d31 = c.tile.shfl(acc.y, 3 % G), d32 = c.tile.shfl(acc.z, 3 % G), d33 = c.tile.shfl(acc.w, 3 % G);
        inv0 = rsqrt_pos(fmaxf(d00, kMinVal));
        l10 = d10 * inv0; l20 = d20 * inv0; l30 = d30 * inv0;
        inv1 = rsqrt_pos(fmaxf(d11 - l10 * l10, kMinVal));
        l21 = (d21 - l20 * l10) * inv1; l31 = (d31 - l30 * l10) * inv1;
        inv2 = rsqrt_pos(fmaxf(d22 - l20 * l20 - l21 * l21, kMinVal));
        l32 = (d32 - l30 * l20 - l31 * l21) * inv2;
        inv3 = rsqrt_pos(fmaxf(d33 - l30 * l30 - l31 * l31 - l32 * l32, kMinVal));
      }
      float4 r;
      r.x = acc.x * inv0;
      r.y = (acc.y - r.x * l10) * inv1;
      r.z = (acc.z - r.x * l20 - r.y * l21) * inv2;
      r.w = (acc.w - r.x * l30 - r.y * l31 - r.z * l32) * inv3;
      const int q = i - J;     // rows of the diagonal block: inverse pivot on the diagonal, zeros above it
      const bool q0 = q == 0, q1 = q == 1, q2 = q == 2, q3 = q == 3;
      r.x = q0 ? inv0 : r.x;
      r.y = q1 ? inv1 : (q0 ? 0.f : r.y);
      r.z = q2 ? inv2 : ((q0 || q1) ? 0.f : r.z);
      r.w = q3 ? inv3 : ((q0 || q1 || q2) ? 0.f : r.w);
      if (on) *reinterpret_cast<float4*>(Li + J) = r;
    }
    c.tile.sync();
  }
  constexpr int NSET = 64 / G;     // nv <= 64 (pack_model)
  float y[NSET];
#pragma unroll
  for (int q = 0; q < NSET; q++) { const int i = c.lane + q * G; y[q] = i < n ? H[roff[n4] + i] : 0.f; }
  // y_j from the lane that owns it
  auto fetch = [&](int j) {
    const int jq = j / G;
    float v = y[0];
#pragma unroll
    for (int q = 1; q < NSET; q++) v = (jq == q) ? y[q] : v;
    return c.tile.shfl(v, j - jq * G);
  };
  // back substitution L' x = y by blocks of four columns, last block first: the 4 x 4 diagonal block (stored as the
  // factorisation left it: inverse pivots on the diagonal) is solved redundantly in registers, then every lane
  // removes the four new x from the rows it owns
  for (int J = n4 - 4; J >= 0; J -= 4) {
    const float* R0 = H + roff[J]; const float* R1 = H + roff[J + 1]; const float* R2 = H + roff[J + 2]; const float* R3 = H + roff[J + 3];
    const float4 d0 = *reinterpret_cast<const float4*>(R0 + J), d1 = *reinterpret_cast<const float4*>(R1 + J);
    const float4 d2 = *reinterpret_cast<const float4*>(R2 + J), d3 = *reinterpret_cast<const float4*>(R3 + J);
    const float y0 = fetch(J), y1 = fetch(J + 1), y2 = fetch(J + 2), y3 = fetch(J + 3);
    const float x3 = y3 * d3.w;
    const float x2 = (y2 - d3.z * x3) * d2.z;
    const float x1 = (y1 - d3.y * x3 - d2.y * x2) * d1.y;
    const float x0 = (y0 - d3.x * x3 - d2.x * x2 - d1.x * x1) * d0.x;
#pragma unroll
    for (int q = 0; q < NSET; q++) {
      const int i = c.lane + q * G;
      if (i < J) y[q] -= R0[i] * x0 + R1[i] * x1 + R2[i] * x2 + R3[i] * x3;
    }
    if (c.lane == 0) {
      if (J + 3 < n) *reinterpret_cast<float4*>(x + J) = make_float4(x0, x1, x2, x3);
      else { x[J] = x0; if (J + 1 < n) x[J + 1] = x1; if (J + 2 < n) x[J + 2] = x2; }
    }
  }
  c.tile.sync();
}

// x <- (M + hdamp diag(damping))^-1 x  (mj_factorM + mj_solveM; hdamp = h in mj_Euler's implicit damping).
// The coupled dofs [0, m.nd) go through the dense blocked Cholesky above (the Newton Hessian's scratch is free outside
// the constraint solve); the simple dofs behind them (free bodies with diagonal inertia: dof_simplenum) divide by
// their diagonal entry.
template <int G, int V>
MYO_PHASE void solve_M_dense(int mslot, Ctx<G, V> c, int ox, float hdamp) {
  MYO_M
  float* H = SF(o_H); const float* M = SF(o_M); float* x = SO(ox);
  const int nd = m.nd, n4 = (nd + 3) & ~3;
  const int* roff = m.h_roff.ptr();
  for (int k = c.lane; k < n4; k += G) H[roff[n4] + k] = k < nd ? x[k] : 0.f;
  for (int i = nd + c.lane; i < n4; i += G)
    for (int k = 0; k <= i; k++) H[roff[i] + k] = (k == i) ? 1.f : 0.f;
  for (int i = c.lane; i < nd; i += G) {
    float* Hi = H + roff[i];
    float4* row4 = reinterpret_cast<float4*>(Hi);
    for (int k = 0; k <= i / 4; k++) row4[k] = make_float4(0.f, 0.f, 0.f, 0.f);
    int adr = m.d_Madr[i], j = i;
    Hi[i] = M[adr++] + hdamp * m.d_damping[i];
    j = m.d_parent[j];
    while (j >= 0) { Hi[j] = M[adr++]; j = m.d_parent[j]; }
  }
  for (int i = nd + c.lane; i < m.nv; i += G) x[i] = x[i] / fmaxf(M[m.d_Madr[i]] + hdamp * m.d_damping[i], kMinVal);
  c.tile.sync();
  if (nd > 0) chol_factor_solve<G>(mslot, c, m.o_H, ox, nd);
}


// a10.8 constraint solve: primal Newton with exact line search on
//   cost(a) = 1/2 (a - a_s)' M (a - a_s) + sum_r 1/2 D_r min(0, J_r a - aref_r)^2
// warm-started from the better of (qacc_warmstart, qacc_smooth) as MuJoCo's warmstart() does.
// All warps of a CTA walk the phases together: the step is ~200 KB of straight-line code, far more
// than the instruction cache holds, so keeping the CTA inside one phase at a time lets every fetched
// line serve all of its warps. (Every tile of the CTA executes every phase of every substep.)
// Every phase boundary of a substep carries the CTA barrier. Worlds are independent, so the barriers are a performance
// device only (instruction-cache sharing); see DESIGN.md for the measured choices.
#define MYO_SYNC if (SYNC) __syncthreads();      // SYNC: template flag of the step functions

constexpr float kNewtonStepTol = 2e-5f;      // last Newton step relative to max(1, |qacc|_inf) below which the solve stops (fp32 floor)
template <int G, int RMAX, int V>
MYO_PHASE void phase_solve(int mslot, Ctx<G, V> c, bool fast) {
  MYO_M
  int* misc = SI(o_misc);
  const int nv = m.nv, nefc = misc[MI_NEFC];
  float* a = SF(o_qacc); float* qcon = SF(o_qcon);
  const float* as = SF(o_qaccs); const float* fs = SF(o_smooth);
  float* rows = SF(o_row);
  bool active = nefc > 0;
  if (!active) {
    for (int i = c.lane; i < nv; i += G) { a[i] = as[i]; SF(o_warm)[i] = as[i]; qcon[i] = 0.f; }
    if (c.lane == 0) misc[MI_ITER] = 0;
    c.tile.sync();
    return;
  }
  float* Ma = SF(o_Ma); float* grad = SF(o_grad); float* p = SF(o_p); float* Mp = SF(o_Mp);
  // constraint rows in registers for the reductions and the line search: lane owns rows lane, lane + G, ...
  // RMAX rows per lane: nefc_max <= RMAX * G (pack_model: kFastRows for the fast layout, kSoloRowsPerLane * G for the full one)
  auto row_cost = [&](int field) {
    float part = 0.f;
    for (int r = c.lane; r < nefc; r += G) { const float* row = rows + r * ROW_WORDS; const float j = row[field]; if (j < 0.f) part += 0.5f * row[R_D] * j * j; }
    return part;
  };
  // Starting point; jar and M a are then kept current incrementally (jar += alpha J p, Ma += alpha M p).
  // Test / dump modes follow MuJoCo's warmstart(): the better of qacc_warmstart and qacc_smooth by cost. The env step
  // (fast) starts from qacc_warmstart without evaluating qacc_smooth at all - the minimiser of the convex cost does not
  // depend on the starting point, and skipping M^-1 f_smooth and one pass over the rows saves ~8 % of a substep; only a
  // non-finite warm start falls back to qacc_smooth.
  if (active) {
    const float* w = SF(o_warm);
    bool use_smooth;
    if (fast) {
      float chk = 0.f;
      for (int i = c.lane; i < nv; i += G) chk += fabsf(w[i]);
      use_smooth = !(tile_sum<G>(c, chk) < 3.0e38f);
      if (use_smooth) {
        solve_M_dense<G>(mslot, c, m.o_qaccs, 0.f);
        rows_dot<G>(mslot, c, m.o_qaccs, R_JAR, true);
      } else {
        rows_dot<G>(mslot, c, m.o_warm, R_JAR, true, false);
        mul_M<G>(mslot, c, m.o_M, m.o_warm, m.o_Ma);
      }
    } else {
      rows_dot<G>(mslot, c, m.o_qaccs, R_JAR, true);
      const float cost_s = tile_sum<G>(c, row_cost(R_JAR));          // Gauss term vanishes at qacc_smooth
      rows_dot<G>(mslot, c, m.o_warm, R_JP, true, false);
      mul_M<G>(mslot, c, m.o_M, m.o_warm, m.o_Ma);
      float part = row_cost(R_JP);
      for (int i = c.lane; i < nv; i += G) part += 0.5f * (Ma[i] - fs[i]) * (w[i] - as[i]);
      const float cost_w = tile_sum<G>(c, part);
      use_smooth = !(cost_w <= cost_s);   // also catches NaN in the warm start
      if (!use_smooth) for (int r = c.lane; r < nefc; r += G) rows[r * ROW_WORDS + R_JAR] = rows[r * ROW_WORDS + R_JP];
    }
    if (use_smooth) {
      for (int i = c.lane; i < nv; i += G) { a[i] = as[i]; Ma[i] = fs[i]; }     // M a_s = f_s
    } else {
      for (int i = c.lane; i < nv; i += G) a[i] = w[i];
    }
    c.tile.sync();
  }
  const float scale = 1.f / (m.meaninertia * (float)max(1, nv));
  int iter = 0;
  MYO_PH_BEGIN
  float prev_step = 3.0e38f;
  for (int it = 0; it < m.solver_iter; it++) {
    if (!active) break;
    if (active) {
      MYO_PH_RESTART newton_system<G>(mslot, c); MYO_PH(11)
      float g2 = 0.f;
      for (int i = c.lane; i < nv; i += G) g2 += grad[i] * grad[i];
      g2 = tile_sum<G>(c, g2);
      if (sqrtf(g2) * scale < m.solver_tol) active = false;
    }
    if (active) { chol_factor_solve<G>(mslot, c, m.o_H, m.o_p, nv); MYO_PH(12) }
    if (active) {
    rows_dot<G>(mslot, c, m.o_p, R_JP, false, false);
    mul_M<G>(mslot, c, m.o_M, m.o_p, m.o_Mp);
    float pMp = 0.f, gp = 0.f, pmax = 0.f, amax = 0.f;
    for (int i = c.lane; i < nv; i += G) { pMp += p[i] * Mp[i]; gp += (Ma[i] - fs[i]) * p[i]; pmax = fmaxf(pmax, fabsf(p[i])); amax = fmaxf(amax, fabsf(a[i])); }
    pMp = tile_sum<G>(c, pMp); gp = tile_sum<G>(c, gp); pmax = tile_max<G>(c, pmax); amax = tile_max<G>(c, amax);
    float rD[RMAX], rJ[RMAX], rP[RMAX];
#pragma unroll
    for (int q = 0; q < RMAX; q++) {
      const int r = c.lane + q * G;
      if (r < nefc) { const float4 v = *reinterpret_cast<const float4*>(rows + r * ROW_WORDS); rD[q] = v.x; rJ[q] = v.z; rP[q] = v.w; }
      else { rD[q] = 0.f; rJ[q] = 1.f; rP[q] = 0.f; }      // inert: never active, never changes side
    }
    // exact line search on the piecewise-quadratic phi(alpha): safeguarded Newton on phi'
    float alpha = 0.f, lo = 0.f, hi = -1.f, d1_0 = 0.f;
    for (int ls = 0; ls < 12; ls++) {
      float d1 = 0.f, d2 = 0.f;
#pragma unroll
      for (int q = 0; q < RMAX; q++) {
        const float x = rJ[q] + alpha * rP[q];
        if (x < 0.f) { d1 += rD[q] * x * rP[q]; d2 += rD[q] * rP[q] * rP[q]; }
      }
      d1 = tile_sum<G>(c, d1) + gp + alpha * pMp;
      d2 = tile_sum<G>(c, d2) + pMp;
      if (ls == 0) d1_0 = fabsf(d1);
      if (fabsf(d1) <= 1e-6f * d1_0) break;
      if (d1 < 0.f) lo = alpha; else hi = alpha;
      float nxt = alpha - d1 / fmaxf(d2, kMinVal);
      if (hi >= 0.f && (nxt <= lo || nxt >= hi)) nxt = 0.5f * (lo + hi);
      if (nxt < lo) nxt = lo;
      if (nxt == alpha) break;
      alpha = nxt;
    }
    MYO_PH(14)
    // did any row change side along the step? if not, and the full Newton step was taken, a + p is the
    // exact minimiser of a cost that is quadratic on this active set: converged without a checking pass
    int changed = 0;
#pragma unroll
    for (int q = 0; q < RMAX; q++) {
      const float x1 = rJ[q] + alpha * rP[q];
      if ((rJ[q] < 0.f) != (x1 < 0.f)) changed = 1;
      const int r = c.lane + q * G;
      if (r < nefc) rows[r * ROW_WORDS + R_JAR] = x1;
    }
    changed = c.tile.ballot(changed != 0) != 0u;
    for (int i = c.lane; i < nv; i += G) { a[i] += alpha * p[i]; Ma[i] += alpha * Mp[i]; }
    c.tile.sync();
    iter++;
    if (!changed && fabsf(alpha - 1.f) <= 1e-3f) active = false;
    // fp32 termination: the Newton step is at the rounding floor of qacc (quadratic convergence makes
    // the remaining error far smaller than the last step), or it stopped shrinking (noise-level cycling).
    // The empty `if (active)` is kept on purpose: without it the compiler lays the solve out differently, and the kernels
    // built from this phase get larger stack frames and more spills (world_kernel<32>: 512 -> 528 B of stack).
    const float step = alpha * pmax, aref_mag = fmaxf(1.f, amax);
    if (step <= kNewtonStepTol * aref_mag || (iter > 1 && step >= 0.5f * prev_step && step <= 1e-3f * aref_mag)) { if (active) {} active = false; }
    prev_step = step;
    }
  }
  if (nefc == 0) return;
  // final forces at the solution (jar is current)
  for (int i = c.lane; i < nv; i += G) { qcon[i] = 0.f; SF(o_warm)[i] = a[i]; }
  c.tile.sync();
  rows_JT_force<G>(mslot, c, m.o_qcon, 1.f);
  if (c.lane == 0) misc[MI_ITER] = iter;
  c.tile.sync();
}

// ------------------------------------------------------------------------------------------------
// a10.9 mj_Euler (implicit in joint damping) + mj_advance
template <int G, int V>
MYO_PHASE void phase_integrate(int mslot, Ctx<G, V> c) {
  MYO_M
  const float h = m.timestep;
  float* qacc = SF(o_qacc); float* qvel = SF(o_qvel); float* qpos = SF(o_qpos); float* act = SF(o_act);
  float* x = SF(o_grad);
  if (m.any_damping) {
    for (int i = c.lane; i < m.nv; i += G) x[i] = SF(o_smooth)[i] + SF(o_qcon)[i];
    c.tile.sync();
    solve_M_dense<G>(mslot, c, m.o_grad, h);
  } else {
    for (int i = c.lane; i < m.nv; i += G) x[i] = qacc[i];
    c.tile.sync();
  }
  for (int i = c.lane; i < m.na; i += G) {
    const int u = i + (m.nu - m.na);
    float v = act[i] + h * SF(o_actdot)[i];
    if (m.a_dyntype[u] == 3) v = clipf(v, 0.f, 1.f);
    act[i] = v;
  }
  for (int i = c.lane; i < m.nv; i += G) qvel[i] += h * x[i];
  c.tile.sync();
  for (int j = c.lane; j < m.njnt; j += G) {
    const int qa = m.j_qposadr[j], da = m.j_dofadr[j];
    if (m.j_type[j] == J_FREE) {
      qpos[qa] += h * qvel[da]; qpos[qa + 1] += h * qvel[da + 1]; qpos[qa + 2] += h * qvel[da + 2];
      float w[3] = {qvel[da + 3], qvel[da + 4], qvel[da + 5]};
      const float ang = h * normalize3(w);
      float sn, cs;
      sincosf(0.5f * ang, &sn, &cs);
      const float ql[4] = {cs, w[0] * sn, w[1] * sn, w[2] * sn};
      float q[4] = {qpos[qa + 3], qpos[qa + 4], qpos[qa + 5], qpos[qa + 6]};
      if (ang != 0.f) mulquat(q, q, ql);
      normalize4(q);
      qpos[qa + 3] = q[0]; qpos[qa + 4] = q[1]; qpos[qa + 5] = q[2]; qpos[qa + 6] = q[3];
    } else qpos[qa] += h * qvel[da];
  }
  c.tile.sync();
}

// one full mj_step on the world in scratch
// SYNC: the CTA's tiles walk the phases in lock step (fast kernel); false where tiles run on their own (full-capacity passes)
template <int G, int RMAX, bool SYNC, int V>
MYO_PHASE void mj_forward_dev(int mslot, Ctx<G, V> c, int* status, bool fast) {
  MYO_M
  MYO_PH_BEGIN
  MYO_SYNC phase_tree_forward<G>(mslot, c, true); MYO_PH(0)
  MYO_PH(2)
  MYO_SYNC phase_mass_bias<G>(mslot, c); MYO_PH(3)
  // the velocity-stage temporaries are dead from here on: the tendon phase reuses their scratch (with the Hessian's)
  MYO_SYNC phase_tendon<G>(mslot, c, status); MYO_PH(1)
  MYO_SYNC phase_collision<G>(mslot, c, status); MYO_PH(5)
  MYO_SYNC phase_constraints<G>(mslot, c, status); MYO_PH(6)
  MYO_SYNC phase_actuation<G>(mslot, c); MYO_PH(7)
  if (!fast || SI(o_misc)[MI_NEFC] == 0) solve_M_dense<G>(mslot, c, m.o_qaccs, 0.f);   // qacc_smooth (see phase_solve)
  MYO_PH(8)
  MYO_SYNC phase_solve<G, RMAX>(mslot, c, fast); MYO_PH(9)
}
template <int G, int RMAX, bool SYNC, int V>
MYO_PHASE void mj_step_dev(int mslot, Ctx<G, V> c, int* status, bool fast) {
  MYO_M
  mj_forward_dev<G, RMAX, SYNC>(mslot, c, status, fast);
  MYO_PH_BEGIN
  MYO_SYNC MYO_PH(15) phase_integrate<G>(mslot, c); MYO_PH(10)
}

}  // namespace myo
