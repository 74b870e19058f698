// Model -> device tables. Everything derived here is static per model: tree levels, dof chains,
// descendant lists for the gather-form L'DL, tendon / contact supports, the collision candidate
// list with MuJoCo's static filters (mj_collision: same weld body, parent-child, contype/conaffinity),
// and the shared-memory scratch layout of one world.
#include "myo_pack.hpp"

#include <algorithm>
#include <cmath>
#include <cstddef>
#include <cstdlib>
#include <cstring>
#include <set>

namespace myo {

namespace {

struct Builder {
  PackedModel& pm;
  explicit Builder(PackedModel& p) : pm(p) {}
  void I(TabI& field, const std::vector<int>& v) {
    field.off = (int)pm.ibuf.size();
    pm.ibuf.insert(pm.ibuf.end(), v.begin(), v.end());
    if (v.empty()) pm.ibuf.push_back(0);
    while (pm.ibuf.size() % 4) pm.ibuf.push_back(0);
  }
  void F(TabF& field, const std::vector<float>& v) {
    field.off = (int)pm.fbuf.size();
    pm.ffix.push_back(&field);
    pm.fbuf.insert(pm.fbuf.end(), v.begin(), v.end());
    if (v.empty()) pm.fbuf.push_back(0.f);
    while (pm.fbuf.size() % 4) pm.fbuf.push_back(0.f);
  }
  // cold table: kept in the global copy only (read with plain loads through m.g_tables, served by L1 / L2), not staged
  // into shared memory - for tables that are touched once per substep by a lane-per-item loop
  void Fcold(TabF& field, const std::vector<float>& v) {
    field.off = (int)cbuf.size();
    cfix.push_back(&field);
    cbuf.insert(cbuf.end(), v.begin(), v.end());
    if (v.empty()) cbuf.push_back(0.f);
    while (cbuf.size() % 4) cbuf.push_back(0.f);
  }
  void finish() {
    const int ni = (int)pm.ibuf.size(), nf = (int)pm.fbuf.size();
    for (TabF* f : pm.ffix) f->off += ni;
    for (TabF* f : cfix) f->off += ni + nf;
    pm.tables.resize(pm.ibuf.size() + pm.fbuf.size() + cbuf.size());
    memcpy(pm.tables.data(), pm.ibuf.data(), pm.ibuf.size() * sizeof(int));
    memcpy(pm.tables.data() + ni, pm.fbuf.data(), pm.fbuf.size() * sizeof(float));
    memcpy(pm.tables.data() + ni + nf, cbuf.data(), cbuf.size() * sizeof(float));
    pm.dm.tab_words = ni + nf;      // the part staged into shared memory
  }
  std::vector<float> cbuf;
  std::vector<TabF*> cfix;
};

std::vector<int> ivec(const Model& m, const char* name) {
  const Array* a = m.arr(name);
  std::vector<int> v(a->count());
  if (a->dtype == DT_I32) { const int* p = a->as<int>(); for (size_t k = 0; k < v.size(); k++) v[k] = p[k]; }
  else if (a->dtype == DT_U8) { const uint8_t* p = a->as<uint8_t>(); for (size_t k = 0; k < v.size(); k++) v[k] = p[k]; }
  return v;
}
std::vector<float> fvec(const Model& m, const char* name) {
  const Array* a = m.arr(name);
  std::vector<float> v(a->count());
  const double* p = a->as<double>();
  for (size_t k = 0; k < v.size(); k++) v[k] = (float)p[k];
  return v;
}
// keep the first `keep` columns of a row-major [rows][cols] float table
std::vector<float> take_cols(const std::vector<float>& v, int rows, int cols, int keep) {
  std::vector<float> o((size_t)rows * keep);
  for (int r = 0; r < rows; r++) for (int c = 0; c < keep; c++) o[(size_t)r * keep + c] = v[(size_t)r * cols + c];
  return o;
}
void quat2mat_h(const double* q, float* R) {
  double q00 = q[0]*q[0], q01 = q[0]*q[1], q02 = q[0]*q[2], q03 = q[0]*q[3], q11 = q[1]*q[1], q12 = q[1]*q[2],
         q13 = q[1]*q[3], q22 = q[2]*q[2], q23 = q[2]*q[3], q33 = q[3]*q[3];
  R[0] = (float)(q00 + q11 - q22 - q33); R[4] = (float)(q00 - q11 + q22 - q33); R[8] = (float)(q00 - q11 - q22 + q33);
  R[1] = (float)(2*(q12 - q03)); R[2] = (float)(2*(q13 + q02)); R[3] = (float)(2*(q12 + q03));
  R[5] = (float)(2*(q23 - q01)); R[6] = (float)(2*(q13 - q02)); R[7] = (float)(2*(q23 + q01));
}
int pad4(int n) { return (n + 3) / 4 * 4; }

}  // namespace

std::string pack_model(const Model& m, const myo_task_cfg& cfg, PackedModel& out, int& status) {
  status = MYO_E_UNSUPPORTED;
  DevModel& d = out.dm;
  Builder B(out);
  const int nq = m.sz("nq"), nv = m.sz("nv"), nu = m.sz("nu"), na = m.sz("na"), nbody = m.sz("nbody"),
            njnt = m.sz("njnt"), ngeom = m.sz("ngeom"), nsite = m.sz("nsite"), ntendon = m.sz("ntendon"),
            nwrap = m.sz("nwrap"), nM = m.sz("nM");
  if (nv <= 0 || nbody <= 1) return "model has no degrees of freedom";
  if (m.sz("neq") > 0) return "equality constraints are outside the supported subset";
  if (m.sz("npair") > 0) return "explicit contact pairs (<contact><pair>) are outside the supported subset";
  if (na != 0 && na != nu) return "models mixing stateful and stateless actuators are outside the supported subset";
  if ((int)m.opt.at("integrator") != 0) return "only the Euler integrator is supported";
  if ((int)m.opt.at("cone") != 0) return "only pyramidal friction cones are supported";
  d.nq = nq; d.nv = nv; d.nu = nu; d.na = na; d.nbody = nbody; d.njnt = njnt; d.ngeom = ngeom; d.nsite = nsite;
  d.ntendon = ntendon; d.nwrap = nwrap; d.nM = nM;
  d.nq4 = pad4(nq); d.nv4 = pad4(nv); d.na4 = pad4(std::max(na, 1)); d.nu4 = pad4(std::max(nu, 1));
  d.timestep = (float)m.opt.at("timestep");
  d.gravity[0] = (float)m.opt.at("gravity0"); d.gravity[1] = (float)m.opt.at("gravity1"); d.gravity[2] = (float)m.opt.at("gravity2");
  d.inv_sqrt_impratio = (float)(1.0 / std::sqrt(std::max(1e-15, m.opt.at("impratio"))));
  d.meaninertia = (float)m.opt.at("meaninertia");
  d.solver_iter = cfg.solver_iterations > 0 ? cfg.solver_iterations : (int)m.opt.at("iterations");
  d.solver_tol = cfg.solver_tolerance > 0.f ? cfg.solver_tolerance : (float)m.opt.at("tolerance");
  d.frame_dt = (float)(std::max(1, cfg.frame_skip) * m.opt.at("timestep"));

  // ---------------------------------------------------------------- bodies
  std::vector<int> parent = ivec(m, "body_parentid"), rootid = ivec(m, "body_rootid"), weld = ivec(m, "body_weldid"),
                   jntnum = ivec(m, "body_jntnum"), jntadr = ivec(m, "body_jntadr"), dofnum = ivec(m, "body_dofnum"),
                   dofadr = ivec(m, "body_dofadr"), geomnum = ivec(m, "body_geomnum"), geomadr = ivec(m, "body_geomadr"),
                   sameframe = ivec(m, "body_sameframe");
  std::vector<int> jtype = ivec(m, "jnt_type"), jqadr = ivec(m, "jnt_qposadr"), jdadr = ivec(m, "jnt_dofadr"),
                   jbody = ivec(m, "jnt_bodyid"), jlimited = ivec(m, "jnt_limited");
  for (int j = 0; j < njnt; j++) {
    if (jtype[j] == J_BALL) return "ball joints are outside the supported subset";
    if (jtype[j] == J_FREE && jntnum[jbody[j]] != 1) return "a free joint must be the only joint of its body";
  }
  std::vector<int> dparent = ivec(m, "dof_parentid"), dbody = ivec(m, "dof_bodyid"), djnt = ivec(m, "dof_jntid"),
                   dMadr = ivec(m, "dof_Madr"), dsimple = ivec(m, "dof_simplenum");
  for (auto& s : dsimple) s = s ? 1 : 0;

  // levels (children of the world are level 0)
  std::vector<int> level(nbody, -1);
  int nlevel = 0;
  for (int b = 1; b < nbody; b++) { level[b] = level[parent[b]] + 1; nlevel = std::max(nlevel, level[b] + 1); }
  std::vector<int> lvl_adr(nlevel + 1, 0), lvl_body;
  for (int L = 0; L < nlevel; L++) {
    lvl_adr[L] = (int)lvl_body.size();
    for (int b = 1; b < nbody; b++) if (level[b] == L) lvl_body.push_back(b);
  }
  lvl_adr[nlevel] = (int)lvl_body.size();
  d.nlevel = nlevel;
  std::vector<int> childadr(nbody + 1, 0), child;
  for (int b = 0; b < nbody; b++) {
    childadr[b] = (int)child.size();
    if (b > 0) for (int c = b + 1; c < nbody; c++) if (parent[c] == b) child.push_back(c);
  }
  childadr[nbody] = (int)child.size();
  // dof chains, root first
  std::vector<int> nchain(nbody, 0), chain((size_t)nbody * KC, -1);
  for (int b = 1; b < nbody; b++) {
    int bb = b;
    while (bb && !dofnum[bb]) bb = parent[bb];
    if (!bb) continue;
    std::vector<int> c;
    for (int i = dofadr[bb] + dofnum[bb] - 1; i >= 0; i = dparent[i]) c.push_back(i);
    std::reverse(c.begin(), c.end());
    if ((int)c.size() > KC) { status = MYO_E_LIMIT; return "a body's dof chain exceeds the compiled-in maximum (KC)"; }
    nchain[b] = (int)c.size();
    for (size_t k = 0; k < c.size(); k++) chain[(size_t)b * KC + k] = c[k];
  }
  // dof depth / descendants / levels
  std::vector<int> ddepth(nv, 0);
  int ndlevel = 0;
  for (int i = 0; i < nv; i++) { ddepth[i] = dparent[i] < 0 ? 0 : ddepth[dparent[i]] + 1; ndlevel = std::max(ndlevel, ddepth[i] + 1); }
  for (int i = 0; i < nv; i++) {
    int expect = (i + 1 < nv ? dMadr[i + 1] : nM) - dMadr[i];
    if (expect != ddepth[i] + 1) return "dof_Madr layout does not match the dof tree";
  }
  std::vector<int> descadr(nv + 1, 0), desc;
  for (int i = 0; i < nv; i++) {
    descadr[i] = (int)desc.size();
    for (int k = i + 1; k < nv; k++) {
      int a = dparent[k];
      while (a >= 0 && a != i) a = dparent[a];
      if (a == i) desc.push_back(k);
    }
  }
  descadr[nv] = (int)desc.size();
  std::vector<int> dlvl_adr(ndlevel + 1, 0), dlvl_dof;
  for (int L = 0; L < ndlevel; L++) {
    dlvl_adr[L] = (int)dlvl_dof.size();
    for (int i = 0; i < nv; i++) if (ddepth[i] == L) dlvl_dof.push_back(i);
  }
  dlvl_adr[ndlevel] = (int)dlvl_dof.size();
  d.ndlevel = ndlevel;

  // ---------------------------------------------------------------- override slots
  std::vector<int> mass_slot(nbody, -1), pose_slot(nbody, -1), size_slot(ngeom, -1), fri_slot(ngeom, -1), spos_slot(nsite, -1);
  {
    int np = 0;
    const double* bm = m.d("body_mass"); const double* gs = m.d("geom_size"); const double* gf = m.d("geom_friction");
    const double* sp = m.d("site_pos");
    for (int k = 0; k < cfg.n_ovr_body && k < MYO_MAX_OVERRIDE; k++) {
      int b = cfg.ovr_body[k];
      if (b < 0 || b >= nbody) { status = MYO_E_ARG; return "override body id out of range"; }
      mass_slot[b] = np; out.slots.push_back({MYO_PARAM_BODY_MASS, b, np, 1});
      out.param0.push_back((float)bm[b]); np += 1;
    }
    for (int k = 0; k < cfg.n_ovr_geom && k < MYO_MAX_OVERRIDE; k++) {
      int g = cfg.ovr_geom[k];
      if (g < 0 || g >= ngeom) { status = MYO_E_ARG; return "override geom id out of range"; }
      size_slot[g] = np; out.slots.push_back({MYO_PARAM_GEOM_SIZE, g, np, 3});
      for (int e = 0; e < 3; e++) out.param0.push_back((float)gs[3 * g + e]);
      np += 3;
      fri_slot[g] = np; out.slots.push_back({MYO_PARAM_GEOM_FRICTION, g, np, 3});
      for (int e = 0; e < 3; e++) out.param0.push_back((float)gf[3 * g + e]);
      np += 3;
    }
    // reach: the target sites are the per-world site overrides (reset draws them)
    const bool reach = cfg.kind == MYO_TASK_REACH;
    for (int k = 0; k < (reach ? cfg.reach_nsite : cfg.n_ovr_site) && k < MYO_MAX_OVERRIDE; k++) {
      int s = reach ? cfg.reach_target_site[k] : cfg.ovr_site[k];
      if (s < 0 || s >= nsite) { status = MYO_E_ARG; return "override site id out of range"; }
      spos_slot[s] = np; out.slots.push_back({MYO_PARAM_SITE_POS, s, np, 3});
      for (int e = 0; e < 3; e++) out.param0.push_back((float)sp[3 * s + e]);
      np += 3;
    }
    for (int k = 0; k < cfg.n_ovr_bodypose && k < MYO_MAX_OVERRIDE; k++) {      // body_pos (3) followed by the matrix of body_quat (9)
      int b = cfg.ovr_bodypose[k];
      if (b <= 0 || b >= nbody) { status = MYO_E_ARG; return "override body (pose) id out of range"; }
      pose_slot[b] = np; out.slots.push_back({MYO_PARAM_BODY_POS, b, np, 3}); out.slots.push_back({MYO_PARAM_BODY_MAT, b, np + 3, 9});
      const double* bp = m.d("body_pos") + 3 * b;
      for (int e = 0; e < 3; e++) out.param0.push_back((float)bp[e]);
      float R[9];
      quat2mat_h(m.d("body_quat") + 4 * b, R);
      for (int e = 0; e < 9; e++) out.param0.push_back(R[e]);
      np += 12;
    }
    d.nparam = np; d.nparam4 = pad4(std::max(np, 1));
    out.param0.resize(d.nparam4, 0.f);
  }

  B.I(d.b_parent, parent); B.I(d.b_root, rootid); B.I(d.b_jntadr, jntadr); B.I(d.b_jntnum, jntnum);
  B.I(d.b_dofadr, dofadr); B.I(d.b_dofnum, dofnum); B.I(d.b_nchain, nchain); B.I(d.b_chain, chain);
  B.I(d.b_mass_slot, mass_slot); B.I(d.b_pose_slot, pose_slot); B.I(d.b_sameframe, sameframe);
  B.I(d.lvl_adr, lvl_adr); B.I(d.lvl_body, lvl_body);
  {   // subtree of every body (itself first, then its descendants in body order): composite inertia / force sums
    std::vector<int> subadr(nbody + 1, 0), sub;
    for (int b = 0; b < nbody; b++) {
      subadr[b] = (int)sub.size();
      for (int k = b; k < nbody; k++) {
        int a = k;
        while (a > b) a = parent[a];
        if (a == b && (b > 0 || k == 0)) sub.push_back(k);
      }
    }
    subadr[nbody] = (int)sub.size();
    B.I(d.b_subadr, subadr); B.I(d.b_sub, sub);
  }
  {   // body frame / inertial frame orientations as matrices: the kinematic sweep composes rotation matrices
    std::vector<float> bmat((size_t)nbody * 9), bimat((size_t)nbody * 9);
    const double* bq = m.d("body_quat"); const double* biq = m.d("body_iquat");
    for (int b = 0; b < nbody; b++) { quat2mat_h(bq + 4 * b, bmat.data() + 9 * b); quat2mat_h(biq + 4 * b, bimat.data() + 9 * b); }
    B.F(d.b_mat, bmat); B.F(d.b_imat, bimat);
  }
  B.F(d.b_pos, fvec(m, "body_pos")); B.F(d.b_ipos, fvec(m, "body_ipos"));
  B.F(d.b_mass, fvec(m, "body_mass")); B.F(d.b_inertia, fvec(m, "body_inertia"));
  B.F(d.b_invweight0, fvec(m, "body_invweight0"));

  // ---------------------------------------------------------------- joints / dofs
  {
    const double* q0 = m.d("qpos0"); const double* qs = m.d("qpos_spring"); const double* st = m.d("jnt_stiffness");
    std::vector<float> jq0(njnt), jqs(njnt);
    int any_spring = 0;
    for (int j = 0; j < njnt; j++) { jq0[j] = (float)q0[jqadr[j]]; jqs[j] = (float)qs[jqadr[j]]; if (st[j] != 0) any_spring = 1; }
    d.any_joint_spring = any_spring;
    B.I(d.j_type, jtype); B.I(d.j_qposadr, jqadr); B.I(d.j_dofadr, jdadr); B.I(d.j_body, jbody); B.I(d.j_limited, jlimited);
    B.F(d.j_pos, fvec(m, "jnt_pos")); B.F(d.j_axis, fvec(m, "jnt_axis")); B.F(d.j_qpos0, jq0);
    B.F(d.j_range, fvec(m, "jnt_range")); B.F(d.j_margin, fvec(m, "jnt_margin")); B.F(d.j_solref, fvec(m, "jnt_solref"));
    B.F(d.j_solimp, fvec(m, "jnt_solimp")); B.F(d.j_stiffness, fvec(m, "jnt_stiffness")); B.F(d.j_qpos_spring, jqs);
  }
  {
    const double* dl = m.d("dof_frictionloss");
    for (int i = 0; i < nv; i++) if (dl[i] != 0) return "dof frictionloss is outside the supported subset";
    const double* dd = m.d("dof_damping");
    d.any_damping = 0;
    for (int i = 0; i < nv; i++) if (dd[i] > 0) d.any_damping = 1;
  }

  // ---------------------------------------------------------------- geoms + collision candidates
  std::vector<int> gtype = ivec(m, "geom_type"), gbody = ivec(m, "geom_bodyid"), gcontype = ivec(m, "geom_contype"),
                   gconaff = ivec(m, "geom_conaffinity");
  {
    std::vector<float> gmat((size_t)ngeom * 9);
    const double* gq = m.d("geom_quat");
    for (int g = 0; g < ngeom; g++) quat2mat_h(gq + 4 * g, gmat.data() + 9 * g);
    B.I(d.g_type, gtype); B.I(d.g_body, gbody); B.I(d.g_condim, ivec(m, "geom_condim"));
    B.I(d.g_priority, ivec(m, "geom_priority")); B.I(d.g_size_slot, size_slot); B.I(d.g_fri_slot, fri_slot);
    B.F(d.g_pos, fvec(m, "geom_pos")); B.F(d.g_mat, gmat); B.F(d.g_size, fvec(m, "geom_size"));
    B.F(d.g_rbound, fvec(m, "geom_rbound")); B.F(d.g_friction, fvec(m, "geom_friction"));
    B.F(d.g_solmix, fvec(m, "geom_solmix")); B.F(d.g_solref, fvec(m, "geom_solref")); B.F(d.g_solimp, fvec(m, "geom_solimp"));
    B.F(d.g_margin, fvec(m, "geom_margin")); B.F(d.g_gap, fvec(m, "geom_gap"));
  }
  std::vector<int> p_g1, p_g2, p_sup;
  std::vector<int> excl = m.sz("nexclude") > 0 ? ivec(m, "exclude_signature") : std::vector<int>();
  for (int b1 = 0; b1 < nbody; b1++) for (int b2 = b1 + 1; b2 < nbody; b2++) {
    if (!geomnum[b1] || !geomnum[b2]) continue;
    const int w1 = weld[b1], w2 = weld[b2];
    const int wp1 = weld[parent[w1]], wp2 = weld[parent[w2]];
    if (w1 == w2) continue;
    if (w1 != 0 && w2 != 0 && (w1 == wp2 || w2 == wp1)) continue;
    if (std::find(excl.begin(), excl.end(), (b1 << 16) + b2) != excl.end()) continue;      // <contact><exclude body1 body2>
    for (int ga = geomadr[b1]; ga < geomadr[b1] + geomnum[b1]; ga++)
      for (int gb = geomadr[b2]; gb < geomadr[b2] + geomnum[b2]; gb++) {
        int g1 = ga, g2 = gb;
        if (gtype[g1] > gtype[g2]) std::swap(g1, g2);
        if (!((gcontype[g1] & gconaff[g2]) || (gcontype[g2] & gconaff[g1]))) continue;
        const int t1 = gtype[g1], t2 = gtype[g2];
        const bool sup = (t1 == G_SPHERE && t2 == G_SPHERE) || (t1 == G_SPHERE && t2 == G_CAPSULE) ||
                         (t1 == G_PLANE && t2 == G_SPHERE) || (t1 == G_CAPSULE && t2 == G_BOX);
        p_g1.push_back(g1); p_g2.push_back(g2); p_sup.push_back(sup ? 1 : 0);
        if (t1 == G_CAPSULE && t2 == G_BOX) {      // up to two contacts: the pair is listed twice, p_supported = 1 + contact number
          p_sup.back() = 1;
          p_g1.push_back(g1); p_g2.push_back(g2); p_sup.push_back(2);
        }
      }
  }
  d.npair = (int)p_g1.size();
  B.I(d.p_g1, p_g1); B.I(d.p_g2, p_g2); B.I(d.p_supported, p_sup);

  // ---------------------------------------------------------------- sites
  std::vector<int> sbody = ivec(m, "site_bodyid");
  B.I(d.s_body, sbody); B.I(d.s_pos_slot, spos_slot); B.F(d.s_pos, fvec(m, "site_pos"));

  // ---------------------------------------------------------------- tendons
  std::vector<int> tadr = ivec(m, "tendon_adr"), tnum = ivec(m, "tendon_num"), wtype = ivec(m, "wrap_type"),
                   wobj = ivec(m, "wrap_objid");
  std::vector<int> wside(nwrap, -1), tndof(ntendon, 0), tdof((size_t)ntendon * KT, -1);
  {
    const double* wprm = m.d("wrap_prm");
    auto common_prefix = [&](int ba, int bb) {
      if (rootid[ba] != rootid[bb]) return 0;
      int cp = 0;
      while (cp < nchain[ba] && cp < nchain[bb] && chain[(size_t)ba * KC + cp] == chain[(size_t)bb * KC + cp]) cp++;
      return cp;
    };
    for (int t = 0; t < ntendon; t++) {
      std::set<int> sup;
      auto add_seg = [&](int ba, int bb) {
        if (ba == bb) return;
        const int cp = common_prefix(ba, bb);
        for (int k = cp; k < nchain[ba]; k++) sup.insert(chain[(size_t)ba * KC + k]);
        for (int k = cp; k < nchain[bb]; k++) sup.insert(chain[(size_t)bb * KC + k]);
      };
      const int adr = tadr[t], num = tnum[t];
      if (num < 2) return "tendon with fewer than two wrap objects";
      if (wtype[adr] == 1) return "fixed (joint) tendons are outside the supported subset";
      int j = 0;
      while (j < num - 1) {
        const int tp0 = wtype[adr + j], tp1 = wtype[adr + j + 1];
        if (tp0 == W_PULLEY || tp1 == W_PULLEY) { j++; continue; }
        if (tp0 != W_SITE) return "malformed tendon path (segment must start at a site)";
        const int b0 = sbody[wobj[adr + j]];
        if (tp1 == W_SPHERE || tp1 == W_CYLINDER) {
          if (j + 2 >= num || wtype[adr + j + 2] != W_SITE) return "malformed tendon path (wrap geom must be followed by a site)";
          const int g = wobj[adr + j + 1];
          const int side = (int)std::lround(wprm[adr + j + 1]);
          wside[adr + j + 1] = (side >= 0 && side < nsite) ? side : -1;
          const int bw = gbody[g], b1 = sbody[wobj[adr + j + 2]];
          add_seg(b0, b1); add_seg(b0, bw); add_seg(bw, b1);
          j += 2;
        } else {
          add_seg(b0, sbody[wobj[adr + j + 1]]);
          j += 1;
        }
      }
      if ((int)sup.size() > KT) { status = MYO_E_LIMIT; return "a tendon touches more dofs than the compiled-in maximum (KT)"; }
      tndof[t] = (int)sup.size();
      int e = 0;
      for (int dof : sup) tdof[(size_t)t * KT + e++] = dof;
    }
    int any_tp = 0;
    const double* ts = m.d("tendon_stiffness"); const double* td = m.d("tendon_damping"); const double* tf = m.d("tendon_frictionloss");
    for (int t = 0; t < ntendon; t++) {
      if (ts[t] != 0 || td[t] != 0) any_tp = 1;
      if (tf[t] != 0) return "tendon frictionloss is outside the supported subset";
    }
    d.any_tendon_passive = any_tp;
  }
  // segment tasks of the tendon phase: one record per path segment (site -> site, or site -> wrap geom -> site), wrap
  // segments first so the divergent wrap geometry shares one pass; moment-arm lists per (body, body) pair:
  // header n | rootA << 8 | rootB << 20, then n entries dof | slot << 8 | end << 16 (slot in the tendon's dof list)
  std::vector<int> seg_rec, seg_list, t_segadr(ntendon + 1, 0), t_seg;
  std::vector<float> seg_invdiv;
  {
    const double* wprm = m.d("wrap_prm");
    auto make_list = [&](int t, int ba, int bb) -> int {
      if (ba == bb) return -1;
      int cp = 0;
      if (rootid[ba] == rootid[bb])
        while (cp < nchain[ba] && cp < nchain[bb] && chain[(size_t)ba * KC + cp] == chain[(size_t)bb * KC + cp]) cp++;
      const int adr = (int)seg_list.size();
      seg_list.push_back(0);
      int n = 0;
      for (int end = 0; end < 2; end++) {
        const int body = end ? bb : ba;
        for (int k = cp; k < nchain[body]; k++) {
          const int dof = chain[(size_t)body * KC + k];
          int slot = -1;
          for (int e = 0; e < tndof[t]; e++) if (tdof[(size_t)t * KT + e] == dof) slot = e;
          seg_list.push_back(dof | (slot << 8) | (end << 16));
          n++;
        }
      }
      seg_list[adr] = n | (rootid[ba] << 8) | (rootid[bb] << 20);
      return adr;
    };
    struct Seg { int t, type, s0, s1, g, side, l0, l1, l2; float inv_div; };
    std::vector<Seg> segs;
    for (int t = 0; t < ntendon; t++) {
      const int adr = tadr[t], num = tnum[t];
      float inv_div = 1.f;
      int j = 0;
      while (j < num - 1) {
        const int tp0 = wtype[adr + j], tp1 = wtype[adr + j + 1];
        if (tp0 == W_PULLEY || tp1 == W_PULLEY) {
          if (tp0 == W_PULLEY) inv_div = (float)(1.0 / wprm[adr + j]);
          j++;
          continue;
        }
        Seg sg{};
        sg.t = t; sg.s0 = wobj[adr + j]; sg.inv_div = inv_div; sg.g = -1; sg.side = -1; sg.l1 = sg.l2 = -1; sg.type = 0;
        const int b0 = sbody[sg.s0];
        if (tp1 == W_SPHERE || tp1 == W_CYLINDER) {
          sg.type = tp1; sg.g = wobj[adr + j + 1]; sg.side = wside[adr + j + 1]; sg.s1 = wobj[adr + j + 2];
          const int bw = gbody[sg.g], b1 = sbody[sg.s1];
          sg.l0 = make_list(t, b0, b1); sg.l1 = make_list(t, b0, bw); sg.l2 = make_list(t, bw, b1);
          j += 2;
        } else {
          sg.s1 = wobj[adr + j + 1];
          sg.l0 = make_list(t, b0, sbody[sg.s1]);
          j += 1;
        }
        segs.push_back(sg);
      }
    }
    std::vector<int> order;
    for (int k = 0; k < (int)segs.size(); k++) if (segs[k].type != 0) order.push_back(k);
    for (int k = 0; k < (int)segs.size(); k++) if (segs[k].type == 0) order.push_back(k);
    std::vector<int> newid(segs.size(), 0);
    for (int k = 0; k < (int)order.size(); k++) newid[order[k]] = k;
    if (seg_list.size() >= (1u << 16) || nbody >= 4096 || nv >= 256) { status = MYO_E_LIMIT; return "tendon segment tables exceed their packed field widths"; }
    for (int k : order) {
      const Seg& sg = segs[k];
      seg_rec.insert(seg_rec.end(), {sg.t | (sg.type << 16), sg.s0, sg.s1, sg.g, sg.side, sg.l0, sg.l1, sg.l2});
      seg_invdiv.push_back(sg.inv_div);
    }
    for (int t = 0, k = 0; t < ntendon; t++) {
      t_segadr[t] = (int)t_seg.size();
      for (; k < (int)segs.size() && segs[k].t == t; k++) t_seg.push_back(newid[k]);
    }
    t_segadr[ntendon] = (int)t_seg.size();
    d.nseg = (int)segs.size();
  }
  B.I(d.seg_rec, seg_rec); B.I(d.seg_list, seg_list); B.I(d.t_segadr, t_segadr); B.I(d.t_seg, t_seg); B.F(d.seg_invdiv, seg_invdiv);
  B.I(d.t_limited, ivec(m, "tendon_limited")); B.I(d.t_ndof, tndof); B.I(d.t_dof, tdof);
  B.F(d.t_range, fvec(m, "tendon_range")); B.F(d.t_margin, fvec(m, "tendon_margin")); B.F(d.t_solref, fvec(m, "tendon_solref_lim"));
  B.F(d.t_solimp, fvec(m, "tendon_solimp_lim")); B.F(d.t_invweight0, fvec(m, "tendon_invweight0"));
  B.F(d.t_stiffness, fvec(m, "tendon_stiffness")); B.F(d.t_damping, fvec(m, "tendon_damping"));
  B.F(d.t_lengthspring, fvec(m, "tendon_lengthspring"));

  // ---------------------------------------------------------------- actuators
  std::vector<int> atendon(nu, 0);
  {
    std::vector<int> trntype = ivec(m, "actuator_trntype"), trnid = ivec(m, "actuator_trnid");
    for (int i = 0; i < nu; i++) {
      if (trntype[i] != 3) return "only tendon transmissions are supported";
      atendon[i] = trnid[2 * i];
    }
    std::vector<float> gear = take_cols(fvec(m, "actuator_gear"), nu, 6, 1);
    B.I(d.a_tendon, atendon); B.I(d.a_dyntype, ivec(m, "actuator_dyntype")); B.I(d.a_gaintype, ivec(m, "actuator_gaintype"));
    B.I(d.a_biastype, ivec(m, "actuator_biastype")); B.I(d.a_ctrllimited, ivec(m, "actuator_ctrllimited"));
    B.I(d.a_forcelimited, ivec(m, "actuator_forcelimited"));
    B.Fcold(d.a_dynprm, take_cols(fvec(m, "actuator_dynprm"), nu, 10, 3));
    B.Fcold(d.a_gainprm, take_cols(fvec(m, "actuator_gainprm"), nu, 10, 9));
    B.Fcold(d.a_biasprm, take_cols(fvec(m, "actuator_biasprm"), nu, 10, 9));
    B.Fcold(d.a_ctrlrange, fvec(m, "actuator_ctrlrange")); B.Fcold(d.a_forcerange, fvec(m, "actuator_forcerange"));
    B.Fcold(d.a_gear, gear); B.Fcold(d.a_acc0, fvec(m, "actuator_acc0")); B.Fcold(d.a_lengthrange, fvec(m, "actuator_lengthrange"));
  }
  // per-dof actuator gather list: code = actuator << 8 | slot in the tendon's dof list
  std::vector<int> actadr(nv + 1, 0), actlist;
  for (int dof = 0; dof < nv; dof++) {
    actadr[dof] = (int)actlist.size();
    for (int a = 0; a < nu; a++) {
      const int t = atendon[a];
      for (int e = 0; e < tndof[t]; e++) if (tdof[(size_t)t * KT + e] == dof) actlist.push_back((a << 8) | e);
    }
  }
  actadr[nv] = (int)actlist.size();
  B.I(d.d_body, dbody); B.I(d.d_parent, dparent); B.I(d.d_simple, dsimple); B.I(d.d_Madr, dMadr); B.I(d.d_depth, ddepth);
  B.I(d.d_jnt, djnt);
  {   // full symmetric rows of the mass matrix for mj_mulM: entry = column | index into qM << 8, columns ascending
    std::vector<int> radr(nv + 1, 0), rlist;
    for (int i = 0; i < nv; i++) {
      radr[i] = (int)rlist.size();
      std::vector<std::pair<int, int>> ent;
      { int adr = dMadr[i], j = i; while (j >= 0) { ent.push_back({j, adr++}); j = dparent[j]; } }       // i and its ancestors
      if (!dsimple[i])
        for (int k = descadr[i]; k < descadr[i + 1]; k++) { const int dk = desc[k]; ent.push_back({dk, dMadr[dk] + ddepth[dk] - ddepth[i]}); }
      std::sort(ent.begin(), ent.end());
      for (auto& e : ent) {
        if (e.second >= (1 << 23)) { status = MYO_E_LIMIT; return "mass matrix too large for the packed row table"; }
        rlist.push_back(e.first | (e.second << 8));
      }
    }
    radr[nv] = (int)rlist.size();
    B.I(d.m_rowadr, radr); B.I(d.m_row, rlist);
  }
  {   // dofs whose motion precedes dof i when mj_comVel forms cdof_dot_i = cvel_so_far x cdof_i: the dofs before it on its
      // chain - except the rotational dofs of a free joint, which see the joint's three translations only
    std::vector<int> prefadr(nv + 1, 0), pref;
    for (int i = 0; i < nv; i++) {
      prefadr[i] = (int)pref.size();
      const int j = djnt[i], body = dbody[i];
      if (jtype[j] == J_FREE) {
        const int d0 = jdadr[j];
        if (i >= d0 + 3) for (int k = d0; k < d0 + 3; k++) pref.push_back(k);
      } else {
        for (int k = 0; k < nchain[body]; k++) { const int dk = chain[(size_t)body * KC + k]; if (dk < i) pref.push_back(dk); }
      }
    }
    prefadr[nv] = (int)pref.size();
    B.I(d.d_prefadr, prefadr); B.I(d.d_pref, pref);
  }
  B.I(d.d_actadr, actadr); B.I(d.d_actlist, actlist);
  B.F(d.d_armature, fvec(m, "dof_armature")); B.F(d.d_damping, fvec(m, "dof_damping"));
  B.F(d.d_invweight0, fvec(m, "dof_invweight0")); B.F(d.d_M0, fvec(m, "dof_M0"));

  // ---------------------------------------------------------------- task-dependent sizes
  // canonical observation (task_obs): the default obs_keys of the kind, each key's (first word, width) in it
  std::vector<std::pair<int, int>> keys;      // indexed by MYO_OBS_<KIND>_* id; {-1, 1}: t
  if (cfg.kind == MYO_TASK_BAODING) {
    const int nh = nq - 14;
    d.nobs_scr = nh + 24 + na;
    keys = {{-1, 1}, {0, nh}};
    for (int k = 0; k < 8; k++) keys.push_back({nh + 3 * k, 3});      // object1_pos .. target2_err
    keys.push_back({nh + 24, na});
  } else if (cfg.kind == MYO_TASK_POSE) {
    d.nobs_scr = nq + nv + nq + na;
    keys = {{-1, 1}, {0, nq}, {nq, nv}, {2 * nq + nv, na}, {nq + nv, nq}};      // t qpos qvel act pose_err
  } else if (cfg.kind == MYO_TASK_REORIENT) {
    const int nh = nq - 7, nhv = nv - 6, o0 = nh + nhv;
    d.nobs_scr = o0 + 18 + na;
    keys = {{-1, 1}, {0, nh}, {nh, nhv}};
    for (int k = 0; k < 6; k++) keys.push_back({o0 + 3 * k, 3});       // obj_pos .. rot_err
    keys.push_back({o0 + 18, na});
  } else if (cfg.kind == MYO_TASK_REACH) {
    const int o0 = nq + nv, w3 = 3 * cfg.reach_nsite;      // qpos qvel*dt tip_pos reach_err act
    d.nobs_scr = o0 + 2 * w3 + na;
    keys = {{-1, 1}, {0, nq}, {nq, nv}, {o0 + 2 * w3, na}, {o0, w3}, {-2, w3}, {o0 + w3, w3}};   // target_pos = tip_pos + reach_err
  } else {
    d.nobs_scr = nq + nv + na;
  }
  d.nobs = d.nobs_scr;
  d.nobs_run = 0;
  if (cfg.n_obs_keys != 0) {
    if (cfg.n_obs_keys < 0 || cfg.n_obs_keys > MYO_MAX_OBS_KEYS) { status = MYO_E_LIMIT; return "obs_keys: 1 .. MYO_MAX_OBS_KEYS keys"; }
    if (keys.empty()) { status = MYO_E_ARG; return "obs_keys: this task kind has no observation keys"; }
    d.nobs = 0;
    for (int k = 0; k < cfg.n_obs_keys; k++) {
      const int id = cfg.obs_keys[k];
      if (id < 0 || id >= (int)keys.size()) {
        status = MYO_E_ARG;
        return "obs_keys: key id " + std::to_string(id) + " is not one of this task kind's " + std::to_string(keys.size()) + " keys";
      }
      int src = keys[id].first, width = keys[id].second, op = OBS_RUN_COPY;
      if (src == -1) { src = 0; op = OBS_RUN_TIME; }
      else if (src == -2) { src = nq + nv; op = OBS_RUN_SUM; }
      d.nobs += width;
      if (width == 0) continue;
      if (d.nobs_run > 0 && op == OBS_RUN_COPY) {
        int& last = d.obs_run[d.nobs_run - 1];
        const int lw = (last >> 16) & 0xfff;
        if ((last >> 28) == OBS_RUN_COPY && (last & 0xffff) + lw == src && lw + width < 0x1000) {
          last += width << 16;      // continues the previous run
          continue;
        }
      }
      if (src >= 0x10000 || width >= 0x1000) { status = MYO_E_LIMIT; return "obs_keys: observation too wide for the gather table"; }
      d.obs_run[d.nobs_run++] = src | (width << 16) | (op << 28);
    }
  }
  d.nobs4 = pad4(d.nobs);
  {
    const double* q0 = m.d("qpos0");
    out.init_qpos.assign(d.nq4, 0.f);
    for (int k = 0; k < nq; k++) out.init_qpos[k] = (float)q0[k];
    if (cfg.kind == MYO_TASK_BAODING) {   // CustomBaodingP2Env._setup: init_qpos[:-14] = 0; init_qpos[0] = -1.57
      for (int k = 0; k < nq - 14; k++) out.init_qpos[k] = 0.f;
      out.init_qpos[0] = -1.57f;
    }
    if (cfg.kind == MYO_TASK_REORIENT) {   // CustomReorientEnv._setup: init_qpos[:-7] = 0; init_qpos[0] = -1.5 (/root/reference/src/envs/reorient.py:123-124)
      for (int k = 0; k < nq - 7; k++) out.init_qpos[k] = 0.f;
      out.init_qpos[0] = -1.5f;
    }
    B.F(d.init_qpos, out.init_qpos);
    B.F(d.param0, out.param0);
  }

  // ---------------------------------------------------------------- capacities + scratch layout
  // Two layouts of the same tables: the FAST one (out.dm) keeps a world small enough that many share an SM - 16 contacts, 32
  // limit rows - and the FULL one (out.dm_full) has MuJoCo's own capacities (nconmax contacts, njmax rows). A world that
  // outgrows the fast layout during an env step is stepped again, from the same state, by the full-capacity kernel
  // (myo_kernels.cu: redo list), so the capacities are a performance knob, never a change of results.
  int nlim = 0;      // limited joints + tendons; each can raise a row on either side (both at once only if its range is narrower than 2 x margin)
  for (int j = 0; j < njnt; j++) if (jlimited[j] && (jtype[j] == J_HINGE || jtype[j] == J_SLIDE)) nlim++;
  d.any_tendon_limit = 0;
  { std::vector<int> tl = ivec(m, "tendon_limited"); for (int t = 0; t < ntendon; t++) if (tl[t]) { nlim++; d.any_tendon_limit = 1; } }
  if (nv > 64) { status = MYO_E_LIMIT; return "nv exceeds the dense solver limit (64)"; }
  out.lanes = nv <= 8 ? 8 : (nv <= 16 ? 16 : 32);
  if (const char* ov = getenv("MYO_LANES")) {   // test hook: override of the tile width (8, 16 or 32), so that tests cover every instantiation
    const int g = atoi(ov);
    if (g == 8 || g == 16 || g == 32) out.lanes = g;
  }
  {
    d.nd = 0;
    for (int i = 0; i < nv; i++) if (!dsimple[i]) d.nd = i + 1;
    // dense Hessian, lower triangle by rows: rows 4a..4a+3 have the same length, ((a + 1) | 1) float4s (odd, so the four
    // rows of a group start on different banks); one more row (pad4(nv) words) for the right-hand side
    const int n4 = pad4(nv);
    std::vector<int> roff(n4 + 1, 0);
    int hw = 0;
    for (int i = 0; i < n4; i++) { roff[i] = hw; hw += 4 * ((i / 4 + 1) | 1); }
    roff[n4] = hw;
    B.I(d.h_roff, roff);
    // (a, b), a >= b, of pair e = a (a + 1) / 2 + b for the contact blocks of the Hessian: a | b << 8
    std::vector<int> pair_ab;
    for (int a = 0; a < KS; a++) for (int b2 = 0; b2 <= a; b2++) pair_ab.push_back(a | (b2 << 8));
    B.I(d.pair_ab, pair_ab);
  }
  const int ncon_fast = 16, nlim_fast = 32;      // fast-layout capacities
  B.finish();
  const int njmax = std::max(1, m.sz("njmax")), nconmax = std::max(1, m.sz("nconmax"));
  // alias: the fast layout, which only the env step (and reset / get_obs, which run no physics) uses. Words of vectors
  // whose lifetimes within a substep do not overlap are shared, so that more worlds fit an SM. The substep runs
  //   tree_forward -> mass_bias -> tendon -> collision -> constraints -> actuation -> (qacc_smooth) -> solve -> integrate
  // and the shared groups are
  //   * solver vectors (solve .. integrate), observation (after the last substep), qfrc_bias (mass_bias .. actuation) and
  //     ten_length / ten_velocity (tendon .. actuation);
  //   * Newton Hessian (solve, and the M solves after actuation and in integrate) with xpos / xmat (tree_forward ..
  //     collision, and the task's kinematics after the last substep), beside them the velocity-stage temporaries
  //     (tree_forward .. mass_bias), the tendon phase's per-segment results and actuator force / qfrc_actuator /
  //     qfrc_passive (actuation; never read after it).
  // The full layout keeps every field in words of its own: the stage dumps of forward / mj_step read it.
  auto layout = [&](DevModel& dd, bool alias, int nlim_sides, int nlim_cap, int ncon_cap, int nefc_cap) {
    dd.nlim_max = std::max(1, std::min(nlim * nlim_sides, nlim_cap));
    dd.ncon_max = std::max(1, std::min(dd.npair, ncon_cap));
    dd.nefc_max = std::min(dd.nlim_max + 4 * dd.ncon_max, nefc_cap);
    int off = 0;
    auto take = [&](int words) { int o = off; off += pad4(std::max(words, 1)); return o; };
    dd.o_qpos = take(nq); dd.o_qvel = take(nv); dd.o_act = take(na); dd.o_ctrl = take(nu); dd.o_warm = take(nv);
    dd.o_wparam = take(dd.nparam4);
    if (!alias) { dd.o_xpos = take(3 * nbody); dd.o_xmat = take(9 * nbody); }
    dd.o_xipos = take(3 * nbody);
    dd.o_cdof = take(6 * nv);
    dd.o_M = take(nM);
    if (!alias) { dd.o_tenL = take(ntendon); dd.o_tenV = take(ntendon); }
    dd.o_tenJ = take(ntendon * KT);
    if (!alias) { dd.o_actF = take(nu); dd.o_bias = take(nv); dd.o_passive = take(nv); dd.o_qact = take(nv); }
    dd.o_smooth = take(nv); dd.o_qaccs = take(nv);
    dd.o_qacc = take(nv); dd.o_qcon = take(nv); dd.o_actdot = take(na);
    // solver vectors; the observation (assembled after the last substep, when they are dead) shares their words
    {
      const int a0 = off;
      dd.o_grad = take(nv); dd.o_p = take(nv); dd.o_Mp = take(nv); dd.o_Ma = take(nv);
      int words = off - a0;
      if (alias) {
        off = a0;
        dd.o_bias = take(nv); dd.o_tenL = take(ntendon); dd.o_tenV = take(ntendon);
        words = std::max(words, off - a0);
      }
      dd.o_obs = a0;
      off = a0 + std::max(words, pad4(dd.nobs_scr));
    }
    dd.o_misc = take(MI_WORDS);
    // velocity-stage temporaries and the composite inertias are dead once M and qfrc_bias exist; the Newton Hessian
    // (and the tendon phase's per-segment results) reuse their words
    {
      const int a0 = off;
      dd.o_H = a0;
      const int n4 = pad4(nv);
      int hw = 0;
      for (int i = 0; i < n4; i++) hw += 4 * ((i / 4 + 1) | 1);
      hw += n4;
      if (alias) { dd.o_xpos = take(3 * nbody); dd.o_xmat = take(9 * nbody); }
      const int a1 = off;      // from here on: words that are dead while the world's kinematics are live
      dd.o_cdofdot = take(6 * nv); dd.o_cfrc = take(6 * nbody);
      dd.o_cinert = take(10 * nbody);
      int end = off;
      if (alias) {
        off = a1;
        dd.o_actF = take(nu); dd.o_passive = take(nv); dd.o_qact = take(nv);
        end = std::max(end, off);
      }
      dd.o_seg = a1;
      off = std::max(end, a0 + hw);
      // limit / contact / row records follow directly: the tendon phase runs before they are rebuilt, so its per-segment
      // results may run on from the Hessian's words into theirs
      dd.o_lim = take(dd.nlim_max * LIM_WORDS); dd.o_con = take(dd.ncon_max * CON_WORDS); dd.o_row = take(dd.nefc_max * ROW_WORDS);
      off = std::max(off, a1 + pad4(dd.nseg * SEG_OUT));
    }
    // world stride: tiles of one warp land on different banks
    if (out.lanes < 32) { while (off % 32 != out.lanes) off += 4; }
    else if (off % 32 == 0) off += 4;
    dd.scratch_words = off;
  };
  layout(d, true, 1, nlim_fast, ncon_fast, nlim_fast + 4 * ncon_fast);
  out.dm_full = d;
  // full capacities, bounded by what the solo kernel keeps in registers per lane (kSoloRowsPerLane rows)
  layout(out.dm_full, false, 2, njmax, nconmax, std::min(njmax, kSoloRowsPerLane * out.lanes));
  status = MYO_OK;
  return "";
}

// Every feature of a model that keeps it outside the supported subset, one line each (empty: it runs). Unlike pack_model,
// which stops at the first obstacle, this walks the whole model: a user holding the real myo_hand_*.mjb learns in one call
// what stands between the file and the kernels.
std::string check_model(const Model& m) {
  std::string out;
  auto add = [&](const std::string& line) { out += "- " + line + "\n"; };
  const int nv = m.sz("nv"), nu = m.sz("nu"), na = m.sz("na"), nbody = m.sz("nbody"), njnt = m.sz("njnt"), ngeom = m.sz("ngeom"),
            ntendon = m.sz("ntendon");
  if (nv <= 0 || nbody <= 1) add("model has no degrees of freedom");
  if (nv > 64) add("nv = " + std::to_string(nv) + " exceeds the dense solver limit (64)");
  if (m.sz("neq") > 0) add(std::to_string(m.sz("neq")) + " equality constraint(s): not supported");
  if (m.sz("npair") > 0) add(std::to_string(m.sz("npair")) + " explicit contact pair(s) (<contact><pair>): not supported (excludes are)");
  if (na != 0 && na != nu) add("mix of stateful and stateless actuators (na = " + std::to_string(na) + ", nu = " + std::to_string(nu) + ")");
  if ((int)m.opt.at("integrator") != 0) add("integrator is not Euler");
  if ((int)m.opt.at("cone") != 0) add("elliptic friction cones (only pyramidal)");
  std::vector<int> jtype = ivec(m, "jnt_type"), jbody = ivec(m, "jnt_bodyid"), jntnum = ivec(m, "body_jntnum");
  int nball = 0;
  for (int j = 0; j < njnt; j++) {
    if (jtype[j] == J_BALL) nball++;
    if (jtype[j] == J_FREE && jntnum[jbody[j]] != 1) add("free joint " + std::to_string(j) + " shares its body with other joints");
  }
  if (nball) add(std::to_string(nball) + " ball joint(s): not supported");
  { int n = 0; const double* dl = m.d("dof_frictionloss"); for (int i = 0; i < nv; i++) if (dl[i] != 0) n++; if (n) add(std::to_string(n) + " dof(s) with frictionloss: not supported"); }
  if (ntendon) { int n = 0; const double* tf = m.d("tendon_frictionloss"); for (int t = 0; t < ntendon; t++) if (tf[t] != 0) n++; if (n) add(std::to_string(n) + " tendon(s) with frictionloss: not supported"); }
  if (nu) { std::vector<int> tr = ivec(m, "actuator_trntype"); int n = 0; for (int i = 0; i < nu; i++) if (tr[i] != 3) n++; if (n) add(std::to_string(n) + " actuator(s) not driven through a tendon (only tendon transmissions)"); }
  if (m.sz("nwrap")) { std::vector<int> wt = ivec(m, "wrap_type"); int n = 0; for (int w : wt) if (w == 1) n++; if (n) add(std::to_string(n) + " fixed (joint) tendon term(s): only spatial tendons"); }
  // colliding geom type pairs the narrow phase does not cover
  std::vector<int> gtype = ivec(m, "geom_type"), gbody = ivec(m, "geom_bodyid"), ct = ivec(m, "geom_contype"), ca = ivec(m, "geom_conaffinity"),
                   weld = ivec(m, "body_weldid"), parent = ivec(m, "body_parentid"), condim = ivec(m, "geom_condim");
  static const char* tn[] = {"plane", "hfield", "sphere", "capsule", "ellipsoid", "cylinder", "box", "mesh"};
  std::set<std::pair<int, int>> bad;
  std::vector<int> excl = m.sz("nexclude") > 0 ? ivec(m, "exclude_signature") : std::vector<int>();
  for (int g1 = 0; g1 < ngeom; g1++) for (int g2 = g1 + 1; g2 < ngeom; g2++) {
    const int b1 = std::min(gbody[g1], gbody[g2]), b2 = std::max(gbody[g1], gbody[g2]);
    if (b1 == b2) continue;
    const int w1 = weld[b1], w2 = weld[b2];
    if (w1 == w2 || (w1 != 0 && w2 != 0 && (w1 == weld[parent[w2]] || w2 == weld[parent[w1]]))) continue;
    if (std::find(excl.begin(), excl.end(), (b1 << 16) + b2) != excl.end()) continue;
    if (!((ct[g1] & ca[g2]) || (ct[g2] & ca[g1]))) continue;
    const int t1 = std::min(gtype[g1], gtype[g2]), t2 = std::max(gtype[g1], gtype[g2]);
    const bool sup = (t1 == G_SPHERE && t2 == G_SPHERE) || (t1 == G_SPHERE && t2 == G_CAPSULE) || (t1 == G_PLANE && t2 == G_SPHERE) ||
                     (t1 == G_CAPSULE && t2 == G_BOX);
    if (!sup) bad.insert({t1, t2});
    const int dim = std::max(condim[g1], condim[g2]);
    if (dim != 1 && dim != 3) bad.insert({100 + dim, 0});
  }
  // advisory ("~"): such pairs are accepted; a world in which one of them comes into broad-phase range raises status bit 0
  for (auto& pr : bad) {
    if (pr.first >= 100) out += "~ contact dimension " + std::to_string(pr.first - 100) + " between some geoms (rows are built for condim 1 and 3; others raise status bit 0 when they touch)\n";
    else out += std::string("~ geom pair type ") + tn[pr.first & 7] + " - " + tn[pr.second & 7] + " can collide but has no narrow phase (have sphere-sphere, sphere-capsule, plane-sphere, capsule-box): status bit 0 if such a pair ever comes into range\n";
  }
  return out;
}

}  // namespace myo
