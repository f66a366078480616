// dev_model_build.h — host builder of the fp32 device image (see dev_model.h).
#pragma once
#include <algorithm>
#include <array>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <map>
#include <stdexcept>
#include <vector>

#include "../../include/mjb.h"
#include "dev_model.h"
#include "hmath.h"
#include "host_kin.h"
#include "model_view.h"
#include "replicate.h"

namespace mjb {

struct DevImage {
  DevModel dm;
  std::vector<uint32_t> words;
  RenderHdr rhdr{};                // camera table (pack == 1 images of models with cameras)
  std::vector<uint32_t> render;
};

namespace detail {
inline uint32_t f2w(double v) {
  float f = (float)v;
  uint32_t w;
  memcpy(&w, &f, 4);
  return w;
}
struct ImageWriter {
  std::vector<uint32_t>& words;
  DevModel& dm;
  void begin(int field) {
    while (words.size() % 4) words.push_back(0);
    dm.off[field] = (int)words.size();
  }
  void i(int v) { words.push_back((uint32_t)v); }
  void u(uint32_t v) { words.push_back(v); }
  void f(double v) { words.push_back(f2w(v)); }
};
}  // namespace detail

inline int env_int(const char* name, int dflt) {
  const char* s = getenv(name);
  return (s && *s) ? atoi(s) : dflt;
}

// why a spec's parameter-table fields cannot be used (nullptr: they can), see mjb_env_spec.params
inline const char* param_spec_error(const mjb_env_spec& spec) {
  if ((spec.flags & MJB_SPEC_RANDOMIZE) && !spec.params) return "MJB_SPEC_RANDOMIZE needs spec.params";
  if (spec.params && spec.skip_frames == 0) return "spec.params needs skip_frames >= 1 (the physics-free step reads no parameter)";
  if (spec.flags & MJB_SPEC_RANDOMIZE)
    for (int f = 0; f < 4; f++) {
      const float lo = spec.param_lo[f], hi = spec.param_hi[f];
      if (!std::isfinite(lo) || !std::isfinite(hi)) return "param_lo / param_hi must be finite";
      if (lo > hi) return "param_lo must be <= param_hi";
      if (lo < 0.f || (f == 0 && lo <= 0.f)) return "param_lo must be >= 0 (> 0 for body mass)";
    }
  return nullptr;
}

inline void build_dev_model(const ModelView& m, const mjb_env_spec& spec, DevImage& out, bool lite = false, int pack = 1) {
  DevModel& dm = out.dm;
  memset(&dm, 0, sizeof(dm));
  std::vector<uint32_t>& W = out.words;
  W.clear();
  detail::ImageWriter w{W, dm};
  const int nbody = m.nbody;
  if (m.nv > 32) throw std::runtime_error("kernel limit: nv <= 32 (one lane per degree of freedom)");
  if (m.nv < 1) throw std::runtime_error("model has no degrees of freedom");
  if (m.ngeom >= 4096) throw std::runtime_error("kernel limit: ngeom < 4096");

  // ---- moving bodies, kernel order (by depth)
  std::vector<int> moving(nbody, 0), kdepth(nbody, 0);
  for (int b = 1; b < nbody; b++) {
    int p = m.body_parentid[b];
    moving[b] = (m.body_dofnum[b] > 0) || moving[p];
    if (moving[b]) kdepth[b] = moving[p] ? kdepth[p] + 1 : 1;
  }
  int nlevel = 0;
  for (int b = 0; b < nbody; b++) nlevel = std::max(nlevel, kdepth[b]);
  std::vector<int> korder;  // kernel index -> body id
  std::vector<int> level_adr(nlevel + 1, 0);
  for (int l = 1; l <= nlevel; l++) {
    level_adr[l - 1] = (int)korder.size();
    for (int b = 1; b < nbody; b++)
      if (moving[b] && kdepth[b] == l) korder.push_back(b);
  }
  level_adr[nlevel] = (int)korder.size();
  const int nmb = (int)korder.size();
  std::vector<int> b2k(nbody, -1);
  for (int k = 0; k < nmb; k++) b2k[korder[k]] = k;

  HostKin kin;
  host_fk(m, m.qpos0, kin);

  dm.nq = m.nq; dm.nv = m.nv; dm.nu = m.nu; dm.nmb = nmb; dm.njnt = m.njnt; dm.ngeom = m.ngeom;
  dm.nsite = m.nsite; dm.nsensor = m.nsensor; dm.nsensordata = m.nsensordata; dm.npair = m.npair;
  dm.nlevel = nlevel; dm.integrator = m.integrator; dm.timestep = (float)m.timestep; dm.timestep_d = m.timestep;
  for (int i = 0; i < 3; i++) dm.gravity[i] = (float)m.gravity[i];
  dm.ldj = m.nv | 1;  // narrowed below to the widest contact dof mask
  dm.solver_iterations = spec.solver_iterations > 0 ? spec.solver_iterations : env_int("MJB_SOLVER_ITERS", 24);
  dm.reset_noise = spec.reset_noise > 0 ? spec.reset_noise : 0.f;
  dm.njnt1 = m.njnt / pack;
  dm.ls_iterations = spec.ls_iterations > 0 ? spec.ls_iterations : env_int("MJB_LS_ITERS", 12);
  {
    const char* ts = getenv("MJB_SOLVER_TOL");
    dm.solver_tol = (ts && *ts) ? (float)atof(ts) : 1e-6f;
  }

  w.begin(IF_level_adr); for (int v : level_adr) w.i(v);
  w.begin(IF_mb_parent); for (int k = 0; k < nmb; k++) w.i(b2k[m.body_parentid[korder[k]]]);
  w.begin(IF_mb_root);
  for (int k = 0; k < nmb; k++) {
    int b = korder[k];
    while (moving[m.body_parentid[b]]) b = m.body_parentid[b];
    w.i(b2k[b]);
  }
  w.begin(IF_mb_jntadr); for (int k = 0; k < nmb; k++) w.i(m.body_jntadr[korder[k]]);
  w.begin(IF_mb_jntnum); for (int k = 0; k < nmb; k++) w.i(m.body_jntnum[korder[k]]);
  w.begin(IF_mb_dofadr); for (int k = 0; k < nmb; k++) w.i(m.body_dofadr[korder[k]]);
  w.begin(IF_mb_dofnum); for (int k = 0; k < nmb; k++) w.i(m.body_dofnum[korder[k]]);
  {
    std::vector<std::vector<int>> children(nmb);
    for (int k = 0; k < nmb; k++) {
      int pk = b2k[m.body_parentid[korder[k]]];
      if (pk >= 0) children[pk].push_back(k);
    }
    w.begin(IF_mb_childadr);
    int adr = 0;
    for (int k = 0; k < nmb; k++) { w.i(adr); adr += (int)children[k].size(); }
    w.i(adr);
    w.begin(IF_mb_child);
    for (int k = 0; k < nmb; k++) for (int c : children[k]) w.i(c);
    if (adr == 0) w.i(0);
  }
  w.begin(IF_mb_dofmask);
  for (int k = 0; k < nmb; k++) {
    uint64_t mask = 0;
    for (int b = korder[k]; b > 0; b = m.body_parentid[b])
      for (int d = m.body_dofadr[b]; d >= 0 && d < m.body_dofadr[b] + m.body_dofnum[b]; d++) mask |= (1ull << d);
    w.u((uint32_t)(mask & 0xffffffffu)); w.u((uint32_t)(mask >> 32));
  }
  w.begin(IF_mb_pos);
  for (int k = 0; k < nmb; k++) {
    int b = korder[k], p = m.body_parentid[b];
    V3 bp(m.body_pos[3 * b], m.body_pos[3 * b + 1], m.body_pos[3 * b + 2]);
    if (!moving[p]) bp = kin.xpos[p] + mulv(kin.xmat[p], bp);
    for (int i = 0; i < 3; i++) w.f(bp[i]);
  }
  w.begin(IF_mb_quat);
  for (int k = 0; k < nmb; k++) {
    int b = korder[k], p = m.body_parentid[b];
    Quat q{m.body_quat[4 * b], m.body_quat[4 * b + 1], m.body_quat[4 * b + 2], m.body_quat[4 * b + 3]};
    if (!moving[p]) q = qnormalized(qmul(kin.xquat[p], q));
    w.f(q.w); w.f(q.x); w.f(q.y); w.f(q.z);
  }
  w.begin(IF_mb_ipos); for (int k = 0; k < nmb; k++) for (int i = 0; i < 3; i++) w.f(m.body_ipos[3 * korder[k] + i]);
  w.begin(IF_mb_iquat); for (int k = 0; k < nmb; k++) for (int i = 0; i < 4; i++) w.f(m.body_iquat[4 * korder[k] + i]);
  w.begin(IF_mb_mass); for (int k = 0; k < nmb; k++) w.f(m.body_mass[korder[k]]);
  w.begin(IF_mb_inertia); for (int k = 0; k < nmb; k++) for (int i = 0; i < 3; i++) w.f(m.body_inertia[3 * korder[k] + i]);
  w.begin(IF_mb_invweight); for (int k = 0; k < nmb; k++) w.f(m.body_invweight0[2 * korder[k]]);

  // ---- joints / dofs
  w.begin(IF_jnt_type); for (int j = 0; j < m.njnt; j++) w.i(m.jnt_type[j]);
  w.begin(IF_jnt_qposadr); for (int j = 0; j < m.njnt; j++) w.i(m.jnt_qposadr[j]);
  w.begin(IF_jnt_dofadr); for (int j = 0; j < m.njnt; j++) w.i(m.jnt_dofadr[j]);
  w.begin(IF_jnt_pos); for (int j = 0; j < 3 * m.njnt; j++) w.f(m.jnt_pos[j]);
  w.begin(IF_jnt_axis); for (int j = 0; j < 3 * m.njnt; j++) w.f(m.jnt_axis[j]);
  w.begin(IF_jnt_qpos0); for (int j = 0; j < m.njnt; j++) w.f(m.qpos0[m.jnt_qposadr[j]]);
  auto kb_of = [&](const double* solref, const double* solimp, double& K, double& B) {
    double dmax = solimp[1];
    if (solref[0] > 0) {
      double tc = std::max(solref[0], 2 * m.timestep), dr = solref[1];
      K = 1.0 / std::max(1e-15, dmax * dmax * tc * tc * dr * dr);
      B = 2.0 / std::max(1e-15, dmax * tc);
    } else {
      K = -solref[0] / std::max(1e-15, dmax * dmax);
      B = -solref[1] / std::max(1e-15, dmax);
    }
  };
  std::vector<int> lim;
  for (int j = 0; j < m.njnt; j++)
    if (m.jnt_limited[j] && m.jnt_type[j] != MJB_JNT_FREE) lim.push_back(j);
  dm.nlim = (int)lim.size();
  w.begin(IF_lim_dof); for (int j : lim) w.i(m.jnt_dofadr[j]); if (lim.empty()) w.i(0);
  w.begin(IF_lim_qposadr); for (int j : lim) w.i(m.jnt_qposadr[j]); if (lim.empty()) w.i(0);
  w.begin(IF_lim_param);
  for (int j : lim) {
    double K, B;
    kb_of(&m.jnt_solref[2 * j], &m.jnt_solimp[5 * j], K, B);
    w.f(m.jnt_range[2 * j]); w.f(m.jnt_range[2 * j + 1]); w.f(m.jnt_margin[j]); w.f(K); w.f(B);
    w.f(m.dof_invweight0[m.jnt_dofadr[j]]);
    for (int i = 0; i < 5; i++) w.f(m.jnt_solimp[5 * j + i]);
    w.f(0);
  }
  if (lim.empty()) for (int i = 0; i < LIM_STRIDE; i++) w.f(0);
  w.begin(IF_dof_mb); for (int d = 0; d < m.nv; d++) w.i(b2k[m.dof_bodyid[d]]);
  w.begin(IF_dof_parent); for (int d = 0; d < m.nv; d++) w.i(m.dof_parentid[d]);
  w.begin(IF_dof_kind);
  for (int d = 0; d < m.nv; d++) {
    int j = m.dof_jntid[d];
    if (m.jnt_type[j] == MJB_JNT_FREE) w.i(d - m.jnt_dofadr[j] < 3 ? DOF_FREE_TRANS : DOF_FREE_ROT);
    else w.i(DOF_AXIS);
  }
  {
    // kinematic-tree dof ranges (trees own contiguous dof ranges); used to factor block by block
    std::vector<int> t0(32, 0), t1(32, 0);
    int maxtree = 0;
    for (int d = 0; d < m.nv; d++) {
      int lo = d, hi = d;
      int tree = m.body_treeid[m.dof_bodyid[d]];
      while (lo > 0 && m.body_treeid[m.dof_bodyid[lo - 1]] == tree) lo--;
      while (hi + 1 < m.nv && m.body_treeid[m.dof_bodyid[hi + 1]] == tree) hi++;
      t0[d] = lo; t1[d] = hi + 1;
      maxtree = std::max(maxtree, hi + 1 - lo);
    }
    dm.maxtree = maxtree;
    w.begin(IF_dof_t0); for (int v : t0) w.i(v);
    w.begin(IF_dof_t1); for (int v : t1) w.i(v);
  }
  {
    int dl[32];
    for (int d = 0; d < 32; d++) dl[d] = -1;
    for (size_t k = 0; k < lim.size(); k++) { int d = m.jnt_dofadr[lim[k]]; if (d >= 0 && d < 32) dl[d] = (int)k; }
    w.begin(IF_dof_lim); for (int v : dl) w.i(v);
  }
  w.begin(IF_dof_armature); for (int d = 0; d < m.nv; d++) w.f(m.dof_armature[d]);
  w.begin(IF_dof_damping);
  for (int d = 0; d < m.nv; d++) { w.f(m.dof_damping[d]); if (m.dof_damping[d] > 0) dm.has_damping = 1; }

  // ---- geoms
  std::vector<int> geom_slot(m.ngeom, -1);
  int ngdyn = 0;
  for (int g = 0; g < m.ngeom; g++)
    if (moving[m.geom_bodyid[g]]) geom_slot[g] = ngdyn++;
  dm.ngdyn = ngdyn;
  w.begin(IF_geom_type); for (int g = 0; g < m.ngeom; g++) w.i(m.geom_type[g]);
  w.begin(IF_geom_mb); for (int g = 0; g < m.ngeom; g++) w.i(b2k[m.geom_bodyid[g]]);
  w.begin(IF_geom_slot); for (int g = 0; g < m.ngeom; g++) w.i(geom_slot[g]);
  w.begin(IF_geom_size); for (int g = 0; g < 3 * m.ngeom; g++) w.f(m.geom_size[g]);
  w.begin(IF_geom_rbound); for (int g = 0; g < m.ngeom; g++) w.f(m.geom_rbound[g]);
  std::vector<V3> gworld(m.ngeom);
  std::vector<M3> gworldR(m.ngeom);
  for (int g = 0; g < m.ngeom; g++) {
    int b = m.geom_bodyid[g];
    V3 lp(m.geom_pos[3 * g], m.geom_pos[3 * g + 1], m.geom_pos[3 * g + 2]);
    Quat lq{m.geom_quat[4 * g], m.geom_quat[4 * g + 1], m.geom_quat[4 * g + 2], m.geom_quat[4 * g + 3]};
    gworld[g] = kin.xpos[b] + mulv(kin.xmat[b], lp);
    gworldR[g] = q2m(qmul(kin.xquat[b], lq));
  }
  w.begin(IF_geom_pos);
  for (int g = 0; g < m.ngeom; g++)
    for (int i = 0; i < 3; i++) w.f(geom_slot[g] >= 0 ? m.geom_pos[3 * g + i] : gworld[g][i]);
  w.begin(IF_geom_mat);
  for (int g = 0; g < m.ngeom; g++) for (int i = 0; i < 9; i++) w.f(gworldR[g].m[i]);
  w.begin(IF_geom_quat); for (int g = 0; g < 4 * m.ngeom; g++) w.f(m.geom_quat[g]);
  w.begin(IF_geom_ray); for (int g = 0; g < m.ngeom; g++) w.i(m.geom_rgba[4 * g + 3] != 0 ? 1 : 0);

  // ---- collision pairs, sorted by type pair; parameter classes de-duplicated
  {
    std::vector<int> order(m.npair);
    for (int k = 0; k < m.npair; k++) order[k] = k;
    // Pair blocks for the two-level broad phase: all pairs between one kinematic tree and another tree / one
    // static geom.  A tree is bounded by a sphere about its root body's origin whose radius is the farthest any of
    // its geoms can get from that origin in any joint configuration (`reach`, below); a 32-pair pass of the flat
    // broad phase is skipped when none of its blocks can touch.
    std::vector<double> reach_body(nbody, 0.0), reach_tree(nbody, 0.0);   // indexed by body / by root body
    std::vector<int> root_of(nbody, 0);
    for (int b = 1; b < nbody; b++) {
      if (!moving[b]) continue;
      int p = m.body_parentid[b];
      if (!moving[p]) { root_of[b] = b; reach_body[b] = 0; continue; }
      root_of[b] = root_of[p];
      double jp = 0, slide = 0;
      for (int j = m.body_jntadr[b]; j >= 0 && j < m.body_jntadr[b] + m.body_jntnum[b]; j++) {
        jp = std::max(jp, std::sqrt(m.jnt_pos[3 * j] * m.jnt_pos[3 * j] + m.jnt_pos[3 * j + 1] * m.jnt_pos[3 * j + 1] + m.jnt_pos[3 * j + 2] * m.jnt_pos[3 * j + 2]));
        if (m.jnt_type[j] == MJB_JNT_SLIDE)
          slide += m.jnt_limited[j] ? std::max(std::fabs(m.jnt_range[2 * j]), std::fabs(m.jnt_range[2 * j + 1])) : 1e9;
        if (m.jnt_type[j] == MJB_JNT_FREE) slide += 1e9;   // a free joint below the root: unbounded
      }
      double bp = std::sqrt(m.body_pos[3 * b] * m.body_pos[3 * b] + m.body_pos[3 * b + 1] * m.body_pos[3 * b + 1] + m.body_pos[3 * b + 2] * m.body_pos[3 * b + 2]);
      reach_body[b] = reach_body[p] + bp + 2 * jp + slide;
    }
    for (int g = 0; g < m.ngeom; g++) {
      int b = m.geom_bodyid[g];
      if (!moving[b]) continue;
      double gp = std::sqrt(m.geom_pos[3 * g] * m.geom_pos[3 * g] + m.geom_pos[3 * g + 1] * m.geom_pos[3 * g + 1] + m.geom_pos[3 * g + 2] * m.geom_pos[3 * g + 2]);
      double r = m.geom_type[g] == MJB_GEOM_PLANE ? 1e9 : m.geom_rbound[g];
      reach_tree[root_of[b]] = std::max(reach_tree[root_of[b]], reach_body[b] + gp + r);
    }
    auto group = [&](int g) { int b = m.geom_bodyid[g]; return moving[b] ? root_of[b] : -1 - g; };   // tree root body | static geom
    std::map<std::pair<int, int>, int> block_id;
    std::vector<std::array<double, 4>> blocks;   // rootA kernel body, partner, reach, margin
    std::vector<int> pair_block(m.npair, 0);
    for (int k = 0; k < m.npair; k++) {
      int ga = group(m.pair_geom1[k]), gb = group(m.pair_geom2[k]);
      if (ga < 0 && gb >= 0) std::swap(ga, gb);          // the tree first
      else if (ga >= 0 && gb >= 0 && gb < ga) std::swap(ga, gb);
      auto key = std::make_pair(ga, gb);
      auto it = block_id.find(key);
      int id;
      if (it == block_id.end()) {
        id = (int)blocks.size();
        block_id[key] = id;
        std::array<double, 4> rec{0, (double)BP_ALWAYS, 0, 0};
        if (ga >= 0 && gb >= 0 && ga != gb) { rec = {(double)b2k[ga], (double)b2k[gb], reach_tree[ga] + reach_tree[gb], 0}; }
        else if (ga >= 0 && gb < 0) { rec = {(double)b2k[ga], (double)gb, reach_tree[ga], 0}; }
        blocks.push_back(rec);
      } else id = it->second;
      blocks[id][3] = std::max(blocks[id][3], m.pair_margin[k]);
      pair_block[k] = id;
    }
    const bool use_blocks = !blocks.empty() && blocks.size() <= 64;
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) {
      int ta = m.geom_type[m.pair_geom1[a]] * 16 + m.geom_type[m.pair_geom2[a]];
      int tb = m.geom_type[m.pair_geom1[b]] * 16 + m.geom_type[m.pair_geom2[b]];
      if (use_blocks && pair_block[a] != pair_block[b]) return pair_block[a] < pair_block[b];
      return ta < tb;
    });
    dm.nblock = use_blocks ? (int)blocks.size() : 0;
    w.begin(IF_bp_block);
    for (int i = 0; i < dm.nblock; i++) {
      w.i((int)blocks[i][0]); w.i((int)blocks[i][1]); w.f(std::min(blocks[i][2], 1e9)); w.f(blocks[i][3]);
    }
    if (!dm.nblock) for (int i = 0; i < BP_STRIDE; i++) w.i(0);
    w.begin(IF_bp_passmask);
    for (int base = 0; base < std::max(1, m.npair); base += 32) {
      uint64_t mask = 0;
      for (int i = base; i < std::min(m.npair, base + 32); i++) mask |= use_blocks ? (1ull << pair_block[order[i]]) : ~0ull;
      if (!use_blocks) mask = ~0ull;
      w.u((uint32_t)(mask & 0xffffffffu)); w.u((uint32_t)(mask >> 32));
    }
    std::map<std::vector<float>, int> classes;
    std::vector<std::vector<float>> class_list;
    std::vector<uint32_t> packed;
    for (int k : order) {
      double K, B;
      kb_of(&m.pair_solref[2 * k], &m.pair_solimp[5 * k], K, B);
      std::vector<float> key = {(float)m.pair_margin[k], (float)m.pair_includemargin[k], (float)m.pair_friction[3 * k],
                                (float)K, (float)B};
      for (int i = 0; i < 5; i++) key.push_back((float)m.pair_solimp[5 * k + i]);
      key.push_back((float)m.pair_condim[k]);
      key.push_back(0.f);
      auto it = classes.find(key);
      int cid;
      if (it == classes.end()) { cid = (int)class_list.size(); classes[key] = cid; class_list.push_back(key); }
      else cid = it->second;
      if (cid > 255) throw std::runtime_error("kernel limit: more than 256 contact parameter classes");
      packed.push_back((uint32_t)m.pair_geom1[k] | ((uint32_t)m.pair_geom2[k] << 12) | ((uint32_t)cid << 24));
    }
    w.begin(IF_pair_pack); for (uint32_t p : packed) w.u(p); if (packed.empty()) w.u(0);
    dm.nclass = (int)class_list.size();
    w.begin(IF_pclass);
    for (auto& c : class_list) for (float v : c) w.f(v);
    if (class_list.empty()) for (int i = 0; i < PC_STRIDE; i++) w.f(0);
  }

  // ---- camera table (not part of the step image: only the render kernel stages it)
  out.render.clear();
  out.rhdr = RenderHdr{};
  if (m.ncam > 0 && pack == 1) {
    std::vector<uint32_t>& T = out.render;
    out.rhdr.ncam = m.ncam; out.rhdr.ngeom = m.ngeom; out.rhdr.off_cam = 0;
    for (int k = 0; k < m.ncam; k++) {
      int b = m.cam_bodyid[k];
      V3 lp(m.cam_pos[3 * k], m.cam_pos[3 * k + 1], m.cam_pos[3 * k + 2]);
      Quat q{m.cam_quat[4 * k], m.cam_quat[4 * k + 1], m.cam_quat[4 * k + 2], m.cam_quat[4 * k + 3]};
      if (!moving[b]) { lp = kin.xpos[b] + mulv(kin.xmat[b], lp); q = qnormalized(qmul(kin.xquat[b], q)); }
      T.push_back((uint32_t)b2k[b]); T.push_back((uint32_t)m.cam_mode[k]);
      for (int i = 0; i < 3; i++) T.push_back(detail::f2w(lp[i]));
      T.push_back(detail::f2w(q.w)); T.push_back(detail::f2w(q.x)); T.push_back(detail::f2w(q.y)); T.push_back(detail::f2w(q.z));
      T.push_back(detail::f2w(std::tan(0.5 * m.cam_fovy[k] * 3.14159265358979323846 / 180.0)));
      T.push_back(0); T.push_back(0);
    }
    out.rhdr.off_rgba = (int)T.size();
    for (int g = 0; g < m.ngeom; g++)
      for (int i = 0; i < 4; i++) T.push_back(detail::f2w(std::min(1.0, std::max(0.0, m.geom_rgba[4 * g + i]))));
    while (T.size() % 4) T.push_back(0);
    out.rhdr.words = (int)T.size();
  }

  // ---- sites / sensors / actuators
  w.begin(IF_site_mb); for (int t = 0; t < m.nsite; t++) w.i(b2k[m.site_bodyid[t]]); if (!m.nsite) w.i(0);
  w.begin(IF_site_type); for (int t = 0; t < m.nsite; t++) w.i(m.site_type[t]); if (!m.nsite) w.i(0);
  w.begin(IF_site_pos);
  for (int t = 0; t < m.nsite; t++) {
    int b = m.site_bodyid[t];
    V3 lp(m.site_pos[3 * t], m.site_pos[3 * t + 1], m.site_pos[3 * t + 2]);
    if (!moving[b]) lp = kin.xpos[b] + mulv(kin.xmat[b], lp);
    for (int i = 0; i < 3; i++) w.f(lp[i]);
  }
  w.begin(IF_site_quat);
  for (int t = 0; t < m.nsite; t++) {
    int b = m.site_bodyid[t];
    Quat q{m.site_quat[4 * t], m.site_quat[4 * t + 1], m.site_quat[4 * t + 2], m.site_quat[4 * t + 3]};
    if (!moving[b]) q = qnormalized(qmul(kin.xquat[b], q));
    w.f(q.w); w.f(q.x); w.f(q.y); w.f(q.z);
  }
  w.begin(IF_site_size); for (int t = 0; t < 3 * m.nsite; t++) w.f(m.site_size[t]);
  // frame / velocity / joint sensors (DESIGN §5f): evaluated by their own pass from an object record each (SO_*)
  auto frame_axis = [](int t) { return t >= MJB_SENS_FRAMEXAXIS && t <= MJB_SENS_FRAMEZAXIS; };
  auto ext_sensor = [&](int i) {
    const int t = m.sensor_type[i];
    return t == MJB_SENS_VELOCIMETER || t == MJB_SENS_GYRO || t == MJB_SENS_JOINTPOS || t == MJB_SENS_JOINTVEL ||
           t == MJB_SENS_FRAMEPOS || t == MJB_SENS_FRAMEQUAT || t == MJB_SENS_FRAMELINVEL || t == MJB_SENS_FRAMEANGVEL ||
           (frame_axis(t) && m.sensor_objtype[i] != MJB_OBJ_SITE);
  };
  for (int i = 0; i < m.nsensor; i++) if (ext_sensor(i)) dm.ext_sensors = 1;
  w.begin(IF_sensor_type);
  for (int i = 0; i < m.nsensor; i++) {
    const int t = m.sensor_type[i];
    w.i(frame_axis(t) && ext_sensor(i) ? KSENS_OBJ_AXIS + (t - MJB_SENS_FRAMEXAXIS) : t);
  }
  if (!m.nsensor) w.i(0);
  w.begin(IF_sensor_site);
  for (int i = 0; i < m.nsensor; i++) {
    const int t = m.sensor_type[i], id = m.sensor_objid[i];
    if (m.sensor_objtype[i] == MJB_OBJ_JOINT) w.i(t == MJB_SENS_JOINTPOS ? m.jnt_qposadr[id] : m.jnt_dofadr[id]);
    else w.i(m.sensor_objtype[i] == MJB_OBJ_SITE ? id : 0);
  }
  if (!m.nsensor) w.i(0);
  w.begin(IF_sensor_adr); for (int i = 0; i < m.nsensor; i++) w.i(m.sensor_adr[i]); if (!m.nsensor) w.i(0);
  w.begin(IF_sensor_dim); for (int i = 0; i < m.nsensor; i++) w.i(m.sensor_dim[i]); if (!m.nsensor) w.i(0);
  w.begin(IF_sensor_dtype); for (int i = 0; i < m.nsensor; i++) w.i(m.sensor_datatype[i]); if (!m.nsensor) w.i(0);
  w.begin(IF_sensor_cutoff); for (int i = 0; i < m.nsensor; i++) w.f(m.sensor_cutoff[i]); if (!m.nsensor) w.f(0);
  for (int i = 0; i < m.nsensor; i++)
    if (m.sensor_type[i] == MJB_SENS_ACCELEROMETER || m.sensor_type[i] == MJB_SENS_TOUCH) dm.need_acc_sensors = 1;
  w.begin(IF_act_dof); for (int u = 0; u < m.nu; u++) w.i(m.jnt_dofadr[m.actuator_trnid[u]]); if (!m.nu) w.i(0);
  w.begin(IF_act_param);
  for (int u = 0; u < m.nu; u++) {
    w.f(m.actuator_gear[u]); w.f(m.actuator_ctrllimited[u]); w.f(m.actuator_ctrlrange[2 * u]); w.f(m.actuator_ctrlrange[2 * u + 1]);
  }
  if (!m.nu) for (int i = 0; i < 4; i++) w.f(0);
  {
    std::vector<int> adr(m.nv, 0), num(m.nv, 0), list;
    for (int d = 0; d < m.nv; d++) {
      adr[d] = (int)list.size();
      for (int u = 0; u < m.nu; u++)
        if (m.jnt_dofadr[m.actuator_trnid[u]] == d) { list.push_back(u); num[d]++; }
    }
    w.begin(IF_dof_actadr); for (int v : adr) w.i(v);
    w.begin(IF_dof_actnum); for (int v : num) w.i(v);
    w.begin(IF_act_list); for (int v : list) w.i(v); if (list.empty()) w.i(0);
  }

  // ---- env spec: agents, probes, plugins
  if (spec.n_agents < 0 || spec.n_agents > MJB_MAX_AGENTS) throw std::runtime_error("n_agents out of range");
  dm.n_agents = spec.n_agents; dm.free_joint = spec.free_joint; dm.skip_frames = spec.skip_frames;
  dm.max_steps = spec.max_steps; dm.n_phys_act = spec.n_phys_act; dm.act_dim = spec.act_dim; dm.seed = spec.seed;
  dm.n_dynamics = spec.n_dynamics; dm.n_rewards = spec.n_rewards; dm.n_dones = spec.n_dones; dm.n_targets = spec.n_targets;
  if (spec.n_dynamics > MJB_MAX_PLUGINS || spec.n_rewards > MJB_MAX_PLUGINS || spec.n_dones > MJB_MAX_PLUGINS)
    throw std::runtime_error("too many plugins");
  if (spec.n_targets > MJB_MAX_TARGETS) throw std::runtime_error("too many targets");
  auto cp = [](DevPlugin& d, const mjb_plugin& s) {
    d.kind = s.kind; d.act_lo = s.act_lo; d.act_hi = s.act_hi; d.n_obs = s.n_obs;
    for (int i = 0; i < 4; i++) d.param[i] = s.param[i];
  };
  for (int i = 0; i < spec.n_dynamics; i++) cp(dm.dynamics[i], spec.dynamics[i]);
  dm.autoreset = (spec.flags & MJB_SPEC_AUTORESET) ? 1 : 0;
  dm.final_obs = dm.autoreset ? spec.final_obs : nullptr;
  dm.final_qpos = dm.autoreset ? spec.final_qpos : nullptr;
  for (int i = 0; i < spec.n_dynamics; i++) {
    const int d = spec.dynamics[i].act_lo;
    if (dm.autoreset && spec.dynamics[i].act_hi > d) {
      if (d < 0 || d >= spec.act_dim || d >= 64) throw std::runtime_error("dynamic action slot out of range");
      dm.dyn_act_low[i] = spec.act_low[d]; dm.dyn_act_high[i] = spec.act_high[d];
    }
  }
  if (spec.n_start < 0) throw std::runtime_error("n_start < 0");
  if (spec.n_start > 0) { dm.start_qpos = spec.start_qpos; dm.start_qvel = spec.start_qvel; dm.n_start = spec.n_start; }
  for (int i = 0; i < spec.n_rewards; i++) cp(dm.rewards[i], spec.rewards[i]);
  for (int i = 0; i < spec.n_dones; i++) cp(dm.dones[i], spec.dones[i]);
  std::vector<int> pk, pid;
  std::vector<V3> pconst;
  auto add_probe = [&](int objtype, int objid) {
    int idx = (int)pk.size();
    if (objtype == MJB_OBJ_BODY) {
      if (objid < 0 || objid >= nbody) throw std::runtime_error("probe: bad body id");
      if (moving[objid]) { pk.push_back(PROBE_BODY); pid.push_back(b2k[objid]); pconst.push_back(V3()); }
      else { pk.push_back(PROBE_CONST); pid.push_back(objid); pconst.push_back(kin.xipos[objid]); }
    } else {
      if (objid < 0 || objid >= m.ngeom) throw std::runtime_error("probe: bad geom id");
      if (geom_slot[objid] >= 0) { pk.push_back(PROBE_GEOM); pid.push_back(geom_slot[objid]); pconst.push_back(V3()); }
      else { pk.push_back(PROBE_CONST); pid.push_back(objid); pconst.push_back(gworld[objid]); }
    }
    return idx;
  };
  for (int a = 0; a < spec.n_agents; a++) {
    dm.agent_probe[a] = add_probe(MJB_OBJ_BODY, spec.agent_body[a]);
    dm.obs_dim[a] = spec.obs_dim[a];
  }
  for (int a = 0; a <= spec.n_agents; a++) dm.obs_adr[a] = spec.obs_adr[a];
  for (int t = 0; t < spec.n_targets; t++) dm.target_probe[t] = add_probe(spec.target_objtype[t], spec.target_objid[t]);
  if (spec.n_extra_probes < 0 || spec.n_extra_probes > MJB_MAX_EXTRA_PROBES) throw std::runtime_error("too many extra probes");
  if (spec.n_extra_probes > 0 && pack > 1) throw std::runtime_error("extra probes need an unpacked batch");
  for (int x = 0; x < spec.n_extra_probes; x++) add_probe(spec.extra_objtype[x], spec.extra_objid[x]);
  dm.nprobe = (int)pk.size();
  w.begin(IF_probe_kind); for (int v : pk) w.i(v); if (pk.empty()) w.i(0);
  w.begin(IF_probe_id); for (int v : pid) w.i(v); if (pid.empty()) w.i(0);
  w.begin(IF_probe_const); for (auto& v : pconst) for (int i = 0; i < 3; i++) w.f(v[i]); if (pconst.empty()) w.f(0);
  w.begin(IF_act_index);
  for (int i = 0; i < spec.n_agents * spec.n_phys_act; i++) {
    int idx = spec.act_index[i];
    if (idx < 0 || idx >= (spec.free_joint ? m.nv : m.nu)) throw std::runtime_error("act_index out of range");
    w.i(idx);
  }
  if (spec.n_agents * spec.n_phys_act == 0) w.i(0);
  w.begin(IF_obs_index);
  for (int i = 0; i < spec.obs_adr[spec.n_agents]; i++) {
    int e = spec.obs_index[i], kind = e >> 24, adr = e & 0xffffff;
    int lim_n = kind == 0 ? m.nsensordata : (kind == 1 ? m.nq : m.nv);
    if (kind < 0 || kind > 2 || adr >= lim_n) throw std::runtime_error("obs_index out of range");
    w.i(e);
  }
  if (spec.obs_adr[spec.n_agents] == 0) w.i(0);
  w.begin(IF_tri_lut);
  for (int r = 0; r < 16; r++) for (int cc = 0; cc <= r; cc++) w.u((uint32_t)r | ((uint32_t)cc << 8));
  w.begin(IF_qpos0); for (int i = 0; i < m.nq; i++) w.f(m.qpos0[i]);
  if (spec.params && !lite) {
    // per-env parameter table: where every word of the PRM scratch block comes from in the env's row, its draw key and
    // its nominal value.  Rows are per REAL env: copy c of a packed env reads row e0 + c, with the real model's ids.
    if (const char* e = param_spec_error(spec)) throw std::runtime_error(e);
    const int nb1 = (nbody - 1) / pack + 1, ng1 = m.ngeom / pack, nu1 = m.nu / pack, nv1 = m.nv / pack;
    const int o_inertia = nb1, o_friction = 4 * nb1, o_gear = 4 * nb1 + ng1, o_damping = 4 * nb1 + ng1 + nu1;
    dm.n_params = 4 * nb1 + ng1 + nu1 + nv1;
    if (dm.n_params >= 65536) throw std::runtime_error("kernel limit: parameter row of more than 65535 floats");
    if (nb1 >= 4096) throw std::runtime_error("kernel limit: a parameter table needs fewer than 4096 bodies");
    std::vector<uint32_t> map;
    std::vector<double> nominal;
    auto add = [&](int off, int index, int family, int copy, double v) {
      map.push_back((uint32_t)off | ((uint32_t)index << 16) | ((uint32_t)family << 28) | ((uint32_t)copy << 30));
      nominal.push_back(v);
    };
    for (int k = 0; k < nmb; k++) {
      const int vb = korder[k], c = (vb - 1) / (nb1 - 1), b = 1 + (vb - 1) % (nb1 - 1);
      add(b, b, 0, c, m.body_mass[vb]);
    }
    for (int k = 0; k < nmb; k++) {
      const int vb = korder[k], c = (vb - 1) / (nb1 - 1), b = 1 + (vb - 1) % (nb1 - 1);
      for (int i = 0; i < 3; i++) add(o_inertia + 3 * b + i, b, 0, c, m.body_inertia[3 * vb + i]);
    }
    for (int d = 0; d < m.nv; d++) add(o_damping + d % nv1, d % nv1, 3, d / nv1, m.dof_damping[d]);
    for (int u = 0; u < m.nu; u++) add(o_gear + u % nu1, u % nu1, 2, u / nu1, m.actuator_gear[u]);
    for (int g = 0; g < m.ngeom; g++) add(o_friction + g % ng1, g % ng1, 1, g / ng1, m.geom_friction[3 * g]);
    dm.params = spec.params;
    dm.prm_n = (int)map.size();
    dm.randomize = (spec.flags & MJB_SPEC_RANDOMIZE) ? 1 : 0;
    for (int f = 0; f < 4; f++) { dm.prm_lo[f] = spec.param_lo[f]; dm.prm_hi[f] = spec.param_hi[f]; }
    while (W.size() % 4) W.push_back(0);
    dm.off_prm_map = (int)W.size();
    for (uint32_t v : map) w.u(v);
    while (W.size() % 4) W.push_back(0);
    dm.off_prm_nominal = (int)W.size();
    for (double v : nominal) w.f(v);
  }
  if (dm.ext_sensors && !lite) {
    while (W.size() % 4) W.push_back(0);
    dm.off_sens_obj = (int)W.size();
    for (int i = 0; i < m.nsensor; i++) {
      // body the object rides on and its pose there: site / geom frame, inertial frame (body), body frame (xbody)
      const int ot = m.sensor_objtype[i], id = m.sensor_objid[i];
      int b = 0;
      V3 lp;
      Quat lq;
      if (ot == MJB_OBJ_SITE) {
        b = m.site_bodyid[id]; lp = V3(m.site_pos[3 * id], m.site_pos[3 * id + 1], m.site_pos[3 * id + 2]);
        lq = Quat{m.site_quat[4 * id], m.site_quat[4 * id + 1], m.site_quat[4 * id + 2], m.site_quat[4 * id + 3]};
      } else if (ot == MJB_OBJ_GEOM) {
        b = m.geom_bodyid[id]; lp = V3(m.geom_pos[3 * id], m.geom_pos[3 * id + 1], m.geom_pos[3 * id + 2]);
        lq = Quat{m.geom_quat[4 * id], m.geom_quat[4 * id + 1], m.geom_quat[4 * id + 2], m.geom_quat[4 * id + 3]};
      } else if (ot == MJB_OBJ_BODY) {
        b = id; lp = V3(m.body_ipos[3 * id], m.body_ipos[3 * id + 1], m.body_ipos[3 * id + 2]);
        lq = Quat{m.body_iquat[4 * id], m.body_iquat[4 * id + 1], m.body_iquat[4 * id + 2], m.body_iquat[4 * id + 3]};
      } else if (ot == MJB_OBJ_XBODY) {
        b = id;
      }
      if (!moving[b]) { lp = kin.xpos[b] + mulv(kin.xmat[b], lp); lq = qnormalized(qmul(kin.xquat[b], lq)); }
      w.i(moving[b] ? b2k[b] : -1);
      for (int k = 0; k < 3; k++) w.f(lp[k]);
      w.f(lq.w); w.f(lq.x); w.f(lq.y); w.f(lq.z);
    }
  }
  while (W.size() % 4) W.push_back(0);
  dm.image_words = (int)W.size();

  // packed contact Jacobian width: the widest chain(b1) xor chain(b2) over the collision pair table
  {
    auto chain = [&](int body) {
      uint64_t mask = 0;
      for (int b = body; b > 0; b = m.body_parentid[b])
        for (int d = m.body_dofadr[b]; d >= 0 && d < m.body_dofadr[b] + m.body_dofnum[b]; d++) mask |= (1ull << d);
      return mask;
    };
    int widest = 1;
    for (int k = 0; k < m.npair; k++) {
      uint64_t x = chain(m.geom_bodyid[m.pair_geom1[k]]) ^ chain(m.geom_bodyid[m.pair_geom2[k]]);
      widest = std::max(widest, (int)__builtin_popcountll(x));
    }
    dm.ldj = widest | 1;  // odd stride: lane = row accesses stay bank-conflict free
  }
  // ---- limits on per-env scratch
  int dflt_con = (ngdyn / pack) >= 16 ? 12 : 8;
  dm.maxcon1 = std::max(1, env_int("MJB_MAXCON", dflt_con));
  dm.maxcon = dm.maxcon1 * pack;
  dm.maxcand = std::max(32, std::min(m.npair, env_int("MJB_MAXCAND", 160)));
  dm.maxefc = 2 * dm.nlim + 4 * dm.maxcon;

  auto r4 = [](int n) { return (n + 3) & ~3; };
  int sizes[SF_COUNT];
  const int nv = m.nv;
  sizes[SF_qpos] = m.nq; sizes[SF_qvel] = nv; sizes[SF_qacc] = nv; sizes[SF_ctrl] = std::max(1, m.nu); sizes[SF_qfrc] = nv;
  sizes[SF_xpos] = 3 * nmb; sizes[SF_xquat] = 4 * nmb; sizes[SF_xmat] = 9 * nmb; sizes[SF_xipos] = 3 * nmb;
  sizes[SF_cdof] = 6 * nv; sizes[SF_cinert] = 10 * nmb; sizes[SF_cfrc] = 10 * nmb; sizes[SF_cvel] = 6 * nmb; sizes[SF_cacc] = 6 * nmb;
  sizes[SF_gpos] = 3 * std::max(1, ngdyn); sizes[SF_gmat] = 9 * std::max(1, ngdyn);
  sizes[SF_spos] = 3 * std::max(1, m.nsite); sizes[SF_smat] = 9 * std::max(1, m.nsite);
  const int tri = nv * (nv + 1) / 2;  // packed lower triangle
  sizes[SF_M] = tri; sizes[SF_H] = tri;
  sizes[SF_cand] = dm.maxcand;
  sizes[SF_con] = CON_STRIDE * dm.maxcon;
  // (the epilogue re-uses J: plugin store rows, actions, step counter, then the fp64 agent - target distance table)
  const int plug_words = MJB_MAX_AGENTS * (MJB_STORE_I_COUNT + MJB_STORE_F_COUNT) + 64 + 4 + 2 * std::max(1, spec.n_agents * std::max(1, spec.n_targets));
  sizes[SF_J] = std::max(3 * dm.maxcon * dm.ldj, plug_words);
  if (spec.n_agents * MJB_STORE_I_COUNT > 64 || spec.n_agents * r4(std::max(1, spec.act_dim)) > 64 || spec.n_agents * MJB_STORE_F_COUNT > 32)
    throw std::runtime_error("kernel limit: per-env plugin rows exceed the epilogue staging area");
  sizes[SF_efcD] = sizes[SF_efcAref] = sizes[SF_efcJar] = sizes[SF_efcJv] = dm.maxefc;
  sizes[SF_vecA] = sizes[SF_vecB] = sizes[SF_vecC] = sizes[SF_vecD] = nv;
  sizes[SF_rk] = m.integrator == MJB_INT_RK4 ? (m.nq + 3 * nv) : 1;
  sizes[SF_sens] = std::max(1, m.nsensordata);
  if (lite) {
    // skipFrames = 0 ("literal" benchmark configuration): no physics pass ever runs in a step, so an env only
    // needs its state rows and the epilogue staging area -> many more envs in flight per SM
    for (int i = 0; i < SF_COUNT; i++)
      if (i != SF_qpos && i != SF_qvel && i != SF_qacc && i != SF_ctrl && i != SF_qfrc && i != SF_sens && i != SF_J) sizes[i] = 0;
    sizes[SF_J] = plug_words;
  }
  // lifetime aliasing: the Hessian lives where cinert + cfrc were (composite inertias and body forces, dead once
  // dyn_backward has built M and qfrc_smooth), the broad-phase candidate list where cvel + cacc are (dead between the
  // bias pass and the sensors)
  const bool alias_H = !lite && tri <= r4(sizes[SF_cinert]) + r4(sizes[SF_cfrc]);
  if (dm.maxcand > r4(sizes[SF_cvel]) + r4(sizes[SF_cacc])) dm.maxcand = std::max(32, r4(sizes[SF_cvel]) + r4(sizes[SF_cacc]) - 4);
  const bool alias_cand = !lite && dm.maxcand <= r4(sizes[SF_cvel]) + r4(sizes[SF_cacc]);
  // without acceleration-stage sensors nothing touches cvel / cacc after the bias pass: the contact
  // records can live there too (behind the candidate list)
  bool alias_con = false;
  if (alias_cand && !dm.need_acc_sensors) {
    int room = r4(sizes[SF_cvel]) + r4(sizes[SF_cacc]) - r4(sizes[SF_con]);
    if (room >= 64) { alias_con = true; dm.maxcand = std::min(dm.maxcand, room & ~3); }
  }
  sizes[SF_cand] = dm.maxcand;
  // the per-row constraint vectors and the nv-sized solver temporaries live where xquat + xmat + xipos
  // were: those are dead once the kinematics pass has produced geom frames, inertias and probes
  const int solver_fields[8] = {SF_efcD, SF_efcAref, SF_efcJar, SF_efcJv, SF_vecC, SF_vecD, SF_vecA, SF_vecB};
  const int dead_words = r4(sizes[SF_xquat]) + r4(sizes[SF_xmat]) + r4(sizes[SF_xipos]);
  bool aliased[SF_COUNT] = {false};
  {
    int used = 0;  // greedy: as many of the solver fields as fit into the dead region
    for (int f : solver_fields)
      if (!lite && used + r4(sizes[f]) <= dead_words) { aliased[f] = true; used += r4(sizes[f]); }
  }
  int off = 0;
  for (int i = 0; i < SF_COUNT; i++) {
    if (i == SF_H && alias_H) { dm.soff[i] = dm.soff[SF_cinert]; continue; }
    if (i == SF_cand && alias_cand) { dm.soff[i] = dm.soff[SF_cvel]; continue; }
    if (i == SF_con && alias_con) { dm.soff[i] = dm.soff[SF_cvel] + r4(dm.maxcand); continue; }
    if (aliased[i]) continue;  // placed below
    dm.soff[i] = off; off += r4(sizes[i]);
  }
  {
    int o = dm.soff[SF_xquat];
    for (int f : solver_fields)
      if (aliased[f]) { dm.soff[f] = o; o += r4(sizes[f]); }
  }
  if (dm.prm_n > 0) { dm.prm_soff = off; off += r4(dm.prm_n); }   // the env's parameters: live through the whole pass
  dm.env_words = off;

  // ---- HBM row strides (16-byte aligned rows)
  int max_obs = 1;
  for (int a = 0; a < spec.n_agents; a++) max_obs = std::max(max_obs, spec.obs_dim[a]);
  dm.pack = pack; dm.a1 = spec.n_agents / pack; dm.t1 = spec.n_targets / pack; dm.nq1 = m.nq / pack; dm.nv1 = m.nv / pack;
  dm.nu1 = m.nu / pack; dm.ns1 = m.nsensordata / pack; dm.np1 = dm.nprobe / pack; dm.ngeom1 = m.ngeom / pack;
  dm.qpos_stride = r4(dm.nq1); dm.qvel_stride = r4(dm.nv1); dm.ctrl_stride = r4(std::max(1, dm.nu1));
  dm.sensor_stride = r4(std::max(1, dm.ns1)); dm.act_stride = r4(std::max(1, spec.act_dim));
  dm.obs_stride = r4(max_obs); dm.store_i32 = MJB_STORE_I_COUNT; dm.store_f32 = MJB_STORE_F_COUNT;
}

inline void fill_layout(const DevModel& dm, int num_envs, mjb_layout& L) {
  L.num_envs = num_envs; L.qpos_stride = dm.qpos_stride; L.qvel_stride = dm.qvel_stride; L.ctrl_stride = dm.ctrl_stride;
  L.sensor_stride = dm.sensor_stride; L.act_stride = dm.act_stride; L.obs_stride = dm.obs_stride;
  L.probe_count = dm.np1; L.maxcon = dm.maxcon1; L.store_i32 = dm.store_i32; L.store_f32 = dm.store_f32;
}


// ---- env packing: K real envs per warp through a K-fold replicated model + a matching virtual env spec ----
struct PackedModel {
  int K = 1;
  HostModel rep;                       // replicated model (K >= 2 only)
  std::vector<int32_t> act_index, obs_index;
  mjb_env_spec vspec;
};

// how many real envs share one warp: as many copies as fit the lane / agent / target limits
inline int choose_pack(const HostModel& host, const mjb_env_spec& spec, int num_envs) {
  int nv = host.get_int("nv");
  int K = 32 / std::max(1, nv);
  if (spec.n_agents > 0) K = std::min(K, MJB_MAX_AGENTS / spec.n_agents);
  if (spec.n_targets > 0) K = std::min(K, MJB_MAX_TARGETS / spec.n_targets);
  K = std::min(K, std::min(4, env_int("MJB_PACK", 4)));   // 4 = MJB_MAX_PACK (per-copy contact quotas in step_kernel.cuh)
  K = std::min(K, num_envs);
  if (spec.skip_frames == 0) K = 1;   // no physics in the step: nothing to share
  if ((spec.flags & MJB_SPEC_NO_PACK) || spec.n_extra_probes > 0) K = 1;
  return std::max(1, K);
}

inline void make_packed(const HostModel& host, const mjb_env_spec& spec, int K, PackedModel& out) {
  out.K = K;
  out.vspec = spec;
  if (K <= 1) return;
  replicate_model(host, K, out.rep);
  const int nq = host.get_int("nq"), nv = host.get_int("nv"), nu = host.get_int("nu"), ns = host.get_int("nsensordata"),
            nbody = host.get_int("nbody"), ngeom = host.get_int("ngeom");
  mjb_env_spec& v = out.vspec;
  const int A = spec.n_agents, T = spec.n_targets, n_act = A * spec.n_phys_act, n_obs = spec.obs_adr[A];
  v.n_agents = A * K; v.n_targets = T * K;
  out.act_index.clear(); out.obs_index.clear();
  for (int c = 0; c < K; c++) {
    for (int a = 0; a < A; a++) {
      v.obs_dim[c * A + a] = spec.obs_dim[a];
      int b = spec.agent_body[a];
      v.agent_body[c * A + a] = b <= 0 ? b : 1 + c * (nbody - 1) + (b - 1);
      v.obs_adr[c * A + a] = c * n_obs + spec.obs_adr[a];
    }
    for (int i = 0; i < n_act; i++) out.act_index.push_back(spec.act_index[i] + c * (spec.free_joint ? nv : nu));
    for (int i = 0; i < n_obs; i++) {
      int e = spec.obs_index[i], kind = e >> 24, adr = e & 0xffffff;
      adr += c * (kind == 0 ? ns : (kind == 1 ? nq : nv));
      out.obs_index.push_back((kind << 24) | adr);
    }
    for (int t = 0; t < T; t++) {
      v.target_objtype[c * T + t] = spec.target_objtype[t];
      int id = spec.target_objid[t];
      v.target_objid[c * T + t] = spec.target_objtype[t] == MJB_OBJ_BODY ? (id <= 0 ? id : 1 + c * (nbody - 1) + (id - 1)) : id + c * ngeom;
    }
  }
  v.obs_adr[A * K] = K * n_obs;
  if (out.act_index.empty()) out.act_index.push_back(0);
  if (out.obs_index.empty()) out.obs_index.push_back(0);
  v.act_index = out.act_index.data();
  v.obs_index = out.obs_index.data();
}

}  // namespace mjb
