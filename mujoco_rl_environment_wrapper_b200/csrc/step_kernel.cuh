// step_kernel.cuh — one warp = one environment: the batched MuJoCoRL.step hot path.
//
// Replaces, per environment (paths relative to the reference repo):
//   apply_action + skip_frames x mj.mj_step      MuJoCo_Gym/mujoco_parent.py:316-336
//   get_observations                             MuJoCo_Gym/mujoco_parent.py:380-392
//   dynamics / reward / truncation / done loops  MuJoCo_Gym/mujoco_rl.py:215-241,262-288,406-417
//   reset                                        MuJoCo_Gym/mujoco_rl.py:291-331, mujoco_parent.py:341-358
// The physics restates MuJoCo's documented forward-dynamics pipeline for the MJCF subset in use
// (kinematics, composite inertia, RNE bias, primitive collisions, soft limit + pyramidal contact
// constraints, primal Newton solve, semi-implicit Euler with implicit joint damping / RK4, sensors).
//
// Mapping: lane = body / dof / geom / collision pair / constraint row depending on the phase, all
// scratch in shared memory, model constants in shared memory (staged by TMA bulk copy), fp32.
// The file is plain C++ over the primitives in warp_prims.cuh so that it also compiles for the host
// SIMT emulator in tests/emu (debug tooling only).
#pragma once
#include "../../include/mjb.h"
#include "dev_model.h"
#include "warp_prims.cuh"

namespace mjb {

#define MJB_MINVAL 1e-15f
#define MJB_MAX_PACK 4   // real envs per warp at most (replicate.h, choose_pack)
#define MJB_BIG 1e30f

struct f3 { float x, y, z; };
struct q4 { float w, x, y, z; };
MJB_DEV f3 mk3(float x, float y, float z) { f3 r; r.x = x; r.y = y; r.z = z; return r; }
MJB_DEV f3 operator+(f3 a, f3 b) { return mk3(a.x + b.x, a.y + b.y, a.z + b.z); }
MJB_DEV f3 operator-(f3 a, f3 b) { return mk3(a.x - b.x, a.y - b.y, a.z - b.z); }
MJB_DEV f3 operator*(f3 a, float s) { return mk3(a.x * s, a.y * s, a.z * s); }
MJB_DEV float dot(f3 a, f3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
MJB_DEV f3 cross(f3 a, f3 b) { return mk3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x); }
MJB_DEV f3 ld3(const float* p) { return mk3(p[0], p[1], p[2]); }
MJB_DEV void st3(float* p, f3 v) { p[0] = v.x; p[1] = v.y; p[2] = v.z; }
MJB_DEV float comp(f3 v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : v.z); }
MJB_DEV q4 ldq(const float* p) { q4 q; q.w = p[0]; q.x = p[1]; q.y = p[2]; q.z = p[3]; return q; }
MJB_DEV q4 qmul(q4 a, q4 b) {
  q4 r;
  r.w = a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z;
  r.x = a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y;
  r.y = a.w * b.y - a.x * b.z + a.y * b.w + a.z * b.x;
  r.z = a.w * b.z + a.x * b.y - a.y * b.x + a.z * b.w;
  return r;
}
MJB_DEV q4 qnorm(q4 q) {
  float n2 = q.w * q.w + q.x * q.x + q.y * q.y + q.z * q.z;
  if (n2 < 1e-30f) { q.w = 1; q.x = q.y = q.z = 0; return q; }
  float inv = 1.0f / sqrtf(n2);
  q.w *= inv; q.x *= inv; q.y *= inv; q.z *= inv;
  return q;
}
MJB_DEV void q2m(q4 q, float* m) {
  float ww = q.w * q.w, xx = q.x * q.x, yy = q.y * q.y, zz = q.z * q.z;
  m[0] = ww + xx - yy - zz; m[4] = ww - xx + yy - zz; m[8] = ww - xx - yy + zz;
  m[1] = 2 * (q.x * q.y - q.w * q.z); m[2] = 2 * (q.x * q.z + q.w * q.y);
  m[3] = 2 * (q.x * q.y + q.w * q.z); m[5] = 2 * (q.y * q.z - q.w * q.x);
  m[6] = 2 * (q.x * q.z - q.w * q.y); m[7] = 2 * (q.y * q.z + q.w * q.x);
}
MJB_DEV f3 mulv(const float* m, f3 v) {
  return mk3(m[0] * v.x + m[1] * v.y + m[2] * v.z, m[3] * v.x + m[4] * v.y + m[5] * v.z, m[6] * v.x + m[7] * v.y + m[8] * v.z);
}
MJB_DEV f3 mulTv(const float* m, f3 v) {
  return mk3(m[0] * v.x + m[3] * v.y + m[6] * v.z, m[1] * v.x + m[4] * v.y + m[7] * v.z, m[2] * v.x + m[5] * v.y + m[8] * v.z);
}
MJB_DEV f3 colv(const float* m, int c) { return mk3(m[c], m[3 + c], m[6 + c]); }
MJB_DEV f3 qrot(q4 q, f3 v) {
  // v + 2 w (u x v) + 2 u x (u x v)
  f3 u = mk3(q.x, q.y, q.z);
  f3 t = cross(u, v) * 2.0f;
  return v + t * q.w + cross(u, t);
}
MJB_DEV q4 axisangle(f3 ax, float ang) {
  float s, c;
  sincosf(0.5f * ang, &s, &c);
  q4 q; q.w = c; q.x = ax.x * s; q.y = ax.y * s; q.z = ax.z * s;
  return q;
}

// ---- kernel context ----------------------------------------------------------------------------
struct Ctx {
  const DM* dm;
  const uint32_t* img;  // constant image (shared memory)
  float* s;             // this env's scratch (shared memory)
  int lane;
  float* probe;         // exported positions of this env (shared memory, 4 floats per probe)
  int cta_threads;      // threads of the CTA busy in this lock-step round (0 / 32: no CTA-level alignment after the solve)
  float* probe_quat;    // this env's exported orientations in GLOBAL memory (4 floats per probe) or null
  uint64_t* img_bar;    // first round of a launch: barrier of the image's bulk copy, waited on at the first use of the image (else null)
#if defined(MJB_PHASE_PROF)
  long long* t_last;    // profiling build only: clock of the previous phase mark (lane 0)
#endif
};
// Phase profile (debug build -DMJB_PHASE_PROF, tools/phase_prof.py): lane 0 of every env-warp adds the clock cycles since
// its previous mark to a global per-phase counter.  Compiled out of the product build.
enum { PH_LOAD, PH_FK, PH_CRB, PH_RNE, PH_COLLIDE, PH_SENS, PH_CONSTR, PH_NEWTON_INIT, PH_NEWTON_GRAD, PH_NEWTON_HESS, PH_NEWTON_FACTOR,
       PH_NEWTON_LS, PH_INTEGRATE, PH_STORE, PH_EPILOGUE, PH_BARRIER, PH_ALIGN, PH_LS_ROWSMUL, PH_LS_MV, PH_LS_LOOP, PH_EPI_OBS, PH_EPI_STAGE, PH_EPI_PLUG, PH_COUNT };
#if defined(MJB_PHASE_PROF) && !defined(MJB_HOST_EMU)
__device__ unsigned long long g_phase_cycles[32];
__device__ __forceinline__ void mjb_phase(long long* t_last, int lane, int id) {
  __syncwarp();
  if (lane == 0) { long long t = clock64(); atomicAdd(&g_phase_cycles[id], (unsigned long long)(t - *t_last)); *t_last = t; }
}
#define MJB_PH(c, id) mjb_phase((c).t_last, (c).lane, (id))
#define MJB_COUNT(c, slot, n) do { if ((c).lane == 0) atomicAdd(&g_phase_cycles[slot], (unsigned long long)(n)); } while (0)
#else
#define MJB_PH(c, id) ((void)0)
#define MJB_COUNT(c, slot, n) ((void)0)
#endif
#if defined(MJB_SPEC)
#define MJB_OFF(f) spec_off[IF_##f]
#define MJB_SOFF(f) spec_soff[SF_##f]
#else
#define MJB_OFF(f) c.dm->off[IF_##f]
#define MJB_SOFF(f) c.dm->soff[SF_##f]
#endif
#define CI(f) ((const int*)(c.img + MJB_OFF(f)))
#define CU(f) ((const uint32_t*)(c.img + MJB_OFF(f)))
#define CF(f) ((const float*)(c.img + MJB_OFF(f)))
#define SF(f) (c.s + MJB_SOFF(f))
#define SI(f) ((int*)(c.s + MJB_SOFF(f)))
// a parameter of the per-env table (DESIGN §5e): the env's value in its scratch block under PRM, else the image's
#define PF(f, blk) (PRM ? c.s + c.dm->prm_soff + (blk) : CF(f))

// packed lower triangle: element (i, j), j <= i.  Lane i reading (i, k) is bank-conflict free for
// i < 32 (triangular numbers are distinct mod 32).
MJB_DEV int tri(int i, int j) { return ((i * (i + 1)) >> 1) + j; }

// spatial helpers: motion [w; v], force [n; f], inertia {m, h(3), I(6: xx yy zz xy xz yz)} about o
MJB_DEV void inertia_mul(const float* I, f3 w, f3 v, f3& n, f3& f) {
  f3 h = mk3(I[1], I[2], I[3]);
  f = v * I[0] + cross(w, h);
  f3 Iw = mk3(I[4] * w.x + I[7] * w.y + I[8] * w.z, I[7] * w.x + I[5] * w.y + I[9] * w.z, I[8] * w.x + I[9] * w.y + I[6] * w.z);
  n = Iw + cross(h, v);
}

// =================================================================================================
// kinematics: body frames, motion subspaces (about the tree root's origin), inertias, geom frames
MJB_DEV void fk(const Ctx& c) {
  const DM& dm = *c.dm;
  const int* level_adr = CI(level_adr);
  float* qpos = SF(qpos);
  float *xpos = SF(xpos), *xquat = SF(xquat), *xmat = SF(xmat), *xipos = SF(xipos), *cdof = SF(cdof);
  MJB_NOUNROLL
  for (int l = 0; l < dm.nlevel; l++) {
    MJB_NOUNROLL
    for (int b = level_adr[l] + c.lane; b < level_adr[l + 1]; b += 32) {
      int p = CI(mb_parent)[b], root = CI(mb_root)[b];
      f3 pos = ld3(CF(mb_pos) + 3 * b);
      q4 quat = ldq(CF(mb_quat) + 4 * b);
      if (p >= 0) {
        pos = ld3(xpos + 3 * p) + mulv(xmat + 9 * p, pos);
        quat = qmul(ldq(xquat + 4 * p), quat);
      }
      int ja = CI(mb_jntadr)[b], jn = CI(mb_jntnum)[b];
      MJB_NOUNROLL
      for (int j = ja; j < ja + jn; j++) {
        int type = CI(jnt_type)[j], qa = CI(jnt_qposadr)[j], da = CI(jnt_dofadr)[j];
        if (type == MJB_JNT_FREE) {
          pos = ld3(qpos + qa);
          quat = qnorm(ldq(qpos + qa + 3));
          qpos[qa + 3] = quat.w; qpos[qa + 4] = quat.x; qpos[qa + 5] = quat.y; qpos[qa + 6] = quat.z;
        } else {
          f3 jpos = ld3(CF(jnt_pos) + 3 * j), jax = ld3(CF(jnt_axis) + 3 * j);
          f3 anchor = pos + qrot(quat, jpos), axis = qrot(quat, jax);
          float q = qpos[qa] - CF(jnt_qpos0)[j];
          // stash [axis; anchor] now, converted to a motion vector once the tree origin is known
          st3(cdof + 6 * da, axis); st3(cdof + 6 * da + 3, anchor);
          if (type == MJB_JNT_HINGE) {
            quat = qmul(quat, axisangle(jax, q));
            pos = anchor - qrot(quat, jpos);
          } else {
            pos = pos + axis * q;
          }
        }
      }
      quat = qnorm(quat);
      float R[9];
      q2m(quat, R);
      st3(xpos + 3 * b, pos);
      xquat[4 * b] = quat.w; xquat[4 * b + 1] = quat.x; xquat[4 * b + 2] = quat.y; xquat[4 * b + 3] = quat.z;
#pragma unroll
      for (int i = 0; i < 9; i++) xmat[9 * b + i] = R[i];
      st3(xipos + 3 * b, pos + mulv(R, ld3(CF(mb_ipos) + 3 * b)));
      f3 o = (root == b) ? pos : ld3(xpos + 3 * root);
      MJB_NOUNROLL
      for (int j = ja; j < ja + jn; j++) {
        int type = CI(jnt_type)[j], da = CI(jnt_dofadr)[j];
        if (type == MJB_JNT_FREE) {
          for (int i = 0; i < 3; i++) {
            st3(cdof + 6 * (da + i), mk3(0, 0, 0));
            st3(cdof + 6 * (da + i) + 3, mk3(i == 0, i == 1, i == 2));
            f3 ax = colv(R, i);
            st3(cdof + 6 * (da + 3 + i), ax);
            st3(cdof + 6 * (da + 3 + i) + 3, cross(ax, o - pos));
          }
        } else if (type == MJB_JNT_HINGE) {
          f3 axis = ld3(cdof + 6 * da), anchor = ld3(cdof + 6 * da + 3);
          st3(cdof + 6 * da + 3, cross(axis, o - anchor));
        } else {
          f3 axis = ld3(cdof + 6 * da);
          st3(cdof + 6 * da, mk3(0, 0, 0)); st3(cdof + 6 * da + 3, axis);
        }
      }
    }
    MJB_SYNC();
  }
  // body inertias about the tree origin
  float* cinert = SF(cinert);
  MJB_NOUNROLL
  for (int b = c.lane; b < dm.nmb; b += 32) {
    float R[9];
    q2m(qmul(ldq(xquat + 4 * b), ldq(CF(mb_iquat) + 4 * b)), R);
    f3 I = ld3(CF(mb_inertia) + 3 * b);
    float m = CF(mb_mass)[b];
    f3 cc = ld3(xipos + 3 * b) - ld3(xpos + 3 * CI(mb_root)[b]);
    float* o = cinert + 10 * b;
    o[0] = m; o[1] = m * cc.x; o[2] = m * cc.y; o[3] = m * cc.z;
    o[4] = R[0] * R[0] * I.x + R[1] * R[1] * I.y + R[2] * R[2] * I.z + m * (cc.y * cc.y + cc.z * cc.z);
    o[5] = R[3] * R[3] * I.x + R[4] * R[4] * I.y + R[5] * R[5] * I.z + m * (cc.x * cc.x + cc.z * cc.z);
    o[6] = R[6] * R[6] * I.x + R[7] * R[7] * I.y + R[8] * R[8] * I.z + m * (cc.x * cc.x + cc.y * cc.y);
    o[7] = R[0] * R[3] * I.x + R[1] * R[4] * I.y + R[2] * R[5] * I.z - m * cc.x * cc.y;
    o[8] = R[0] * R[6] * I.x + R[1] * R[7] * I.y + R[2] * R[8] * I.z - m * cc.x * cc.z;
    o[9] = R[3] * R[6] * I.x + R[4] * R[7] * I.y + R[5] * R[8] * I.z - m * cc.y * cc.z;
  }
  // dynamic geom frames
  float *gpos = SF(gpos), *gmat = SF(gmat);
  MJB_NOUNROLL
  for (int g = c.lane; g < dm.ngeom; g += 32) {
    int slot = CI(geom_slot)[g];
    if (slot < 0) continue;
    int b = CI(geom_mb)[g];
    st3(gpos + 3 * slot, ld3(xpos + 3 * b) + mulv(xmat + 9 * b, ld3(CF(geom_pos) + 3 * g)));
    q2m(qmul(ldq(xquat + 4 * b), ldq(CF(geom_quat) + 4 * g)), gmat + 9 * slot);
  }
  float *spos = SF(spos), *smat = SF(smat);
  MJB_NOUNROLL
  for (int t = c.lane; t < dm.nsite; t += 32) {
    int b = CI(site_mb)[t];
    f3 lp = ld3(CF(site_pos) + 3 * t);
    q4 lq = ldq(CF(site_quat) + 4 * t);
    if (b >= 0) { lp = ld3(xpos + 3 * b) + mulv(xmat + 9 * b, lp); lq = qmul(ldq(xquat + 4 * b), lq); }
    st3(spos + 3 * t, lp);
    q2m(lq, smat + 9 * t);
  }
  MJB_SYNC();
}

// composite rigid body inertias and the joint-space inertia matrix (packed lower triangle)
MJB_DEV void crb_mass(const Ctx& c) {
  const DM& dm = *c.dm;
  const int* level_adr = CI(level_adr);
  float *cinert = SF(cinert), *crb = SF(crb), *M = SF(M), *cdof = SF(cdof);
  MJB_NOUNROLL
  for (int i = c.lane; i < 10 * dm.nmb; i += 32) crb[i] = cinert[i];
  MJB_NOUNROLL
  for (int i = c.lane; i < (dm.nv * (dm.nv + 1)) / 2; i += 32) M[i] = 0.f;
  MJB_SYNC();
  MJB_NOUNROLL
  for (int l = dm.nlevel - 2; l >= 0; l--) {
    MJB_NOUNROLL
    for (int b = level_adr[l] + c.lane; b < level_adr[l + 1]; b += 32) {
      int ca = CI(mb_childadr)[b], ce = CI(mb_childadr)[b + 1];
      if (ce > ca) {
        float acc[10];
#pragma unroll
        for (int i = 0; i < 10; i++) acc[i] = crb[10 * b + i];
        MJB_NOUNROLL
        for (int k = ca; k < ce; k++) {
          int ch = CI(mb_child)[k];
#pragma unroll
          for (int i = 0; i < 10; i++) acc[i] += crb[10 * ch + i];
        }
#pragma unroll
        for (int i = 0; i < 10; i++) crb[10 * b + i] = acc[i];
      }
    }
    MJB_SYNC();
  }
  MJB_NOUNROLL
  for (int i = c.lane; i < dm.nv; i += 32) {
    int b = CI(dof_mb)[i];
    f3 n, f;
    inertia_mul(crb + 10 * b, ld3(cdof + 6 * i), ld3(cdof + 6 * i + 3), n, f);
    for (int j = i; j >= 0; j = CI(dof_parent)[j]) {
      float v = dot(ld3(cdof + 6 * j), n) + dot(ld3(cdof + 6 * j + 3), f);
      if (j == i) v += CF(dof_armature)[i];
      M[tri(i, j)] = v;  // j is an ancestor dof: j <= i
    }
  }
  MJB_SYNC();
}

// velocity-dependent bias forces (Coriolis, centrifugal, gravity) by recursive Newton-Euler, then
// qfrc_smooth = passive - bias + actuation.  With `with_acc` the pass includes qacc (post-constraint
// body accelerations for the accelerometer) and only fills cvel / cacc.
MJB_DEV void rne_pass(const Ctx& c, bool with_acc) {
  const DM& dm = *c.dm;
  const int* level_adr = CI(level_adr);
  float *cdof = SF(cdof), *cvel = SF(cvel), *cacc = SF(cacc), *qvel = SF(qvel), *qacc = SF(qacc);
  float *cinert = SF(cinert), *cfrc = SF(crb);  // crb is dead after crb_mass: reuse as body force
  MJB_NOUNROLL
  for (int l = 0; l < dm.nlevel; l++) {
    MJB_NOUNROLL
    for (int b = level_adr[l] + c.lane; b < level_adr[l + 1]; b += 32) {
      int p = CI(mb_parent)[b];
      f3 w = mk3(0, 0, 0), v = mk3(0, 0, 0), aw = mk3(0, 0, 0);
      f3 av = mk3(-dm.gravity[0], -dm.gravity[1], -dm.gravity[2]);
      if (p >= 0) { w = ld3(cvel + 6 * p); v = ld3(cvel + 6 * p + 3); aw = ld3(cacc + 6 * p); av = ld3(cacc + 6 * p + 3); }
      int da = CI(mb_dofadr)[b], dn = CI(mb_dofnum)[b];
      f3 wb = w, vb = v;  // velocity snapshot for the free joint's rotational block
      MJB_NOUNROLL
      for (int d = da; d < da + dn; d++) {
        int kind = CI(dof_kind)[d];
        f3 sw = ld3(cdof + 6 * d), sv = ld3(cdof + 6 * d + 3);
        float qd = qvel[d];
        if (kind == DOF_FREE_ROT && d == da + 3) { wb = w; vb = v; }
        if (kind != DOF_FREE_TRANS) {
          f3 uw = kind == DOF_FREE_ROT ? wb : w, uv = kind == DOF_FREE_ROT ? vb : v;
          // cdof_dot = u x_m S
          aw = aw + cross(uw, sw) * qd;
          av = av + (cross(uw, sv) + cross(uv, sw)) * qd;
        }
        if (with_acc) { aw = aw + sw * qacc[d]; av = av + sv * qacc[d]; }
        w = w + sw * qd; v = v + sv * qd;
      }
      st3(cvel + 6 * b, w); st3(cvel + 6 * b + 3, v);
      st3(cacc + 6 * b, aw); st3(cacc + 6 * b + 3, av);
      if (!with_acc) {
        f3 n1, f1, n2, f2;
        inertia_mul(cinert + 10 * b, aw, av, n1, f1);
        inertia_mul(cinert + 10 * b, w, v, n2, f2);
        // v x* (I v) = [w x n + v x f ; w x f]
        st3(cfrc + 10 * b, n1 + cross(w, n2) + cross(v, f2));
        st3(cfrc + 10 * b + 3, f1 + cross(w, f2));
      }
    }
    MJB_SYNC();
  }
  if (with_acc) return;
  MJB_NOUNROLL
  for (int l = dm.nlevel - 2; l >= 0; l--) {
    MJB_NOUNROLL
    for (int b = level_adr[l] + c.lane; b < level_adr[l + 1]; b += 32) {
      int ca = CI(mb_childadr)[b], ce = CI(mb_childadr)[b + 1];
      MJB_NOUNROLL
      for (int k = ca; k < ce; k++) {
        int ch = CI(mb_child)[k];
#pragma unroll
        for (int i = 0; i < 6; i++) cfrc[10 * b + i] += cfrc[10 * ch + i];
      }
    }
    MJB_SYNC();
  }
  float *qfrc = SF(qfrc), *ctrl = SF(ctrl);
  MJB_NOUNROLL
  for (int d = c.lane; d < dm.nv; d += 32) {
    int b = CI(dof_mb)[d];
    float bias = dot(ld3(cdof + 6 * d), ld3(cfrc + 10 * b)) + dot(ld3(cdof + 6 * d + 3), ld3(cfrc + 10 * b + 3));
    float f = -CF(dof_damping)[d] * qvel[d] - bias;
    MJB_NOUNROLL
    for (int k = CI(dof_actadr)[d]; k < CI(dof_actadr)[d] + CI(dof_actnum)[d]; k++) {
      int u = CI(act_list)[k];
      const float* ap = CF(act_param) + 4 * u;
      float cv = ctrl[u];
      if (ap[1] != 0.f) cv = fminf(ap[3], fmaxf(ap[2], cv));
      f += ap[0] * cv;
    }
    qfrc[d] = f;
  }
  MJB_SYNC();
}

// ---- fused passes of the step proper -------------------------------------------------------------------------------
// kin_forward = fk + the outward half of rne_pass in ONE walk over the tree levels: per body its frame, motion subspaces
// (about the tree root's origin), spatial inertia, velocity, bias acceleration and its own inertial force
// I a + v x* I v.  Composite inertias later accumulate IN PLACE in SF_cinert; SF_crb holds the body forces.
// dyn_backward = the inward halves of crb_mass and rne_pass in one walk (16 words per body), then one loop over the dofs
// for the rows of M and qfrc_smooth.  (fk / crb_mass / rne_pass stay for the renderer and the accelerometer pass.)
template <bool PRM = false>
MJB_DEV void kin_forward(const Ctx& c) {
  const DM& dm = *c.dm;
  const int* level_adr = CI(level_adr);
  float *qpos = SF(qpos), *qvel = SF(qvel);
  float *xpos = SF(xpos), *xquat = SF(xquat), *xmat = SF(xmat), *xipos = SF(xipos), *cdof = SF(cdof);
  float *cinert = SF(cinert), *cfrc = SF(crb), *cvel = SF(cvel), *cacc = SF(cacc);
  MJB_NOUNROLL
  for (int l = 0; l < dm.nlevel; l++) {
    MJB_NOUNROLL
    for (int b = level_adr[l] + c.lane; b < level_adr[l + 1]; b += 32) {
      const int p = CI(mb_parent)[b], root = CI(mb_root)[b];
      f3 pos = ld3(CF(mb_pos) + 3 * b);
      q4 quat = ldq(CF(mb_quat) + 4 * b);
      if (p >= 0) {
        pos = ld3(xpos + 3 * p) + mulv(xmat + 9 * p, pos);
        quat = qmul(ldq(xquat + 4 * p), quat);
      }
      const int ja = CI(mb_jntadr)[b], jn = CI(mb_jntnum)[b];
      MJB_NOUNROLL
      for (int j = ja; j < ja + jn; j++) {
        int type = CI(jnt_type)[j], qa = CI(jnt_qposadr)[j], da = CI(jnt_dofadr)[j];
        if (type == MJB_JNT_FREE) {
          pos = ld3(qpos + qa);
          quat = qnorm(ldq(qpos + qa + 3));
          qpos[qa + 3] = quat.w; qpos[qa + 4] = quat.x; qpos[qa + 5] = quat.y; qpos[qa + 6] = quat.z;
        } else {
          f3 jpos = ld3(CF(jnt_pos) + 3 * j), jax = ld3(CF(jnt_axis) + 3 * j);
          f3 anchor = pos + qrot(quat, jpos), axis = qrot(quat, jax);
          float q = qpos[qa] - CF(jnt_qpos0)[j];
          st3(cdof + 6 * da, axis); st3(cdof + 6 * da + 3, anchor);   // [axis; anchor] until the tree origin is known
          if (type == MJB_JNT_HINGE) {
            quat = qmul(quat, axisangle(jax, q));
            pos = anchor - qrot(quat, jpos);
          } else {
            pos = pos + axis * q;
          }
        }
      }
      quat = qnorm(quat);
      float R[9];
      q2m(quat, R);
      st3(xpos + 3 * b, pos);
      xquat[4 * b] = quat.w; xquat[4 * b + 1] = quat.x; xquat[4 * b + 2] = quat.y; xquat[4 * b + 3] = quat.z;
#pragma unroll
      for (int i = 0; i < 9; i++) xmat[9 * b + i] = R[i];
      const f3 ipos = pos + mulv(R, ld3(CF(mb_ipos) + 3 * b));
      st3(xipos + 3 * b, ipos);
      const f3 o = (root == b) ? pos : ld3(xpos + 3 * root);
      MJB_NOUNROLL
      for (int j = ja; j < ja + jn; j++) {
        int type = CI(jnt_type)[j], da = CI(jnt_dofadr)[j];
        if (type == MJB_JNT_FREE) {
          for (int i = 0; i < 3; i++) {
            st3(cdof + 6 * (da + i), mk3(0, 0, 0));
            st3(cdof + 6 * (da + i) + 3, mk3(i == 0, i == 1, i == 2));
            f3 ax = colv(R, i);
            st3(cdof + 6 * (da + 3 + i), ax);
            st3(cdof + 6 * (da + 3 + i) + 3, cross(ax, o - pos));
          }
        } else if (type == MJB_JNT_HINGE) {
          f3 axis = ld3(cdof + 6 * da), anchor = ld3(cdof + 6 * da + 3);
          st3(cdof + 6 * da + 3, cross(axis, o - anchor));
        } else {
          f3 axis = ld3(cdof + 6 * da);
          st3(cdof + 6 * da, mk3(0, 0, 0)); st3(cdof + 6 * da + 3, axis);
        }
      }
      // velocity and bias acceleration of the body (outward pass of the recursive Newton-Euler algorithm)
      f3 w = mk3(0, 0, 0), v = mk3(0, 0, 0), aw = mk3(0, 0, 0);
      f3 av = mk3(-dm.gravity[0], -dm.gravity[1], -dm.gravity[2]);
      if (p >= 0) { w = ld3(cvel + 6 * p); v = ld3(cvel + 6 * p + 3); aw = ld3(cacc + 6 * p); av = ld3(cacc + 6 * p + 3); }
      const int da = CI(mb_dofadr)[b], dn = CI(mb_dofnum)[b];
      if (p < 0 && root == b && dn == 6 && CI(dof_kind)[da] == DOF_FREE_TRANS) {
        // free joint of a tree root (parent at rest, motion subspaces about its own origin): the six-dof loop below
        // collapses to v = qvel[0:3], w = R qvel[3:6], bias acceleration [0 ; v x w] (only 2 of 32 lanes sit at this level)
        v = ld3(qvel + da);
        w = mulv(R, ld3(qvel + da + 3));
        av = av + cross(v, w);
      } else {
        f3 wb = w, vb = v;  // velocity snapshot for the free joint's rotational block
        MJB_NOUNROLL
        for (int d = da; d < da + dn; d++) {
          const int kind = CI(dof_kind)[d];
          const f3 sw = ld3(cdof + 6 * d), sv = ld3(cdof + 6 * d + 3);
          const float qd = qvel[d];
          if (kind == DOF_FREE_ROT && d == da + 3) { wb = w; vb = v; }
          if (kind != DOF_FREE_TRANS) {
            const f3 uw = kind == DOF_FREE_ROT ? wb : w, uv = kind == DOF_FREE_ROT ? vb : v;
            aw = aw + cross(uw, sw) * qd;                              // cdof_dot = u x_m S
            av = av + (cross(uw, sv) + cross(uv, sw)) * qd;
          }
          w = w + sw * qd; v = v + sv * qd;
        }
      }
      st3(cvel + 6 * b, w); st3(cvel + 6 * b + 3, v);
      st3(cacc + 6 * b, aw); st3(cacc + 6 * b + 3, av);
    }
    MJB_SYNC();
  }
  // What does not travel along the tree runs ONCE over all bodies (lane = body) instead of once per level with a
  // handful of live lanes: spatial inertia about the tree origin and the body's inertial force I a + v x* (I v)
  MJB_NOUNROLL
  for (int b = c.lane; b < level_adr[dm.nlevel]; b += 32) {
    const f3 ipos = ld3(xipos + 3 * b), o = ld3(xpos + 3 * CI(mb_root)[b]);
    float I[10];
    {
      float Ri[9];
      q2m(qmul(ldq(xquat + 4 * b), ldq(CF(mb_iquat) + 4 * b)), Ri);
      const f3 In = ld3(PF(mb_inertia, prm_inertia(dm)) + 3 * b);
      const float m = PF(mb_mass, 0)[b];
      const f3 cc = ipos - o;
      I[0] = m; I[1] = m * cc.x; I[2] = m * cc.y; I[3] = m * cc.z;
      I[4] = Ri[0] * Ri[0] * In.x + Ri[1] * Ri[1] * In.y + Ri[2] * Ri[2] * In.z + m * (cc.y * cc.y + cc.z * cc.z);
      I[5] = Ri[3] * Ri[3] * In.x + Ri[4] * Ri[4] * In.y + Ri[5] * Ri[5] * In.z + m * (cc.x * cc.x + cc.z * cc.z);
      I[6] = Ri[6] * Ri[6] * In.x + Ri[7] * Ri[7] * In.y + Ri[8] * Ri[8] * In.z + m * (cc.x * cc.x + cc.y * cc.y);
      I[7] = Ri[0] * Ri[3] * In.x + Ri[1] * Ri[4] * In.y + Ri[2] * Ri[5] * In.z - m * cc.x * cc.y;
      I[8] = Ri[0] * Ri[6] * In.x + Ri[1] * Ri[7] * In.y + Ri[2] * Ri[8] * In.z - m * cc.x * cc.z;
      I[9] = Ri[3] * Ri[6] * In.x + Ri[4] * Ri[7] * In.y + Ri[5] * Ri[8] * In.z - m * cc.y * cc.z;
#pragma unroll
      for (int i = 0; i < 10; i++) cinert[10 * b + i] = I[i];
    }
    const f3 w = ld3(cvel + 6 * b), v = ld3(cvel + 6 * b + 3), aw = ld3(cacc + 6 * b), av = ld3(cacc + 6 * b + 3);
    f3 n1, f1, n2, f2;
    inertia_mul(I, aw, av, n1, f1);
    inertia_mul(I, w, v, n2, f2);
    st3(cfrc + 10 * b, n1 + cross(w, n2) + cross(v, f2));         // v x* (I v) = [w x n + v x f ; w x f]
    st3(cfrc + 10 * b + 3, f1 + cross(w, f2));
  }
  // dynamic geom frames
  float *gpos = SF(gpos), *gmat = SF(gmat);
  MJB_NOUNROLL
  for (int g = c.lane; g < dm.ngeom; g += 32) {
    int slot = CI(geom_slot)[g];
    if (slot < 0) continue;
    int b = CI(geom_mb)[g];
    st3(gpos + 3 * slot, ld3(xpos + 3 * b) + mulv(xmat + 9 * b, ld3(CF(geom_pos) + 3 * g)));
    q2m(qmul(ldq(xquat + 4 * b), ldq(CF(geom_quat) + 4 * g)), gmat + 9 * slot);
  }
  float *spos = SF(spos), *smat = SF(smat);
  MJB_NOUNROLL
  for (int t = c.lane; t < dm.nsite; t += 32) {
    int b = CI(site_mb)[t];
    f3 lp = ld3(CF(site_pos) + 3 * t);
    q4 lq = ldq(CF(site_quat) + 4 * t);
    if (b >= 0) { lp = ld3(xpos + 3 * b) + mulv(xmat + 9 * b, lp); lq = qmul(ldq(xquat + 4 * b), lq); }
    st3(spos + 3 * t, lp);
    q2m(lq, smat + 9 * t);
  }
  // M starts from zero (only ancestor pairs are written below)
  {
    struct alignas(16) W4 { float a, b, c, d; };
    W4* m4 = (W4*)SF(M);
    const W4 z = {0.f, 0.f, 0.f, 0.f};
    MJB_NOUNROLL
    for (int i = c.lane; i < ((dm.nv * (dm.nv + 1)) / 2 + 3) / 4; i += 32) m4[i] = z;
  }
  MJB_SYNC();
}

template <bool PRM = false>
MJB_DEV void dyn_backward(const Ctx& c) {
  const DM& dm = *c.dm;
  const int* level_adr = CI(level_adr);
  float *crb = SF(cinert), *cfrc = SF(crb), *M = SF(M), *cdof = SF(cdof), *qvel = SF(qvel);
  MJB_NOUNROLL
  for (int l = dm.nlevel - 2; l >= 0; l--) {
    MJB_NOUNROLL
    for (int b = level_adr[l] + c.lane; b < level_adr[l + 1]; b += 32) {
      const int ca = CI(mb_childadr)[b], ce = CI(mb_childadr)[b + 1];
      if (ce > ca) {
        float acc[16];
#pragma unroll
        for (int i = 0; i < 10; i++) acc[i] = crb[10 * b + i];
#pragma unroll
        for (int i = 0; i < 6; i++) acc[10 + i] = cfrc[10 * b + i];
        MJB_NOUNROLL
        for (int k = ca; k < ce; k++) {
          const int ch = CI(mb_child)[k];
#pragma unroll
          for (int i = 0; i < 10; i++) acc[i] += crb[10 * ch + i];
#pragma unroll
          for (int i = 0; i < 6; i++) acc[10 + i] += cfrc[10 * ch + i];
        }
#pragma unroll
        for (int i = 0; i < 10; i++) crb[10 * b + i] = acc[i];
#pragma unroll
        for (int i = 0; i < 6; i++) cfrc[10 * b + i] = acc[10 + i];
      }
    }
    MJB_SYNC();
  }
  float *qfrc = SF(qfrc), *ctrl = SF(ctrl);
  MJB_NOUNROLL
  for (int i = c.lane; i < dm.nv; i += 32) {
    const int b = CI(dof_mb)[i];
    const f3 sw = ld3(cdof + 6 * i), sv = ld3(cdof + 6 * i + 3);
    f3 n, f;
    inertia_mul(crb + 10 * b, sw, sv, n, f);
    MJB_NOUNROLL
    for (int j = i; j >= 0; j = CI(dof_parent)[j]) {
      float v = dot(ld3(cdof + 6 * j), n) + dot(ld3(cdof + 6 * j + 3), f);
      if (j == i) v += CF(dof_armature)[i];
      M[tri(i, j)] = v;  // j is an ancestor dof: j <= i
    }
    const float bias = dot(sw, ld3(cfrc + 10 * b)) + dot(sv, ld3(cfrc + 10 * b + 3));
    float fq = -PF(dof_damping, prm_damping(dm))[i] * qvel[i] - bias;
    MJB_NOUNROLL
    for (int k = CI(dof_actadr)[i]; k < CI(dof_actadr)[i] + CI(dof_actnum)[i]; k++) {
      int u = CI(act_list)[k];
      const float* ap = CF(act_param) + 4 * u;
      float cv = ctrl[u];
      if (ap[1] != 0.f) cv = fminf(ap[3], fmaxf(ap[2], cv));
      fq += (PRM ? c.s[dm.prm_soff + prm_gear(dm) + u] : ap[0]) * cv;
    }
    qfrc[i] = fq;
  }
  MJB_SYNC();
}

// =================================================================================================
// collision
struct GeomW { f3 pos; const float* mat; const float* size; int type; };
MJB_DEV GeomW geom_world(const Ctx& c, int g) {
  GeomW r;
  int slot = CI(geom_slot)[g];
  r.type = CI(geom_type)[g];
  r.size = CF(geom_size) + 3 * g;
  if (slot >= 0) { r.pos = ld3(SF(gpos) + 3 * slot); r.mat = SF(gmat) + 9 * slot; }
  else { r.pos = ld3(CF(geom_pos) + 3 * g); r.mat = CF(geom_mat) + 9 * g; }
  return r;
}
struct ConOut { float dist; f3 pos, n, t; };

MJB_DEV int plane_sphere(f3 pp, f3 n, f3 cs, float r, float margin, ConOut& o) {
  float dist = dot(cs - pp, n) - r;
  if (dist > margin) return 0;
  o.dist = dist; o.pos = cs - n * (r + 0.5f * dist); o.n = n; o.t = mk3(0, 0, 0);
  return 1;
}
MJB_DEV int sphere_sphere(f3 c1, float r1, f3 c2, float r2, float margin, ConOut& o) {
  f3 d = c2 - c1;
  float cd = sqrtf(dot(d, d)), dist = cd - r1 - r2;
  if (dist > margin) return 0;
  f3 n = cd < MJB_MINVAL ? mk3(1, 0, 0) : d * (1.0f / cd);
  o.dist = dist; o.pos = c1 + n * (r1 + 0.5f * dist); o.n = n; o.t = mk3(0, 0, 0);
  return 1;
}
MJB_DEV int sphere_box(f3 c1, float r, f3 c2, const float* R2, const float* size, float margin, ConOut& o) {
  f3 cl = mulTv(R2, c1 - c2);
  f3 cp = mk3(fminf(size[0], fmaxf(-size[0], cl.x)), fminf(size[1], fmaxf(-size[1], cl.y)), fminf(size[2], fmaxf(-size[2], cl.z)));
  bool inside = (cp.x == cl.x) && (cp.y == cl.y) && (cp.z == cl.z);
  f3 nl = mk3(0, 0, 0);
  float dist;
  if (inside) {
    float px = size[0] - fabsf(cl.x), py = size[1] - fabsf(cl.y), pz = size[2] - fabsf(cl.z);
    int k = 0; float best = px;
    if (py < best) { best = py; k = 1; }
    if (pz < best) { best = pz; k = 2; }
    float sg = comp(cl, k) >= 0 ? 1.f : -1.f;
    if (k == 0) nl.x = -sg; else if (k == 1) nl.y = -sg; else nl.z = -sg;
    dist = -best - r;
  } else {
    f3 d = cl - cp;
    float len = sqrtf(dot(d, d));
    dist = len - r;
    if (dist > margin) return 0;
    nl = d * (-1.0f / len);
  }
  f3 n = mulv(R2, nl);
  o.dist = dist; o.pos = c1 + n * (r + 0.5f * dist); o.n = n; o.t = mk3(0, 0, 0);
  return 1;
}
MJB_DEV float point_box_dist(f3 p, const float* size) {
  float ex = fabsf(p.x) - size[0], ey = fabsf(p.y) - size[1], ez = fabsf(p.z) - size[2];
  float s2 = (ex > 0 ? ex * ex : 0.f) + (ey > 0 ? ey * ey : 0.f) + (ez > 0 ? ez * ez : 0.f);
  return s2 > 0 ? sqrtf(s2) : fmaxf(ex, fmaxf(ey, ez));
}
// capsule - box (specification: DESIGN.md 3c; the fp64 checker finds the same minimiser exactly, by breakpoints).
//   1. t* = argmin over the capsule axis p(t) = c + t d, t in [-1, 1], of the signed distance to the box
//      (convex in t: golden-section search, then compared with the two ends);
//   2. inside the box: one sphere there;
//   3. else k = dominant axis of (p* - closest box point) = the closest FACE, I = the part of the segment whose
//      projection lies in that face's rectangle; t* in I (within 0.05): spheres at the two ends of I, deeper
//      first (ends closer than 1e-3 count once); otherwise one sphere at t*.
// Every sphere goes through sphere - box with the pair's margin.
MJB_DEV int capsule_box(const GeomW& g1, const GeomW& g2, float margin, ConOut* o) {
  const float r = g1.size[0], h = g1.size[1];
  const f3 ax = colv(g1.mat, 2);
  const f3 c = mulTv(g2.mat, g1.pos - g2.pos), d = mulTv(g2.mat, ax) * h;
  float lo = -1.f, hi = 1.f;
  const float gr = 0.6180339887f;
  float x1 = hi - gr * (hi - lo), x2 = lo + gr * (hi - lo);
  float f1 = point_box_dist(c + d * x1, g2.size), f2 = point_box_dist(c + d * x2, g2.size);
  MJB_NOUNROLL
  for (int it = 0; it < 40; it++) {
    if (f1 <= f2) { hi = x2; x2 = x1; f2 = f1; x1 = hi - gr * (hi - lo); f1 = point_box_dist(c + d * x1, g2.size); }
    else { lo = x1; x1 = x2; f1 = f2; x2 = lo + gr * (hi - lo); f2 = point_box_dist(c + d * x2, g2.size); }
  }
  float ts = 0.5f * (lo + hi), best = point_box_dist(c + d * ts, g2.size);
  const float fm = point_box_dist(c - d, g2.size), fp = point_box_dist(c + d, g2.size);
  if (fm <= best) { best = fm; ts = -1.f; }
  if (fp < best) { best = fp; ts = 1.f; }
  if (best > margin + r) return 0;
  if (best <= 0.f) return sphere_box(g1.pos + ax * (ts * h), r, g2.pos, g2.mat, g2.size, margin, o[0]);
  const f3 p = c + d * ts;
  const float sx = fabsf(p.x - fminf(g2.size[0], fmaxf(-g2.size[0], p.x))), sy = fabsf(p.y - fminf(g2.size[1], fmaxf(-g2.size[1], p.y))),
              sz = fabsf(p.z - fminf(g2.size[2], fmaxf(-g2.size[2], p.z)));
  int kf = 0;
  if (sy > sx) kf = 1;
  if (sz > (kf ? sy : sx)) kf = 2;
  float tl = -1.f, th = 1.f;
#pragma unroll
  for (int j = 0; j < 3; j++) {
    if (j == kf) continue;
    const float cj = comp(c, j), dj = comp(d, j), sj = g2.size[j];
    if (fabsf(dj) < 1e-12f) { if (fabsf(cj) > sj) { tl = 1.f; th = -1.f; } continue; }
    const float inv = 1.f / dj, t0 = (-sj - cj) * inv, t1 = (sj - cj) * inv;
    tl = fmaxf(tl, fminf(t0, t1)); th = fminf(th, fmaxf(t0, t1));
  }
  if (tl > th || ts < tl - 0.05f || ts > th + 0.05f) return sphere_box(g1.pos + ax * (ts * h), r, g2.pos, g2.mat, g2.size, margin, o[0]);
  const bool lo_first = point_box_dist(c + d * tl, g2.size) <= point_box_dist(c + d * th, g2.size);
  const float ta = lo_first ? tl : th, tb = lo_first ? th : tl;
  int n = sphere_box(g1.pos + ax * (ta * h), r, g2.pos, g2.mat, g2.size, margin, o[0]);
  if (th - tl > 1e-3f) n += sphere_box(g1.pos + ax * (tb * h), r, g2.pos, g2.mat, g2.size, margin, o[n]);
  return n;
}
MJB_DEV int capsule_capsule(const GeomW& g1, const GeomW& g2, float margin, ConOut* o) {
  f3 a1 = colv(g1.mat, 2), a2 = colv(g2.mat, 2), dif = g1.pos - g2.pos;
  float len1 = g1.size[1], len2 = g2.size[1], r1 = g1.size[0], r2 = g2.size[0];
  float mb = -dot(a1, a2), u = -dot(a1, dif), v = dot(a2, dif), det = 1.f - mb * mb;
  if (fabsf(det) >= 1e-7f) {
    float x1 = (u - mb * v) / det, x2 = (v - mb * u) / det;
    if (x1 > len1) { x1 = len1; x2 = v - mb * len1; }
    else if (x1 < -len1) { x1 = -len1; x2 = v + mb * len1; }
    if (x2 > len2) { x2 = len2; x1 = u - mb * len2; }
    else if (x2 < -len2) { x2 = -len2; x1 = u + mb * len2; }
    x1 = fminf(len1, fmaxf(-len1, x1));
    return sphere_sphere(g1.pos + a1 * x1, r1, g2.pos + a2 * x2, r2, margin, o[0]);
  }
  int k = 0;
  MJB_NOUNROLL
  for (int e = 0; e < 2 && k < 2; e++) {
    float x1 = e == 0 ? len1 : -len1, x2 = fminf(len2, fmaxf(-len2, v - mb * x1));
    k += sphere_sphere(g1.pos + a1 * x1, r1, g2.pos + a2 * x2, r2, margin, o[k]);
  }
  MJB_NOUNROLL
  for (int e = 0; e < 2 && k < 2; e++) {
    float x2 = e == 0 ? len2 : -len2, x1 = u - mb * x2;
    if (x1 > len1 || x1 < -len1) continue;
    k += sphere_sphere(g1.pos + a1 * x1, r1, g2.pos + a2 * x2, r2, margin, o[k]);
  }
  return k;
}

// box - box, one pair per call, the whole warp cooperating (specification: DESIGN.md 3c; the fp64 checker clips the
// incident face sequentially, Sutherland - Hodgman).  Lanes 0..14 evaluate the 15 separating axes; the contact axis is
// the face axis of largest separation unless an edge axis beats it by 5 % + 1e-6.  Face contact: the vertices of
// (incident face) n (reference rectangle) are enumerated in parallel — lanes 0..3 incident vertices inside the
// rectangle, 4..7 rectangle corners strictly inside the incident quad, 8..23 incident edge x rectangle side
// crossings — and kept when within `margin` of the reference plane.  Edge contact: lane 0, closest points of the two
// supporting edges.  Returns whether this lane holds a contact (at most 8 lanes do).
MJB_DEV bool box_box_lane(int lane, const GeomW& a, const GeomW& b, float margin, ConOut& o) {
  const f3 dc = b.pos - a.pos;
  float sp = -MJB_BIG;
  bool valid = false;
  if (lane < 15) {
    f3 L;
    if (lane < 3) { L = colv(a.mat, lane); valid = true; }
    else if (lane < 6) { L = colv(b.mat, lane - 3); valid = true; }
    else {
      const int e = lane - 6, i = e / 3, j = e - 3 * i;
      L = cross(colv(a.mat, i), colv(b.mat, j));
      const float len = sqrtf(dot(L, L));
      valid = len >= 1e-6f;
      L = L * (1.f / fmaxf(len, 1e-12f));
    }
    const f3 la = mulTv(a.mat, L), lb = mulTv(b.mat, L);
    sp = fabsf(dot(L, dc)) - (a.size[0] * fabsf(la.x) + a.size[1] * fabsf(la.y) + a.size[2] * fabsf(la.z)) -
         (b.size[0] * fabsf(lb.x) + b.size[1] * fabsf(lb.y) + b.size[2] * fabsf(lb.z));
  }
  if (MJB_BALLOT(valid && sp > margin)) return false;
  const float fsep = wmax(lane < 6 ? sp : -MJB_BIG), esep = wmax((lane >= 6 && valid) ? sp : -MJB_BIG);
  const int fax = MJB_FFS(MJB_BALLOT(lane < 6 && sp == fsep)) - 1;
  const int eax = MJB_FFS(MJB_BALLOT(lane >= 6 && valid && sp == esep)) - 7;   // -7 + ... : < 0 when no edge axis is valid
  o.t = mk3(0, 0, 0);
  if (eax >= 0 && esep > fsep + 0.05f * fabsf(fsep) + 1e-6f) {
    if (lane != 0) return false;
    const int i = eax / 3, j = eax - 3 * i;
    const f3 u = colv(a.mat, i), v = colv(b.mat, j);
    f3 L = cross(u, v);
    L = L * (1.f / sqrtf(dot(L, L)));
    if (dot(L, dc) < 0.f) L = L * -1.f;
    f3 pa = a.pos, pb = b.pos;
#pragma unroll
    for (int k = 0; k < 3; k++) {
      const f3 ak = colv(a.mat, k), bk = colv(b.mat, k);
      if (k != i) pa = pa + ak * (a.size[k] * (dot(L, ak) >= 0.f ? 1.f : -1.f));
      if (k != j) pb = pb - bk * (b.size[k] * (dot(L, bk) >= 0.f ? 1.f : -1.f));
    }
    const f3 w = pa - pb;
    const float uv = dot(u, v), den = 1.f - uv * uv, uw = dot(u, w), vw = dot(v, w);
    float ta = (uv * vw - uw) / den, tb = (vw - uv * uw) / den;
    ta = fminf(a.size[i], fmaxf(-a.size[i], ta)); tb = fminf(b.size[j], fmaxf(-b.size[j], tb));
    o.dist = esep; o.pos = (pa + u * ta + pb + v * tb) * 0.5f; o.n = L;
    return true;
  }
  // face contact: A = the box owning the axis (reference), B = the other (incident)
  const bool ref1 = fax < 3;
  const int ri = ref1 ? fax : fax - 3;
  const GeomW& A = ref1 ? a : b;
  const GeomW& B = ref1 ? b : a;
  f3 nA = colv(A.mat, ri);
  if (dot(nA, B.pos - A.pos) < 0.f) nA = nA * -1.f;
  const f3 nb = mulTv(B.mat, nA);   // nA in B's axes
  int bj = 0;
  if (fabsf(nb.y) > fabsf(nb.x)) bj = 1;
  if (fabsf(nb.z) > fabsf(comp(nb, bj))) bj = 2;
  const f3 mB = colv(B.mat, bj) * (comp(nb, bj) > 0.f ? -1.f : 1.f);
  const int bu = bj == 2 ? 0 : bj + 1, bw = bu == 2 ? 0 : bu + 1, au = ri == 2 ? 0 : ri + 1, aw = au == 2 ? 0 : au + 1;
  const f3 Bu = colv(B.mat, bu) * B.size[bu], Bw = colv(B.mat, bw) * B.size[bw], Au = colv(A.mat, au), Aw = colv(A.mat, aw);
  const f3 fc = B.pos + mB * B.size[bj];            // centre of the incident face
  const float su = A.size[au], sw = A.size[aw];
  // corner q of a quad in the order (+,+), (-,+), (-,-), (+,-)
  auto s0 = [](int q) { return (q == 0 || q == 3) ? 1.f : -1.f; };
  auto s1 = [](int q) { return q < 2 ? 1.f : -1.f; };
  bool hit = false;
  f3 x = mk3(0, 0, 0);
  if (lane < 4) {
    x = fc + Bu * s0(lane) + Bw * s1(lane);
    const f3 rel = x - A.pos;
    hit = fabsf(dot(rel, Au)) <= su && fabsf(dot(rel, Aw)) <= sw;
  } else if (lane < 8) {
    const int q = lane - 4;
    const float U = s0(q) * su, W = s1(q) * sw;
    // strictly inside the projected incident quad: same side of all four edges
    int pos_ = 0, neg_ = 0;
#pragma unroll
    for (int e = 0; e < 4; e++) {
      const f3 p0 = fc + Bu * s0(e) + Bw * s1(e) - A.pos, p1 = fc + Bu * s0((e + 1) & 3) + Bw * s1((e + 1) & 3) - A.pos;
      const float u0 = dot(p0, Au), w0 = dot(p0, Aw), u1 = dot(p1, Au), w1 = dot(p1, Aw);
      const float cr = (u1 - u0) * (W - w0) - (w1 - w0) * (U - u0);
      pos_ += cr > 0.f; neg_ += cr < 0.f;
    }
    if (pos_ == 4 || neg_ == 4) {
      const f3 x0 = A.pos + nA * A.size[ri] + Au * U + Aw * W;
      const float t = dot(mB, fc - x0) / dot(mB, nA);   // |mB . nA| >= 1 / sqrt(3): the most anti-parallel face
      x = x0 + nA * t;
      hit = true;
    }
  } else if (lane < 24) {
    const int e = (lane - 8) >> 2, side = (lane - 8) & 3;
    const f3 p0 = fc + Bu * s0(e) + Bw * s1(e), p1 = fc + Bu * s0((e + 1) & 3) + Bw * s1((e + 1) & 3);
    const f3 ax_ = side < 2 ? Au : Aw, ot_ = side < 2 ? Aw : Au;
    const float sg = (side & 1) ? -1.f : 1.f, lim_ = side < 2 ? su : sw, olim = side < 2 ? sw : su;
    const float f0 = sg * dot(p0 - A.pos, ax_) - lim_, f1 = sg * dot(p1 - A.pos, ax_) - lim_;
    if ((f0 < 0.f && f1 > 0.f) || (f0 > 0.f && f1 < 0.f)) {
      x = p0 + (p1 - p0) * (f0 / (f0 - f1));
      hit = fabsf(dot(x - A.pos, ot_)) <= olim;
    }
  }
  if (hit) {
    const float dist = dot(x - A.pos, nA) - A.size[ri];
    if (dist > margin) hit = false;
    o.dist = dist; o.pos = x - nA * (0.5f * dist); o.n = ref1 ? nA : nA * -1.f;
  }
  return hit;
}

MJB_DEV void make_frame(f3 n, f3 t, float* fr) {
  float nn = sqrtf(dot(n, n));
  n = n * (1.0f / nn);
  if (dot(t, t) < 0.25f) {
    t = mk3(0, 0, 0);
    if (n.y < 0.5f && n.y > -0.5f) t.y = 1; else t.z = 1;
  }
  t = t - n * dot(n, t);
  t = t * (1.0f / sqrtf(dot(t, t)));
  st3(fr, n); st3(fr + 3, t); st3(fr + 6, cross(n, t));
}

// append one contact record; `idx` already bounds-checked
MJB_DEV void store_contact(const Ctx& c, int idx, const ConOut& o, int pair, float mu) {
  float* r = SF(con) + CON_STRIDE * idx;
  r[CON_DIST] = o.dist;
  st3(r + CON_POS, o.pos);
  make_frame(o.n, o.t, r + CON_FRAME);
  ((int*)r)[CON_PAIR] = pair;
  r[CON_MU] = mu;
}

// returns the number of contacts stored (warp-uniform); fills SF_con.  `tot[copy]` is ADVANCED by the number of
// contacts found for that copy of a packed env (pack == 1: tot[0]) before the per-copy quota of maxcon1 slots
template <bool PRM = false>
MJB_DEV int collide(const Ctx& c, int* tot) {
  const DM& dm = *c.dm;
  const uint32_t* pairs = CU(pair_pack);
  int* cand = SI(cand);
  int ncand = 0;
  // broad phase, level 1: which pair blocks (tree x tree, tree x static geom) can touch at all — a tree is bounded
  // by a sphere of radius `reach` about its root body's origin (dev_model_build.h)
  uint32_t act_lo = 0xffffffffu, act_hi = 0xffffffffu;
  MJB_NOUNROLL
  for (int b0 = 0; b0 < dm.nblock; b0 += 32) {
    const int bi = b0 + c.lane;
    bool on = false;
    if (bi < dm.nblock) {
      const int* rec = CI(bp_block) + BP_STRIDE * bi;
      const int partner = rec[BP_PARTNER];
      if (partner == BP_ALWAYS) on = true;
      else {
        const float reach = CF(bp_block)[BP_STRIDE * bi + BP_REACH] + CF(bp_block)[BP_STRIDE * bi + BP_MARGIN];
        const f3 ca = ld3(SF(xpos) + 3 * rec[BP_ROOT_A]);
        if (partner >= 0) {
          f3 d = ld3(SF(xpos) + 3 * partner) - ca;
          on = dot(d, d) <= reach * reach;
        } else {
          const int g = -1 - partner;   // static geom: world pose is in the image
          const f3 gp = ld3(CF(geom_pos) + 3 * g);
          const float* gm = CF(geom_mat) + 9 * g;
          const int type = CI(geom_type)[g];
          if (type == MJB_GEOM_PLANE) on = dot(ca - gp, colv(gm, 2)) <= reach;
          else if (type == MJB_GEOM_BOX) on = point_box_dist(mulTv(gm, ca - gp), CF(geom_size) + 3 * g) <= reach;
          else { f3 d = gp - ca; float rr = reach + CF(geom_rbound)[g]; on = dot(d, d) <= rr * rr; }
        }
      }
    }
    const uint32_t bal = MJB_BALLOT(on);
    if (b0 == 0) act_lo = bal; else act_hi = bal;
  }
  if (dm.nblock > 0 && dm.nblock <= 32) act_hi = 0;
  // level 2: bounding spheres of the geoms (planes: signed distance of the centre), 32 pairs per pass
  // (which passes hold a pair of a live block is itself decided lane-parallel: lane = pass, then only those are walked)
  const int npass = (dm.npair + 31) >> 5;
  MJB_NOUNROLL
  for (int pb = 0; pb < npass; pb += 32) {
  uint32_t live = 0;
  {
    const int ps = pb + c.lane;
    bool on = false;
    if (ps < npass) { const uint32_t* pm = CU(bp_passmask) + 2 * ps; on = ((pm[0] & act_lo) | (pm[1] & act_hi)) != 0u; }
    live = MJB_BALLOT(on);
  }
  MJB_NOUNROLL
  while (live) {
    const int base = (pb + MJB_FFS(live) - 1) << 5;
    live &= live - 1u;
    int p = base + c.lane;
    bool keep = false;
    if (p < dm.npair) {
      uint32_t pk = pairs[p];
      int g1 = pk & 0xfff, g2 = (pk >> 12) & 0xfff;
      float margin = CF(pclass)[PC_STRIDE * (pk >> 24) + PC_MARGIN];
      GeomW a = geom_world(c, g1), b = geom_world(c, g2);
      float rb2 = CF(geom_rbound)[g2];
      if (a.type == MJB_GEOM_PLANE) keep = dot(b.pos - a.pos, colv(a.mat, 2)) <= rb2 + margin;
      else if (b.type == MJB_GEOM_BOX) {
        // bounding sphere of geom1 against the oriented box itself: long thin boxes have useless spheres
        keep = point_box_dist(mulTv(b.mat, a.pos - b.pos), b.size) <= CF(geom_rbound)[g1] + margin;
      } else {
        float rr = CF(geom_rbound)[g1] + rb2 + margin;
        f3 d = b.pos - a.pos;
        keep = dot(d, d) <= rr * rr;
      }
    }
    uint32_t bal = MJB_BALLOT(keep);
    int idx = ncand + MJB_POPC(bal & ((1u << c.lane) - 1u));
    if (keep && idx < dm.maxcand) cand[idx] = p;
    ncand += MJB_POPC(bal);
  }
  }
  if (ncand > dm.maxcand) ncand = dm.maxcand;
  MJB_SYNC();
  // narrow phase, lane = candidate (types with at most two contacts)
  int ncon = 0;
  MJB_NOUNROLL
  for (int base = 0; base < ncand; base += 32) {
    int i = base + c.lane;
    int n = 0, p = -1;
    ConOut o[2];
    float mu = 0.f;
    if (i < ncand) {
      p = cand[i];
      uint32_t pk = pairs[p];
      int g1 = pk & 0xfff, g2 = (pk >> 12) & 0xfff;
      const float* pc = CF(pclass) + PC_STRIDE * (pk >> 24);
      float margin = pc[PC_MARGIN];
      mu = PRM ? fmaxf(c.s[dm.prm_soff + prm_friction(dm) + g1], c.s[dm.prm_soff + prm_friction(dm) + g2]) : pc[PC_MU];
      GeomW a = geom_world(c, g1), b = geom_world(c, g2);
      if (a.type == MJB_GEOM_PLANE) {
        f3 nrm = colv(a.mat, 2);
        if (b.type == MJB_GEOM_SPHERE) n = plane_sphere(a.pos, nrm, b.pos, b.size[0], margin, o[0]);
        else if (b.type == MJB_GEOM_CAPSULE) {
          f3 ax = colv(b.mat, 2);
          n = plane_sphere(a.pos, nrm, b.pos + ax * b.size[1], b.size[0], margin, o[0]);
          n += plane_sphere(a.pos, nrm, b.pos - ax * b.size[1], b.size[0], margin, o[n]);
          o[0].t = ax; o[1].t = ax;
        }
      } else if (a.type == MJB_GEOM_SPHERE) {
        if (b.type == MJB_GEOM_SPHERE) n = sphere_sphere(a.pos, a.size[0], b.pos, b.size[0], margin, o[0]);
        else if (b.type == MJB_GEOM_CAPSULE) {
          f3 ax = colv(b.mat, 2);
          float x = fminf(b.size[1], fmaxf(-b.size[1], dot(ax, a.pos - b.pos)));
          n = sphere_sphere(a.pos, a.size[0], b.pos + ax * x, b.size[0], margin, o[0]);
        } else if (b.type == MJB_GEOM_BOX) n = sphere_box(a.pos, a.size[0], b.pos, b.mat, b.size, margin, o[0]);
      } else if (a.type == MJB_GEOM_CAPSULE) {
        if (b.type == MJB_GEOM_CAPSULE) n = capsule_capsule(a, b, margin, o);
        else if (b.type == MJB_GEOM_BOX) n = capsule_box(a, b, margin, o);
      }
    }
    // append in candidate order; every copy of a packed env has its own quota of maxcon1 slots (a contact-heavy
    // copy must not starve its neighbours), `tot` counts what was found so that dropped contacts are visible
    const int copy = (dm.pack > 1 && p >= 0) ? (int)(pairs[p] & 0xfff) / dm.ngeom1 : 0;
    const uint32_t lt = (1u << c.lane) - 1u;
    for (int k = 0; k < 2; k++) {
      const bool has = n > k;
      bool acc = has;
#pragma unroll
      for (int cp = 0; cp < MJB_MAX_PACK; cp++) {
        if (cp < dm.pack) {   // warp-uniform
          const uint32_t bc = MJB_BALLOT(has && copy == cp);
          if (has && copy == cp && tot[cp] + MJB_POPC(bc & lt) >= dm.maxcon1) acc = false;
          tot[cp] += MJB_POPC(bc);
        }
      }
      const uint32_t bal = MJB_BALLOT(acc);
      if (acc) store_contact(c, ncon + MJB_POPC(bal & lt), o[k], p, mu);
      ncon += MJB_POPC(bal);
    }
  }
  // multi-contact types (plane-box, box-box): one candidate at a time, lane = box corner
  // (the candidates of these types are found lane-parallel first: usually there is none)
  MJB_NOUNROLL
  for (int cb = 0; cb < ncand; cb += 32) {
  uint32_t multi = 0;
  {
    const int i = cb + c.lane;
    bool is_multi = false;
    if (i < ncand) {
      const uint32_t pk = pairs[cand[i]];
      const int t1 = CI(geom_type)[pk & 0xfff], t2 = CI(geom_type)[(pk >> 12) & 0xfff];
      is_multi = t2 == MJB_GEOM_BOX && (t1 == MJB_GEOM_PLANE || t1 == MJB_GEOM_BOX);
    }
    multi = MJB_BALLOT(is_multi);
  }
  MJB_NOUNROLL
  while (multi) {
    const int i = cb + MJB_FFS(multi) - 1;
    multi &= multi - 1u;
    int p = cand[i];
    uint32_t pk = pairs[p];
    int g1 = pk & 0xfff, g2 = (pk >> 12) & 0xfff;
    int t1 = CI(geom_type)[g1];
    const float* pc = CF(pclass) + PC_STRIDE * (pk >> 24);
    float margin = pc[PC_MARGIN], mu = PRM ? fmaxf(c.s[dm.prm_soff + prm_friction(dm) + g1], c.s[dm.prm_soff + prm_friction(dm) + g2]) : pc[PC_MU];
    GeomW a = geom_world(c, g1), b = geom_world(c, g2);
    bool hit = false;
    ConOut o;
    o.t = mk3(0, 0, 0);
    int lim = 4;
    if (t1 == MJB_GEOM_PLANE) {
      if (c.lane < 8) {
        f3 nrm = colv(a.mat, 2);
        float dist0 = dot(b.pos - a.pos, nrm);
        f3 vec = mk3(b.size[0] * ((c.lane & 1) ? 1.f : -1.f), b.size[1] * ((c.lane & 2) ? 1.f : -1.f), b.size[2] * ((c.lane & 4) ? 1.f : -1.f));
        f3 corner = mulv(b.mat, vec);
        float ld = dot(nrm, corner);
        if (!(dist0 + ld > margin || ld > 0)) {
          hit = true; o.dist = dist0 + ld; o.pos = corner + b.pos - nrm * (0.5f * o.dist); o.n = nrm;
        }
      }
    } else {
      lim = 8;
      hit = box_box_lane(c.lane, a, b, margin, o);
    }
    uint32_t bal = MJB_BALLOT(hit);
    int rank = MJB_POPC(bal & ((1u << c.lane) - 1u));
    int add = MJB_POPC(bal);
    if (add > lim) add = lim;
    const int copy = dm.pack > 1 ? g1 / dm.ngeom1 : 0;
    int room = 0;
#pragma unroll
    for (int cp = 0; cp < MJB_MAX_PACK; cp++)
      if (cp == copy) { room = dm.maxcon1 - tot[cp]; tot[cp] += add; }
    if (room < 0) room = 0;
    if (add > room) add = room;
    if (hit && rank < add) store_contact(c, ncon + rank, o, p, mu);
    ncon += add;
  }
  }
  MJB_SYNC();
  return ncon;
}

// =================================================================================================
// constraints
// general-power sigmoid (rare: the default power is 2) kept out of line to keep the hot code small
MJB_DEV_NOINLINE float impedance_pow(float x, float mid, float power) {
  if (x <= mid) return powf(x, power) / powf(mid, power - 1.f);
  return 1.f - powf(1.f - x, power) / powf(1.f - mid, power - 1.f);
}
MJB_DEV float impedance(const float* solimp, float pos, float margin) {
  float dmin = solimp[0], dmax = solimp[1], width = solimp[2], mid = solimp[3], power = solimp[4];
  if (dmin == dmax || width <= MJB_MINVAL) return 0.5f * (dmin + dmax);
  float x = fabsf((pos - margin) / width);
  if (x >= 1.f) return dmax;
  if (x <= 0.f) return dmin;
  float y;
  if (power == 1.f) y = x;
  else if (power == 2.f) y = x <= mid ? x * x / mid : 1.f - (1.f - x) * (1.f - x) / (1.f - mid);
  else y = impedance_pow(x, mid, power);
  return dmin + y * (dmax - dmin);
}

// rows: [0, 2 nlim) limit slots (lower, upper per limited joint; inactive -> D = 0), then 4 per contact
template <bool PRM = false>
MJB_DEV void make_constraints(const Ctx& c, int ncon) {
  const DM& dm = *c.dm;
  float *efcD = SF(efcD), *efcAref = SF(efcAref), *qpos = SF(qpos), *qvel = SF(qvel);
  MJB_NOUNROLL
  for (int k = c.lane; k < dm.nlim; k += 32) {
    const float* lp = CF(lim_param) + LIM_STRIDE * k;
    float q = qpos[CI(lim_qposadr)[k]], v = qvel[CI(lim_dof)[k]];
#pragma unroll
    for (int side = 0; side < 2; side++) {
      float dist = side == 0 ? q - lp[LIM_LO] : lp[LIM_HI] - q;
      float D = 0.f, aref = 0.f;
      if (dist < lp[LIM_MARGIN]) {
        float imp = impedance(lp + LIM_SOLIMP, dist, lp[LIM_MARGIN]);
        float R = fmaxf(MJB_MINVAL, (1.f - imp) * lp[LIM_INVW] / imp);
        D = 1.f / R;
        float vel = side == 0 ? v : -v;
        aref = -lp[LIM_B] * vel - lp[LIM_K] * imp * (dist - lp[LIM_MARGIN]);
      }
      efcD[2 * k + side] = D; efcAref[2 * k + side] = aref;
    }
  }
  // contact Jacobians: lane = dof, rows (normal, tangent1, tangent2) per contact.  Only the dofs on the
  // chains of the two bodies are non-zero, so each row is stored PACKED along the set bits of the contact's
  // dof mask (mask = chain(b1) xor chain(b2): shared ancestors cancel), ldj = widest mask + padding.
  float *J = SF(J), *con = SF(con), *cdof = SF(cdof), *xpos = SF(xpos);
  const uint32_t* pairs = CU(pair_pack);
  MJB_NOUNROLL
  for (int k = c.lane; k < ncon; k += 32) {
    float* r = con + CON_STRIDE * k;
    uint32_t pk = pairs[((const int*)r)[CON_PAIR]];
    int b1 = CI(geom_mb)[pk & 0xfff], b2 = CI(geom_mb)[(pk >> 12) & 0xfff];
    uint32_t mask = (b1 >= 0 ? CU(mb_dofmask)[2 * b1] : 0u) ^ (b2 >= 0 ? CU(mb_dofmask)[2 * b2] : 0u);
    ((uint32_t*)r)[CON_MASK] = mask;
    // the dofs of the mask as packed bytes, ascending (four words built in registers, no indexed local array)
#pragma unroll
    for (int wi = 0; wi < 4; wi++) {
      uint32_t word = 0u;
#pragma unroll
      for (int bi = 0; bi < 4; bi++) {
        if (mask) { word |= (uint32_t)(MJB_FFS(mask) - 1) << (8 * bi); mask &= mask - 1; }
      }
      ((uint32_t*)r)[CON_DOFS + wi] = word;
    }
  }
  MJB_SYNC();
  MJB_NOUNROLL
  for (int d = c.lane; d < dm.nv; d += 32) {
    f3 sw = ld3(cdof + 6 * d), sv = ld3(cdof + 6 * d + 3);
    int root = CI(mb_root)[CI(dof_mb)[d]];
    f3 o = ld3(xpos + 3 * root);
    uint32_t bit = 1u << d;
    MJB_NOUNROLL
    for (int k = 0; k < ncon; k++) {
      const float* r = con + CON_STRIDE * k;
      uint32_t mask = ((const uint32_t*)r)[CON_MASK];
      if (!(mask & bit)) continue;
      uint32_t pk = pairs[((const int*)r)[CON_PAIR]];
      int b2 = CI(geom_mb)[(pk >> 12) & 0xfff];
      // the dof is on exactly one of the two chains: + for geom2's body, - for geom1's
      float sgn = (b2 >= 0 && (CU(mb_dofmask)[2 * b2] & bit)) ? 1.f : -1.f;
      f3 vel = (sv + cross(sw, ld3(r + CON_POS) - o)) * sgn;
      int idx = MJB_POPC(mask & (bit - 1u));
      J[(3 * k) * dm.ldj + idx] = dot(ld3(r + CON_FRAME), vel);
      J[(3 * k + 1) * dm.ldj + idx] = dot(ld3(r + CON_FRAME + 3), vel);
      J[(3 * k + 2) * dm.ldj + idx] = dot(ld3(r + CON_FRAME + 6), vel);
    }
  }
  MJB_SYNC();
  // per-contact regulariser and reference acceleration: lane = contact
  int base = 2 * dm.nlim;
  MJB_NOUNROLL
  for (int k = c.lane; k < ncon; k += 32) {
    const float* r = con + CON_STRIDE * k;
    uint32_t pk = pairs[((const int*)r)[CON_PAIR]];
    const float* pc = CF(pclass) + PC_STRIDE * (pk >> 24);
    int b1 = CI(geom_mb)[pk & 0xfff], b2 = CI(geom_mb)[(pk >> 12) & 0xfff];
    float tran = (b1 >= 0 ? CF(mb_invweight)[b1] : 0.f) + (b2 >= 0 ? CF(mb_invweight)[b2] : 0.f);
    float mu = PRM ? r[CON_MU] : pc[PC_MU], dist = r[CON_DIST], inc = pc[PC_INCMARGIN];
    float imp = impedance(pc + PC_SOLIMP, dist, inc);
    float vn = 0.f, v1 = 0.f, v2 = 0.f;
    {
      uint32_t mm = ((const uint32_t*)r)[CON_MASK];
      int m = 0;
      MJB_NOUNROLL
      while (mm) {
        float qd = qvel[MJB_FFS(mm) - 1];
        mm &= mm - 1;
        vn += J[(3 * k) * dm.ldj + m] * qd; v1 += J[(3 * k + 1) * dm.ldj + m] * qd; v2 += J[(3 * k + 2) * dm.ldj + m] * qd;
        m++;
      }
    }
    float kpos = pc[PC_K] * imp * (dist - inc), B = pc[PC_B];
    if (pc[PC_CONDIM] < 2.f) {
      float R = fmaxf(MJB_MINVAL, (1.f - imp) * tran / imp);
      efcD[base + 4 * k] = 1.f / R; efcAref[base + 4 * k] = -B * vn - kpos;
      for (int e = 1; e < 4; e++) { efcD[base + 4 * k + e] = 0.f; efcAref[base + 4 * k + e] = 0.f; }
    } else {
      float R0 = fmaxf(MJB_MINVAL, (1.f - imp) * tran * (1.f + mu * mu) / imp);
      float D = 1.f / (2.f * mu * mu * R0);
      efcD[base + 4 * k] = D; efcAref[base + 4 * k] = -B * (vn + mu * v1) - kpos;
      efcD[base + 4 * k + 1] = D; efcAref[base + 4 * k + 1] = -B * (vn - mu * v1) - kpos;
      efcD[base + 4 * k + 2] = D; efcAref[base + 4 * k + 2] = -B * (vn + mu * v2) - kpos;
      efcD[base + 4 * k + 3] = D; efcAref[base + 4 * k + 3] = -B * (vn - mu * v2) - kpos;
    }
  }
  MJB_SYNC();
}

// =================================================================================================
// dense helpers (nv <= 32: lane = row / dof).  M is block diagonal over kinematic trees and so is the
// Hessian unless a contact couples two trees, so everything works per block [t0, t1) of the lane and the
// blocks of different trees proceed in parallel on their own lanes.
// out = sum_j A(row, j) x[j] over the row's block, A symmetric packed
MJB_DEV float matvec_row(const float* A, const float* x, int row, int t0, int t1) {
  float s0 = 0.f, s1 = 0.f;
  int j = t0;
  MJB_NOUNROLL
  for (; j + 1 <= row && j + 1 < t1; j += 2) { s0 += A[tri(row, j)] * x[j]; s1 += A[tri(row, j + 1)] * x[j + 1]; }
  MJB_NOUNROLL
  for (; j <= row && j < t1; j++) s0 += A[tri(row, j)] * x[j];
  MJB_NOUNROLL
  for (; j < t1; j++) s1 += A[tri(j, row)] * x[j];
  return s0 + s1;
}
// in-place Cholesky of the packed lower triangle, block by block; lane i owns row i.  `nb` = the largest
// block size (warp-uniform).  Returns 1 / L_ii of the lane's row.
MJB_DEV float cholesky(float* A, int lane, int t0, int t1, int nb) {
  float invd = 1.f;
  const bool own = lane < t1;  // lanes >= nv have t0 = t1 = 0
  MJB_NOUNROLL
  for (int jj = 0; jj < nb; jj++) {
    const int j = t0 + jj;
    const bool col = own && j < t1;
    float s0 = 0.f, s1 = 0.f;
    if (col && lane >= j) {
      s0 = A[tri(lane, j)];
      const float* ri = A + tri(lane, 0);
      const float* rj = A + tri(j, 0);
      int k = t0;
      MJB_NOUNROLL
      for (; k + 1 < j; k += 2) { s0 -= ri[k] * rj[k]; s1 -= ri[k + 1] * rj[k + 1]; }
      if (k < j) s0 -= ri[k] * rj[k];
    }
    float s = s0 + s1;
    float sj = MJB_SHFL(s, col ? j : lane);
    float inv = MJB_RSQRT(fmaxf(sj, 1e-20f));
    if (col) {
      if (lane == j) { invd = inv; A[tri(lane, j)] = sj * inv; }
      else if (lane > j) A[tri(lane, j)] = s * inv;
    }
    MJB_SYNC();
  }
  return invd;
}
// solve L L' x = b with lane-resident b / x
MJB_DEV float chol_solve(const float* A, int lane, int t0, int t1, int nb, float invd, float b) {
  float x = b;
  const bool own = lane < t1;
  MJB_NOUNROLL
  for (int kk = 0; kk < nb; kk++) {
    const int k = t0 + kk;
    const bool col = own && k < t1;
    float yk = MJB_SHFL(x * invd, col ? k : lane);
    if (col) {
      if (lane == k) x = yk;
      else if (lane > k) x -= A[tri(lane, k)] * yk;
    }
  }
  MJB_NOUNROLL
  for (int kk = nb - 1; kk >= 0; kk--) {
    const int k = t0 + kk;
    const bool col = own && k < t1;
    float xk = MJB_SHFL(x * invd, col ? k : lane);
    if (col) {
      if (lane == k) x = xk;
      else if (lane < k && lane >= t0) x -= A[tri(k, lane)] * xk;
    }
  }
  return x;
}

// Register-resident variant for blocks of at most NBT rows (every level of the reference: 14 dofs per ant,
// 6 for a free body): lane i keeps row i of its block in registers, row j is broadcast with shuffles, no
// shared-memory traffic and no barriers inside the factorisation.  Solves (A + diag) x = b for the lane's
// block where A is a packed lower triangle in shared memory.  Lanes of a block smaller than NBT (and idle
// lanes) run the same instruction stream on garbage that is never stored: columns past the block's size only
// ever touch the unused upper triangle.
//
// The factorisation is L D L' (unit lower L, no square roots), arranged for LATENCY, which is what this kernel
// runs out of: lane i keeps t_ik = L_ik d_k (raw) and l_ik = L_ik.  Column j needs s_ij = a_ij - sum_k l_ik t_jk;
// the raw t_jk of row j and the pivot d_j travel in two independent shuffles, so the dependent chain per column
// is shuffle -> rcp -> mul -> fma (~55 cycles) instead of shuffle -> rsqrt -> mul -> shuffle -> fma (~90) of the
// L L' form, and neither triangular solve divides.  The unit-lower L is written to `Lout` (packed) for the
// transposed solve.
#define MJB_NB 16
template <int NBT>
MJB_DEV_NOINLINE float factor_solve_regT(const float* A, float* Lout, int lane, int t0, int t1, float diag_add, float b) {
  float t[NBT], l[NBT];
  const bool own = lane < t1;
  const int li = lane - t0;
  const int rowoff = own ? tri(lane, t0) : 0;
#pragma unroll
  for (int k = 0; k < NBT; k++) {
    float v = (own && k <= li) ? A[rowoff + k] : 0.f;
    t[k] = (k == li) ? v + diag_add : v;
  }
  float rdi = 1.f;   // 1 / d_i of the lane's own row
#pragma unroll
  for (int j = 0; j < NBT; j++) {
    const int src = t0 + j;
    float s0 = t[j], s1 = 0.f;   // two partial sums: halves the fma chain of the late columns
#pragma unroll
    for (int k = 0; k < j; k++) {
      const float tjk = MJB_SHFL(t[k], src);
      if (k & 1) s1 -= l[k] * tjk; else s0 -= l[k] * tjk;
    }
    const float s = s0 + s1;
    t[j] = s;                                             // d_j on lane src, raw t_ij below it
    const float rd = 1.f / fmaxf(MJB_SHFL(s, src), 1e-20f);
    l[j] = s * rd;                                        // L_ij (1 on the diagonal)
    if (li == j) rdi = rd;
  }
#pragma unroll
  for (int k = 0; k < NBT; k++)
    if (own && k < li) Lout[rowoff + k] = l[k];
  // L y = b
  float x = b;
#pragma unroll
  for (int k = 0; k < NBT; k++) {
    const float yk = MJB_SHFL(x, t0 + k);
    x = li > k ? x - l[k] * yk : x;
  }
  x *= rdi;   // D z = y
  MJB_SYNC();
  // L' x = z: column k of L' is row k of L, contiguous across lanes in the packed store
  // (&L(k, lane) walks down by k words per step; lanes outside the block, or at / past column k, read a valid dummy
  // word and keep x: branch-free)
  const int nrow = t1 - t0, lq = own ? li : NBT;
  const float* lp = Lout + tri(t0 + NBT - 1, 0) + lane;
#pragma unroll
  for (int kk = NBT - 1; kk >= 1; kk--) {
    const int k = t0 + kk;
    const float xk = MJB_SHFL(x, k);
    const bool in = lq < kk && kk < nrow;
    const float lk = *(in ? lp : Lout);
    x = in ? x - lk * xk : x;
    lp -= k;
  }
  return x;
}
MJB_DEV float factor_solve_reg(const float* A, float* Lout, int lane, int t0, int t1, int nb, float diag_add, float b) {
  if (nb <= 6) return factor_solve_regT<6>(A, Lout, lane, t0, t1, diag_add, b);
  if (nb <= 14) return factor_solve_regT<14>(A, Lout, lane, t0, t1, diag_add, b);
  return factor_solve_regT<MJB_NB>(A, Lout, lane, t0, t1, diag_add, b);
}
// ONE block over all dofs (a contact couples the kinematic trees, or a single large tree), up to NBT <= 32 rows:
// register-resident Cholesky L L' with one array per lane (the L D L' form above needs two, 2 x 28 registers do not
// fit): lane i keeps row i, column j is finished with the row of lane j broadcast by shuffles.  No shared-memory
// traffic and no barrier inside the factorisation; L goes to `Lout` (packed) once, for the transposed solve.
template <int NBT>
MJB_DEV_NOINLINE float chol_solve_regT(const float* A, float* Lout, int lane, int n, float diag_add, float b) {
  float l[NBT];
  const bool own = lane < n;
  const int rowoff = own ? tri(lane, 0) : 0;
#pragma unroll
  for (int k = 0; k < NBT; k++) {
    float v = (own && k <= lane) ? A[rowoff + k] : 0.f;
    l[k] = (k == lane) ? v + diag_add : v;
  }
  float rinv = 1.f;   // 1 / L_ii of the lane's own row
#pragma unroll
  for (int j = 0; j < NBT; j++) {
    float s0 = l[j], s1 = 0.f;
#pragma unroll
    for (int k = 0; k < j; k++) {
      const float ljk = MJB_SHFL(l[k], j);
      if (k & 1) s1 -= l[k] * ljk; else s0 -= l[k] * ljk;
    }
    const float s = s0 + s1;
    const float inv = MJB_RSQRT(fmaxf(MJB_SHFL(s, j), 1e-20f));
    l[j] = s * inv;                       // L_ij for i >= j (lanes above the diagonal carry unused values)
    if (lane == j) rinv = inv;
  }
  MJB_SYNC();   // every lane has read its row of A before L overwrites it (A and Lout may be the same buffer)
#pragma unroll
  for (int k = 0; k < NBT; k++)
    if (own && k <= lane) Lout[rowoff + k] = l[k];
  // L y = b
  float x = b;
#pragma unroll
  for (int k = 0; k < NBT; k++) {
    const float yk = MJB_SHFL(x * rinv, k);
    x = lane > k ? x - l[k] * yk : x;
  }
  x *= rinv;
  MJB_SYNC();
  // L' z = y: column k of L' is row k of L, contiguous across lanes in the packed store
#pragma unroll
  for (int k = NBT - 1; k >= 1; k--) {
    const float zk = MJB_SHFL(x * rinv, k);
    const bool in = lane < k && k < n;
    const float lk = Lout[in ? tri(k, 0) + lane : 0];
    x = in ? x - lk * zk : x;
  }
  return x * rinv;
}

// (A + diag) x = b per block; picks the register path when the blocks are small enough
MJB_DEV float factor_solve(const float* A, float* L, int lane, int t0, int t1, int nb, float diag_add, float b, int nv) {
  if (MJB_LIKELY(nb <= MJB_NB)) return factor_solve_reg(A, L, lane, t0, t1, nb, diag_add, b);
  if (nb == nv) {   // a single block over all dofs
    if (nv <= 28) return chol_solve_regT<28>(A, L, lane, nv, diag_add, b);
    return chol_solve_regT<32>(A, L, lane, nv, diag_add, b);
  }
  if (A != L) {
    MJB_NOUNROLL
    for (int i = lane; i < (nv * (nv + 1)) / 2; i += 32) L[i] = A[i];
    MJB_SYNC();
  }
  if (lane < t1 && diag_add != 0.f) L[tri(lane, lane)] += diag_add;
  MJB_SYNC();
  float invd = cholesky(L, lane, t0, t1, nb);
  return chol_solve(L, lane, t0, t1, nb, invd, b);
}

// jar-like product for every row: out[row] = J_row . x   (limit rows: +-x[dof]; contact rows: pyramid edges)
MJB_DEV void rows_mul(const Ctx& c, int ncon, const float* x, float* out, const float* sub) {
  const DM& dm = *c.dm;
  MJB_NOUNROLL
  for (int k = c.lane; k < dm.nlim; k += 32) {
    float v = x[CI(lim_dof)[k]];
    out[2 * k] = v - (sub ? sub[2 * k] : 0.f);
    out[2 * k + 1] = -v - (sub ? sub[2 * k + 1] : 0.f);
  }
  const float* J = SF(J);
  const float* con = SF(con);
  const int base = 2 * dm.nlim;
  // contact rows: eight lanes per contact (four contacts per pass), each lane the dof slots l8, l8 + 8 of the contact's
  // chain list; three xor-shuffles sum the normal / tangent products over the group, lanes 0..3 of the group then write
  // the four pyramid edges n +- mu t1, n +- mu t2
  MJB_NOUNROLL
  for (int k0 = 0; k0 < ncon; k0 += 4) {
    const int k = k0 + (c.lane >> 3), l8 = c.lane & 7;
    float sn = 0.f, s1 = 0.f, s2 = 0.f;
    if (k < ncon) {
      const uint32_t* rec = (const uint32_t*)(con + CON_STRIDE * k);
      const int nb = MJB_POPC(rec[CON_MASK]);
      const float *Jn = J + (3 * k) * dm.ldj, *J1 = Jn + dm.ldj, *J2 = J1 + dm.ldj;
      MJB_NOUNROLL
      for (int m = l8; m < nb; m += 8) {
        const float xv = x[(rec[CON_DOFS + (m >> 2)] >> (8 * (m & 3))) & 0xff];
        sn += Jn[m] * xv; s1 += J1[m] * xv; s2 += J2[m] * xv;
      }
    }
#pragma unroll
    for (int o = 4; o > 0; o >>= 1) { sn += MJB_SHFL_XOR(sn, o); s1 += MJB_SHFL_XOR(s1, o); s2 += MJB_SHFL_XOR(s2, o); }
    if (k < ncon && l8 < 4) {
      const float mu = con[CON_STRIDE * k + CON_MU];
      const float v = sn + ((l8 & 1) ? -mu : mu) * (l8 < 2 ? s1 : s2);
      out[base + 4 * k + l8] = v - (sub ? sub[base + 4 * k + l8] : 0.f);
    }
  }
  MJB_SYNC();
}

// J' w for a per-row weight vector w (limit rows +-e_dof, contact rows = pyramid edges): the lane's dof component
MJB_DEV float jt_mul(const Ctx& c, int ncon, int base, int mylim, const float* w) {
  const DM& dm = *c.dm;
  const float* J = SF(J);
  const float* con = SF(con);
  float out = mylim >= 0 ? w[2 * mylim] - w[2 * mylim + 1] : 0.f;
  MJB_NOUNROLL
  for (int k = 0; k < ncon; k++) {
    const uint32_t mask = ((const uint32_t*)(con + CON_STRIDE * k))[CON_MASK];
    if (!((mask >> c.lane) & 1u)) continue;
    const float mu = con[CON_STRIDE * k + CON_MU];
    const float w0 = w[base + 4 * k], w1 = w[base + 4 * k + 1], w2 = w[base + 4 * k + 2], w3 = w[base + 4 * k + 3];
    const int idx = MJB_POPC(mask & ((1u << c.lane) - 1u));
    out += J[(3 * k) * dm.ldj + idx] * ((w0 + w1) + (w2 + w3)) + J[(3 * k + 1) * dm.ldj + idx] * (mu * (w0 - w1)) +
           J[(3 * k + 2) * dm.ldj + idx] * (mu * (w2 - w3));
  }
  return out;
}
// the same for two weight vectors at once (one pass over the Jacobian)
MJB_DEV void jt_mul2(const Ctx& c, int ncon, int base, int mylim, const float* w, const float* v, float& ow, float& ov) {
  const DM& dm = *c.dm;
  const float* J = SF(J);
  const float* con = SF(con);
  ow = mylim >= 0 ? w[2 * mylim] - w[2 * mylim + 1] : 0.f;
  ov = mylim >= 0 ? v[2 * mylim] - v[2 * mylim + 1] : 0.f;
  MJB_NOUNROLL
  for (int k = 0; k < ncon; k++) {
    const uint32_t mask = ((const uint32_t*)(con + CON_STRIDE * k))[CON_MASK];
    if (!((mask >> c.lane) & 1u)) continue;
    const float mu = con[CON_STRIDE * k + CON_MU];
    const float w0 = w[base + 4 * k], w1 = w[base + 4 * k + 1], w2 = w[base + 4 * k + 2], w3 = w[base + 4 * k + 3];
    const float v0 = v[base + 4 * k], v1 = v[base + 4 * k + 1], v2 = v[base + 4 * k + 2], v3 = v[base + 4 * k + 3];
    const int idx = MJB_POPC(mask & ((1u << c.lane) - 1u));
    const float jn = J[(3 * k) * dm.ldj + idx], j1 = J[(3 * k + 1) * dm.ldj + idx], j2 = J[(3 * k + 2) * dm.ldj + idx];
    ow += jn * ((w0 + w1) + (w2 + w3)) + j1 * (mu * (w0 - w1)) + j2 * (mu * (w2 - w3));
    ov += jn * ((v0 + v1) + (v2 + v3)) + j1 * (mu * (v0 - v1)) + j2 * (mu * (v2 - v3));
  }
}

// primal Newton solve for qacc.  The cost is s(a) = 1/2 (a - a0)' M (a - a0) + 1/2 sum_r D_r min(x_r, 0)^2 with
// x = J a - aref (a0 = M^-1 qfrc_smooth), its gradient g = M a - qfrc_smooth - J' f, f_r = -D_r min(x_r, 0).
// M a is never formed: the iteration starts at a0 (g = -J' f), and after a step a+ = a + alpha s along the Newton
// direction of the current active set (H s = -g, H = M + J' W J) the gradient follows from the rows that SWITCHED
// between active and inactive alone:      g+ = (1 - alpha) g - J' u,   u_r = D_r |x_r+| on switched rows, else 0
// (every other row's change of force is cancelled exactly by the W J s term of M s = -g - J' W J s).  A step in which
// no row switches and alpha = 1 therefore ends with g = 0: the solve terminates on the exact active set.
// On exit SF_qacc = solution, SF_vecA = qfrc_smooth + J' f (= M a - g: the total force the implicit-damping solve
// needs), SF_vecB = g, SF_efcJar = J a - aref.  Returns iterations used.
MJB_DEV int newton(const Ctx& c, int ncon) {
  const DM& dm = *c.dm;
  const int nv = dm.nv, lane = c.lane;
  const int t0 = CI(dof_t0)[lane], t1 = CI(dof_t1)[lane];
  float *M = SF(M), *H = SF(H), *a = SF(qacc), *sv = SF(vecC);
  float *D = SF(efcD), *frc = SF(efcAref), *jar = SF(efcJar), *jv = SF(efcJv);   // frc overwrites aref once jar is formed
  const float* J = SF(J);
  const float* con = SF(con);
  const uint32_t* pairs = CU(pair_pack);
  const int base = 2 * dm.nlim, nrow = base + 4 * ncon;
  float *qfrc = SF(qfrc), *tot = SF(vecA);   // tot = qfrc_smooth + J' f of the current iterate
  // start from the unconstrained acceleration a0 = M^-1 qfrc_smooth (fewer Newton iterations than the previous step's
  // qacc under fast-changing controls, and exact when no constraint row is active)
  {
    float x = factor_solve(M, H, lane, t0, t1, dm.maxtree, 0.f, lane < nv ? qfrc[lane] : 0.f, nv);
    if (lane < nv) a[lane] = x;
    MJB_SYNC();
  }
  rows_mul(c, ncon, a, jar, frc);
  MJB_NOUNROLL
  for (int r = lane; r < nrow; r += 32) { const float x = jar[r]; frc[r] = x < 0.f ? -D[r] * x : 0.f; }
  MJB_SYNC();
  float g = 0.f;
  if (lane < nv) {
    const float q = jt_mul(c, ncon, base, CI(dof_lim)[lane], frc);   // J' f
    g = -q;
    tot[lane] = qfrc[lane] + q;
  }
  MJB_PH(c, PH_NEWTON_INIT);
  int it = 0;
  float last_step = 0.f;   // |alpha s| of the previous iteration (lane = dof)
  MJB_NOUNROLL
  for (;;) {
    const float qf = lane < nv ? qfrc[lane] : 0.f, ma = lane < nv ? tot[lane] + g : 0.f;   // M a = qfrc_smooth + J' f + g
    // (four independent reductions in one stage: gradient and force norms, and the size of the previous step against
    // the iterate for the stall test)
    const float gn = wsum(g * g), fn = wsum(qf * qf + ma * ma);
    const float amax = wmax(lane < nv ? fabsf(a[lane]) : 0.f), smax = wmax(last_step);
    const bool stalled = it > 0 && smax <= 1e-7f * (1.f + amax);
    const bool done = gn <= dm.solver_tol * dm.solver_tol * (fn + 1e-12f) || it >= dm.solver_iterations || stalled;
    MJB_PH(c, PH_NEWTON_GRAD);
    if (done) break;
    it++;
    // Hessian H = M + J' diag(D active) J (packed lower triangle)
    {
      // both triangles start 16 B aligned and are padded to a multiple of 4 words: copy as 128-bit words
      struct alignas(16) W4 { float a, b, c, d; };
      const W4* src = (const W4*)M;
      W4* dst = (W4*)H;
      MJB_NOUNROLL
      for (int i = lane; i < ((nv * (nv + 1)) / 2 + 3) / 4; i += 32) dst[i] = src[i];
    }
    MJB_SYNC();
    // active limit rows only touch the diagonal: handed to the factorisation as the lane's diagonal term
    float hdiag = 0.f;
    {
      const int mylim = CI(dof_lim)[lane];
      if (mylim >= 0) hdiag = (jar[2 * mylim] < 0 ? D[2 * mylim] : 0.f) + (jar[2 * mylim + 1] < 0 ? D[2 * mylim + 1] : 0.f);
    }
    bool coupled = false;  // does an active contact couple two kinematic trees?
    MJB_NOUNROLL
    for (int k = 0; k < ncon; k++) {
      uint32_t pk = pairs[((const int*)(con + CON_STRIDE * k))[CON_PAIR]];
      int b1 = CI(geom_mb)[pk & 0xfff], b2 = CI(geom_mb)[(pk >> 12) & 0xfff];
      uint32_t mask = ((const uint32_t*)(con + CON_STRIDE * k))[CON_MASK];
      float mu = con[CON_STRIDE * k + CON_MU];
      float w0 = jar[base + 4 * k] < 0 ? D[base + 4 * k] : 0.f, w1 = jar[base + 4 * k + 1] < 0 ? D[base + 4 * k + 1] : 0.f;
      float w2 = jar[base + 4 * k + 2] < 0 ? D[base + 4 * k + 2] : 0.f, w3 = jar[base + 4 * k + 3] < 0 ? D[base + 4 * k + 3] : 0.f;
      float cnn = w0 + w1 + w2 + w3;
      if (cnn == 0.f) continue;  // warp-uniform
      if (b1 >= 0 && b2 >= 0 && CI(mb_root)[b1] != CI(mb_root)[b2]) coupled = true;
      float cn1 = mu * (w0 - w1), c11 = mu * mu * (w0 + w1), cn2 = mu * (w2 - w3), c22 = mu * mu * (w2 + w3);
      // lanes = (row, column) pairs of the contact's dofs: H(di, dj) += sum_edges w_e J_e[di] J_e[dj]
      const int nb = MJB_POPC(mask), npairs = (nb * (nb + 1)) >> 1;
      const uint32_t* dofs = (const uint32_t*)(con + CON_STRIDE * k) + CON_DOFS;
      const float *Jn = J + (3 * k) * dm.ldj, *J1 = Jn + dm.ldj, *J2 = J1 + dm.ldj;
      MJB_NOUNROLL
      for (int p = lane; p < npairs; p += 32) {
        uint32_t rc = CU(tri_lut)[p];
        int mi = rc & 0xff, mj = rc >> 8;
        int di = (dofs[mi >> 2] >> (8 * (mi & 3))) & 0xff, dj = (dofs[mj >> 2] >> (8 * (mj & 3))) & 0xff;
        float ni = Jn[mi], ai = J1[mi], bi = J2[mi], nj = Jn[mj], aj = J1[mj], bj = J2[mj];
        H[tri(di, dj)] += ni * (cnn * nj + cn1 * aj + cn2 * bj) + ai * (cn1 * nj + c11 * aj) + bi * (cn2 * nj + c22 * bj);
      }
      MJB_SYNC();  // the next contact may touch the same entries from other lanes
    }
    MJB_SYNC();
    // factor per tree block unless a contact couples trees (then one block over all dofs)
    const int h0 = coupled ? 0 : t0, h1 = coupled ? (lane < nv ? nv : 0) : t1, hb = coupled ? nv : dm.maxtree;
    MJB_PH(c, PH_NEWTON_HESS);
    float s = factor_solve(H, H, lane, h0, h1, hb, hdiag, -g, nv);
    if (lane < nv) sv[lane] = s; else s = 0.f;
    MJB_SYNC();
    MJB_PH(c, PH_NEWTON_FACTOR);
    rows_mul(c, ncon, sv, jv, nullptr);
    MJB_PH(c, PH_LS_ROWSMUL);
    // slope and curvature of the smooth part along s without M:  s'(M a - qfrc) = g's + f'Js,  s'M s = -g's - (Js)'W(Js)
    float a1 = 0.f, a2 = 0.f;
    MJB_NOUNROLL
    for (int r = lane; r < nrow; r += 32) {
      const float v = jv[r];
      a1 += frc[r] * v;
      if (jar[r] < 0.f) a2 += D[r] * v * v;
    }
    const float d1_0 = wsum(g * s);   // phi'(0)
    const float p1 = d1_0 + wsum(a1), p2 = -d1_0 - wsum(a2);
    MJB_PH(c, PH_LS_MV);
    // exact line search on the convex piecewise-quadratic phi(alpha): safeguarded Newton on phi'.  s is the exact Newton
    // direction of the current active set, so the first trial is alpha = 1 (the minimiser whenever no row switches
    // along the step: then one evaluation ends the search)
    float alpha = 1.f, lo = 0.f, hi = MJB_BIG;
    MJB_NOUNROLL
    for (int ls = 1; ls <= dm.ls_iterations; ls++) {
      float d1 = 0.f, d2 = 0.f;
      MJB_NOUNROLL
      for (int r = lane; r < nrow; r += 32) {
        float x = jar[r] + alpha * jv[r];
        if (x < 0.f) { d1 += D[r] * x * jv[r]; d2 += D[r] * jv[r] * jv[r]; }
      }
      d1 = wsum(d1) + p1 + alpha * p2;
      d2 = wsum(d2) + p2;
      MJB_COUNT(c, 24, 1);   // line-search evaluations
      if (fabsf(d1) <= 1e-6f * fabsf(d1_0)) break;
      if (d1 < 0.f) lo = alpha; else hi = alpha;
      if (ls == dm.ls_iterations) break;
      float nxt = alpha - d1 / fmaxf(d2, MJB_MINVAL);
      if (!(nxt > lo && nxt < hi)) nxt = hi < MJB_BIG ? 0.5f * (lo + hi) : 2.f * alpha;
      alpha = nxt;
    }
    MJB_COUNT(c, 25, 1);     // Newton iterations
    MJB_PH(c, PH_LS_LOOP);
    last_step = fabsf(alpha * s);
    if (lane < nv) a[lane] += alpha * s;
    // rows: new residual, new force, and the switched rows' term of the gradient update (kept in jv)
    MJB_NOUNROLL
    for (int r = lane; r < nrow; r += 32) {
      const float xo = jar[r], xn = xo + alpha * jv[r], d = D[r];
      jar[r] = xn;
      frc[r] = xn < 0.f ? -d * xn : 0.f;
      jv[r] = ((xo < 0.f) != (xn < 0.f)) ? d * fabsf(xn) : 0.f;
#if defined(MJB_PHASE_PROF) && !defined(MJB_HOST_EMU)
      if (((xo < 0.f) != (xn < 0.f)) && d > 0.f) atomicAdd(&g_phase_cycles[25 + (it < 5 ? it : 5)], 1ull);   // switched rows by iteration (slots 26..30)
#endif
    }
#if defined(MJB_PHASE_PROF) && !defined(MJB_HOST_EMU)
    if (lane == 0 && alpha == 1.f) atomicAdd(&g_phase_cycles[31], 1ull);   // steps that ended at alpha = 1
#endif
    MJB_SYNC();
    if (lane < nv) {
      float gu, q;
      jt_mul2(c, ncon, base, CI(dof_lim)[lane], jv, frc, gu, q);
      g = (1.f - alpha) * g - gu;
      tot[lane] = qfrc[lane] + q;
    }
    MJB_PH(c, PH_NEWTON_LS);
  }
  if (lane < nv) SF(vecB)[lane] = g;
  MJB_SYNC();
  return it;
}

// =================================================================================================
// ray casting
MJB_DEV int quad_roots(float a, float b, float cc, float* x) {
  if (a < MJB_MINVAL) return 0;
  float det = b * b - a * cc;
  if (det < 0) return 0;
  float sq = sqrtf(det);
  x[0] = (-b - sq) / a; x[1] = (-b + sq) / a;
  return 2;
}
MJB_DEV float ray_geom(f3 pos, const float* R, const float* size, f3 pnt, f3 vec, int type) {
  if (type == MJB_GEOM_SPHERE) {
    f3 d = pnt - pos;
    float x[2];
    if (!quad_roots(dot(vec, vec), dot(vec, d), dot(d, d) - size[0] * size[0], x)) return -1.f;
    return x[0] >= 0 ? x[0] : (x[1] >= 0 ? x[1] : -1.f);
  }
  f3 lp = mulTv(R, pnt - pos), lv = mulTv(R, vec);
  if (type == MJB_GEOM_PLANE) {
    if (lv.z > -MJB_MINVAL) return -1.f;
    float x = -lp.z / lv.z;
    if (x < 0) return -1.f;
    float p0 = lp.x + x * lv.x, p1 = lp.y + x * lv.y;
    if ((size[0] <= 0 || fabsf(p0) <= size[0]) && (size[1] <= 0 || fabsf(p1) <= size[1])) return x;
    return -1.f;
  }
  float best = -1.f;
  if (type == MJB_GEOM_CAPSULE) {
    float r = size[0], h = size[1], x[2];
    if (quad_roots(lv.x * lv.x + lv.y * lv.y, lp.x * lv.x + lp.y * lv.y, lp.x * lp.x + lp.y * lp.y - r * r, x))
      for (int i = 0; i < 2; i++)
        if (fabsf(lp.z + x[i] * lv.z) <= h && x[i] >= 0 && (best < 0 || x[i] < best)) best = x[i];
    for (int sg = -1; sg <= 1; sg += 2) {
      f3 d = lp - mk3(0, 0, sg * h);
      if (quad_roots(dot(lv, lv), dot(lv, d), dot(d, d) - r * r, x))
        for (int i = 0; i < 2; i++)
          if (sg * (lp.z + x[i] * lv.z) >= h && x[i] >= 0 && (best < 0 || x[i] < best)) best = x[i];
    }
    return best;
  }
  // box, by slabs: the same first non-negative crossing as testing the six faces one by one (origin outside: entry point,
  // inside: exit point), a sixth of the branches
  float tn = -MJB_BIG, tf = MJB_BIG;
#pragma unroll
  for (int a = 0; a < 3; a++) {
    const float p = comp(lp, a), v = comp(lv, a), sz = size[a];
    if (fabsf(v) < MJB_MINVAL) {
      if (fabsf(p) > sz) return -1.f;
    } else {
      const float inv = 1.f / v, t1 = (-sz - p) * inv, t2 = (sz - p) * inv;
      tn = fmaxf(tn, fminf(t1, t2));
      tf = fminf(tf, fmaxf(t1, t2));
    }
  }
  if (tn > tf || tf < 0.f) return -1.f;
  return tn >= 0.f ? tn : tf;
}

MJB_DEV float cutoff(const Ctx& c, int i, float x) {
  float cut = CF(sensor_cutoff)[i];
  if (cut <= 0) return x;
  int dt = CI(sensor_dtype)[i];
  if (dt == 0) return fminf(cut, fmaxf(-cut, x));
  if (dt == 1) return fminf(cut, x);
  return x;
}

// position-stage sensors (rangefinder, frame axes)
MJB_DEV void sensors_pos(const Ctx& c) {
  const DM& dm = *c.dm;
  float* sens = SF(sens);
  MJB_NOUNROLL
  for (int i = 0; i < dm.nsensor; i++) {
    int type = CI(sensor_type)[i], t = CI(sensor_site)[i], adr = CI(sensor_adr)[i];
    if (type == MJB_SENS_RANGEFINDER) {
      f3 pnt = ld3(SF(spos) + 3 * t), vec = colv(SF(smat) + 9 * t, 2);
      int bex = CI(site_mb)[t];
      float best = MJB_BIG;
      MJB_NOUNROLL
      for (int g = c.lane; g < dm.ngeom; g += 32) {
        int gb = CI(geom_mb)[g];
        if ((gb >= 0 && gb == bex) || !CI(geom_ray)[g]) continue;
        GeomW gw = geom_world(c, g);
        if (gw.type != MJB_GEOM_PLANE) {
          // conservative bounding-sphere rejection (the ray direction is a unit vector)
          f3 mvec = gw.pos - pnt;
          float rb = CF(geom_rbound)[g], tca = dot(mvec, vec), mm = dot(mvec, mvec);
          if (mm - tca * tca > rb * rb || (tca < 0.f && mm > rb * rb)) continue;
        }
        float x = ray_geom(gw.pos, gw.mat, gw.size, pnt, vec, gw.type);
        if (x >= 0 && x < best) best = x;
      }
      best = wmin(best);
      if (c.lane == 0) sens[adr] = cutoff(c, i, best >= MJB_BIG ? -1.f : best);
    } else if (type >= MJB_SENS_FRAMEXAXIS && type <= MJB_SENS_FRAMEZAXIS) {
      if (c.lane < 3) sens[adr + c.lane] = cutoff(c, i, SF(smat)[9 * t + 3 * c.lane + (type - MJB_SENS_FRAMEXAXIS)]);
    }
  }
  MJB_SYNC();
}

// acceleration-stage sensors (touch, accelerometer); needs the solved qacc and efcJar
MJB_DEV void sensors_acc(const Ctx& c, int ncon) {
  const DM& dm = *c.dm;
  if (!dm.need_acc_sensors) return;
  float* sens = SF(sens);
  bool did_rne = false;
  const uint32_t* pairs = CU(pair_pack);
  const int base = 2 * dm.nlim;
  MJB_NOUNROLL
  for (int i = 0; i < dm.nsensor; i++) {
    int type = CI(sensor_type)[i], t = CI(sensor_site)[i], adr = CI(sensor_adr)[i];
    if (type == MJB_SENS_TOUCH) {
      int body = CI(site_mb)[t];
      float total = 0.f;
      MJB_NOUNROLL
      for (int k = c.lane; k < ncon; k += 32) {
        const float* r = SF(con) + CON_STRIDE * k;
        uint32_t pk = pairs[((const int*)r)[CON_PAIR]];
        int b1 = CI(geom_mb)[pk & 0xfff], b2 = CI(geom_mb)[(pk >> 12) & 0xfff];
        if (body < 0 || (b1 != body && b2 != body)) continue;
        float fn = 0.f;
        for (int e = 0; e < 4; e++) {
          float x = SF(efcJar)[base + 4 * k + e];
          if (x < 0) fn -= SF(efcD)[base + 4 * k + e] * x;
        }
        if (fn <= MJB_MINVAL) continue;
        f3 ray = ld3(r + CON_FRAME);
        if (b2 == body) ray = ray * -1.f;
        if (ray_geom(ld3(SF(spos) + 3 * t), SF(smat) + 9 * t, CF(site_size) + 3 * t, ld3(r + CON_POS), ray, CI(site_type)[t]) >= 0)
          total += fn;
      }
      total = wsum(total);
      if (c.lane == 0) sens[adr] = cutoff(c, i, total);
    } else if (type == MJB_SENS_ACCELEROMETER) {
      if (!did_rne) { rne_pass(c, true); did_rne = true; }
      int b = CI(site_mb)[t];
      if (c.lane == 0) {
        f3 acc = mk3(-dm.gravity[0], -dm.gravity[1], -dm.gravity[2]);
        if (b >= 0) {
          f3 w = ld3(SF(cvel) + 6 * b), v = ld3(SF(cvel) + 6 * b + 3), aw = ld3(SF(cacc) + 6 * b), av = ld3(SF(cacc) + 6 * b + 3);
          f3 r = ld3(SF(spos) + 3 * t) - ld3(SF(xpos) + 3 * CI(mb_root)[b]);
          acc = av + cross(aw, r) + cross(w, v + cross(w, r));
        }
        f3 loc = mulTv(SF(smat) + 9 * t, acc);
        sens[adr] = cutoff(c, i, loc.x); sens[adr + 1] = cutoff(c, i, loc.y); sens[adr + 2] = cutoff(c, i, loc.z);
      }
    }
  }
  MJB_SYNC();
}

// frame, velocity and joint sensors (DESIGN §5f), lane = sensor.  Runs between the bias pass and the collision pass:
// the only window where cvel and the body frames are both live (the broad phase's candidates overwrite cvel, the
// constraint rows overwrite xquat / xmat).  Velocities as the accelerometer's: cvel is about the tree root's origin.
MJB_DEV void sensors_frame(const Ctx& c) {
  const DM& dm = *c.dm;
  float* sens = SF(sens);
  const float *xpos = SF(xpos), *xquat = SF(xquat), *xmat = SF(xmat), *cvel = SF(cvel);
  MJB_NOUNROLL
  for (int i = c.lane; i < dm.nsensor; i += 32) {
    const int type = CI(sensor_type)[i], adr = CI(sensor_adr)[i];
    if (type == MJB_SENS_JOINTPOS || type == MJB_SENS_JOINTVEL) {
      const int a = CI(sensor_site)[i];
      sens[adr] = cutoff(c, i, type == MJB_SENS_JOINTPOS ? SF(qpos)[a] : SF(qvel)[a]);
      continue;
    }
    const bool axis = type >= KSENS_OBJ_AXIS;
    if (!axis && type != MJB_SENS_VELOCIMETER && type != MJB_SENS_GYRO && type != MJB_SENS_FRAMEPOS && type != MJB_SENS_FRAMEQUAT &&
        type != MJB_SENS_FRAMELINVEL && type != MJB_SENS_FRAMEANGVEL)
      continue;
    const float* rec = (const float*)(c.img + dm.off_sens_obj + SO_STRIDE * i);
    const int b = ((const int*)rec)[SO_MB];
    f3 p = ld3(rec + SO_POS), w = mk3(0, 0, 0), v = mk3(0, 0, 0);
    q4 q = ldq(rec + SO_QUAT);
    if (b >= 0) {
      p = ld3(xpos + 3 * b) + mulv(xmat + 9 * b, p);
      q = qmul(ldq(xquat + 4 * b), q);
      w = ld3(cvel + 6 * b);
      v = ld3(cvel + 6 * b + 3) + cross(w, p - ld3(xpos + 3 * CI(mb_root)[b]));
    }
    if (type == MJB_SENS_FRAMEQUAT) {   // never clamped
      q = qnorm(q);
      sens[adr] = q.w; sens[adr + 1] = q.x; sens[adr + 2] = q.y; sens[adr + 3] = q.z;
      continue;
    }
    f3 r = type == MJB_SENS_FRAMEPOS ? p : (type == MJB_SENS_FRAMEANGVEL ? w : v);
    if (axis) {   // column of the object's rotation
      const int a = type - KSENS_OBJ_AXIS;
      r = qrot(q, mk3(a == 0, a == 1, a == 2));
    } else if (type == MJB_SENS_GYRO || type == MJB_SENS_VELOCIMETER) {   // in the object's frame: R' x
      q4 qc = q;
      qc.x = -q.x; qc.y = -q.y; qc.z = -q.z;
      r = qrot(qc, type == MJB_SENS_GYRO ? w : v);
    }
    sens[adr] = cutoff(c, i, r.x); sens[adr + 1] = cutoff(c, i, r.y); sens[adr + 2] = cutoff(c, i, r.z);
  }
  MJB_SYNC();
}

// =================================================================================================
// one forward-dynamics evaluation: SF_qpos / qvel / ctrl -> SF_qacc.  Returns the contact count.
template <bool PRM = false>
MJB_DEV int forward(const Ctx& c, bool sensors, bool probes, int* iters_out, int* found) {
  MJB_PH(c, PH_INTEGRATE);
  kin_forward<PRM>(c);
  if (probes) {
    // exported positions belong to the LAST forward pass of the step (what `data.xipos` holds after
    // mj_step): for Euler that is the state before the integration (SURVEY 3.3), for RK4 the fourth stage.
    // Taken now because xipos is recycled by the solver scratch below
    const DM& dm = *c.dm;
    MJB_NOUNROLL
    for (int p = c.lane; p < dm.nprobe; p += 32) {
      int kind = CI(probe_kind)[p], id = CI(probe_id)[p];
      f3 v = kind == PROBE_BODY ? ld3(SF(xipos) + 3 * id) : (kind == PROBE_GEOM ? ld3(SF(gpos) + 3 * id) : ld3(CF(probe_const) + 3 * p));
      c.probe[4 * p] = v.x; c.probe[4 * p + 1] = v.y; c.probe[4 * p + 2] = v.z; c.probe[4 * p + 3] = 0.f;
      if (c.probe_quat && kind != PROBE_CONST) {
        // orientation of the body frame (data.body(n).xmat) / of the geom frame (data.geom(n).xmat), as a quaternion
        q4 q;
        if (kind == PROBE_BODY) q = ldq(SF(xquat) + 4 * id);
        else {
          int g = 0;   // geom id of the dynamic slot
          MJB_NOUNROLL
          for (int k = 0; k < dm.ngeom; k++) if (CI(geom_slot)[k] == id) g = k;
          q = qnorm(qmul(ldq(SF(xquat) + 4 * CI(geom_mb)[g]), ldq(CF(geom_quat) + 4 * g)));
        }
        c.probe_quat[4 * p] = q.w; c.probe_quat[4 * p + 1] = q.x; c.probe_quat[4 * p + 2] = q.y; c.probe_quat[4 * p + 3] = q.z;
      }
    }
    MJB_SYNC();
  }
  MJB_PH(c, PH_FK);
  dyn_backward<PRM>(c);
  MJB_PH(c, PH_RNE);
  if (sensors && c.dm->ext_sensors) sensors_frame(c);
  int tot[MJB_MAX_PACK] = {0, 0, 0, 0};
  int ncon = collide<PRM>(c, tot);
  MJB_PH(c, PH_COLLIDE);
  if (found) {   // contacts found beyond a copy's quota were dropped: keep the count visible (mjb_buffers.ncon_dropped)
#pragma unroll
    for (int cp = 0; cp < MJB_MAX_PACK; cp++) found[cp] += tot[cp] > c.dm->maxcon1 ? tot[cp] - c.dm->maxcon1 : 0;
  }
  if (sensors) sensors_pos(c);
  MJB_PH(c, PH_SENS);
  make_constraints<PRM>(c, ncon);
  MJB_PH(c, PH_CONSTR);
  int it = newton(c, ncon);
  // The Newton solve is where the envs of a round drift apart (1 .. 5 iterations).  Waiting for the slowest one HERE
  // instead of at the end of the round costs the same wait, and the rest of the step (sensors, integration, stores,
  // epilogue) then runs with the warps walking the code together: their instruction fetches hit lines a neighbour
  // has just brought in (the tail used to be the part with the most instruction-fetch stalls)
  MJB_CTA_SYNC(c.cta_threads);
  MJB_PH(c, PH_ALIGN);
  if (iters_out) *iters_out = it;
  if (sensors) sensors_acc(c, ncon);
  MJB_PH(c, PH_SENS);
  return ncon;
}

// qpos += h * qvel-like `v` (lane = joint)
MJB_DEV void integrate_pos(const Ctx& c, float* qpos, const float* v, float h) {
  const DM& dm = *c.dm;
  MJB_NOUNROLL
  for (int j = c.lane; j < dm.njnt; j += 32) {
    int qa = CI(jnt_qposadr)[j], da = CI(jnt_dofadr)[j];
    if (CI(jnt_type)[j] == MJB_JNT_FREE) {
      for (int i = 0; i < 3; i++) qpos[qa + i] += h * v[da + i];
      f3 w = ld3(v + da + 3);
      float nw = sqrtf(dot(w, w)), ang = nw * h;
      if (ang > 0.f) {
        q4 q = qnorm(qmul(ldq(qpos + qa + 3), axisangle(w * (1.0f / nw), ang)));
        qpos[qa + 3] = q.w; qpos[qa + 4] = q.x; qpos[qa + 5] = q.y; qpos[qa + 6] = q.z;
      }
    } else {
      qpos[qa] += h * v[da];
    }
  }
}

// One mj_forward (`integrate` = false) or one mj_step (forward + integration).  `sensors` selects sensor
// evaluation (only the final substep's sensors are observable).  The forward pass has ONE call site: Euler
// is a single stage, RK4 four stages of the same loop (stages 2..4 without sensors).  SF_qacc keeps the
// solver's qacc (not the damping-corrected one): it is the warm start of the next solve, as MuJoCo's
// qacc_warmstart.
// PRM: the env's physical parameters come from its scratch block (DESIGN §5e); the implicit-damping solve then always
// runs, since a row may hold damping where the model has none.
template <bool PRM = false>
MJB_DEV int substep(const Ctx& c, bool sensors, bool integrate, int* iters_out, int* dropped) {
  const DM& dm = *c.dm;
  const int nv = dm.nv, lane = c.lane;
  float *qpos = SF(qpos), *qvel = SF(qvel), *qacc = SF(qacc);
  const float h = dm.timestep;
  const bool rk4 = integrate && dm.integrator == MJB_INT_RK4;
  const int nstage = rk4 ? 4 : 1;
  float* rk = SF(rk);
  float *q0 = rk, *v0 = rk + dm.nq, *dq = rk + dm.nq + nv, *dv = rk + dm.nq + 2 * nv;
  int ncon = 0;
  MJB_NOUNROLL
  for (int st = 0; st < nstage; st++) {
    if (st > 0) {
      // stage state: q = q0 (+) h A x_{st-1}.v ; v = v0 + h A f_{st-1}   (A = 1/2, 1/2, 1)
      const float A = st == 3 ? 1.0f : 0.5f;
      float vprev = lane < nv ? qvel[lane] : 0.f, aprev = lane < nv ? qacc[lane] : 0.f;
      MJB_SYNC();
      if (lane < nv) SF(vecC)[lane] = A * vprev;
      MJB_NOUNROLL
      for (int i = lane; i < dm.nq; i += 32) qpos[i] = q0[i];
      MJB_SYNC();
      integrate_pos(c, qpos, SF(vecC), h);
      if (lane < nv) qvel[lane] = v0[lane] + h * A * aprev;
      MJB_SYNC();
    }
    ncon = forward<PRM>(c, sensors && st == 0, sensors && st == nstage - 1, st == 0 ? iters_out : nullptr, dropped);
    if (rk4) {
      const float Bw = (st == 0 || st == 3) ? (1.f / 6) : (1.f / 3);
      if (st == 0) {
        MJB_NOUNROLL
        for (int i = lane; i < dm.nq; i += 32) q0[i] = qpos[i];
        if (lane < nv) { v0[lane] = qvel[lane]; dq[lane] = 0.f; dv[lane] = 0.f; }
      }
      if (lane < nv) { dq[lane] += Bw * qvel[lane]; dv[lane] += Bw * qacc[lane]; }
      MJB_SYNC();
    }
  }
  if (!integrate) return ncon;
  if (rk4) {
    if (lane < nv) qvel[lane] = v0[lane] + h * dv[lane];
    MJB_NOUNROLL
    for (int i = lane; i < dm.nq; i += 32) qpos[i] = q0[i];
    MJB_SYNC();
    integrate_pos(c, qpos, dq, h);
    MJB_SYNC();
    return ncon;
  }
  float acc = lane < nv ? qacc[lane] : 0.f;
  if (PRM || dm.has_damping) {
    // (M + h D) a' = qfrc_smooth + qfrc_constraint
    float *M = SF(M), *H = SF(H);
    const int t0 = CI(dof_t0)[lane], t1 = CI(dof_t1)[lane];
    float rhs = lane < nv ? SF(vecA)[lane] : 0.f;   // qfrc_smooth + J' f at the solver's exit point
    MJB_SYNC();
    acc = factor_solve(M, H, lane, t0, t1, dm.maxtree, lane < nv ? h * PF(dof_damping, prm_damping(dm))[lane] : 0.f, rhs, nv);
  }
  if (lane < nv) qvel[lane] += h * acc;
  MJB_SYNC();
  integrate_pos(c, qpos, qvel, h);
  MJB_SYNC();
  return ncon;
}

}  // namespace mjb
