// dev_model.h — fp32 device image of a compiled model + the per-env shared-memory plan.
//
// Host side (build_dev_model): turns the fp64 blob (ModelView) + the env spec into ONE flat
// 4-byte-word image that the step kernel stages into shared memory with a single TMA bulk copy
// (cp.async.bulk, SASS UBLKCP), plus a small POD header (DevModel) passed as a kernel parameter.
// Device side: typed accessors over the image.
#pragma once
#if !defined(__CUDACC_RTC__)
#include <stdint.h>
#endif

#ifndef MJB_HD
#if defined(__CUDACC__)
#define MJB_HD __host__ __device__ __forceinline__
#else
#define MJB_HD inline
#endif
#endif

namespace mjb {

// ---- constant image fields --------------------------------------------------------------------
// Moving bodies are renumbered ("kernel order") by tree depth so that one FK level is a contiguous
// lane range.  Static bodies do not exist on the device: their geoms carry precomputed world frames.
#define MJB_IMAGE_FIELDS(X)                                                                         \
  X(level_adr)      /* int [nlevel+1]  kernel-body range of every depth level                    */ \
  X(mb_parent)      /* int [nmb]       parent kernel body, -1 = static parent (pose folded in)   */ \
  X(mb_root)        /* int [nmb]       kernel body of the tree root                              */ \
  X(mb_jntadr)      /* int [nmb]                                                                 */ \
  X(mb_jntnum)      /* int [nmb]                                                                 */ \
  X(mb_dofadr)      /* int [nmb]       first dof, -1 if none                                     */ \
  X(mb_dofnum)      /* int [nmb]                                                                 */ \
  X(mb_childadr)    /* int [nmb+1]                                                               */ \
  X(mb_child)       /* int [nmb]       children lists                                            */ \
  X(mb_dofmask)     /* u32 [nmb*2]     dofs on the chain world->body (bit d), nv <= 64           */ \
  X(mb_pos)         /* f32 [nmb*3]     frame in parent (world frame when mb_parent == -1)        */ \
  X(mb_quat)        /* f32 [nmb*4]                                                               */ \
  X(mb_ipos)        /* f32 [nmb*3]                                                               */ \
  X(mb_iquat)       /* f32 [nmb*4]                                                               */ \
  X(mb_mass)        /* f32 [nmb]                                                                 */ \
  X(mb_inertia)     /* f32 [nmb*3]                                                               */ \
  X(mb_invweight)   /* f32 [nmb]       body_invweight0 (translational)                           */ \
  X(jnt_type)       /* int [njnt]                                                                */ \
  X(jnt_qposadr)    /* int [njnt]                                                                */ \
  X(jnt_dofadr)     /* int [njnt]                                                                */ \
  X(jnt_pos)        /* f32 [njnt*3]                                                              */ \
  X(jnt_axis)       /* f32 [njnt*3]                                                              */ \
  X(jnt_qpos0)      /* f32 [njnt]      reference angle (hinge / slide)                           */ \
  X(lim_dof)        /* int [nlim]      limited joints: dof, qpos address                         */ \
  X(lim_qposadr)    /* int [nlim]                                                                */ \
  X(lim_param)      /* f32 [nlim*12]   range lo, hi, margin, K, B, invweight, solimp[5], pad     */ \
  X(dof_mb)         /* int [nv]                                                                  */ \
  X(dof_parent)     /* int [nv]                                                                  */ \
  X(dof_kind)       /* int [nv]        0 hinge/slide axis in body, 1 free translation, 2 free rotation */ \
  X(dof_t0)         /* int [32]        first dof of the lane's kinematic tree (lane = dof)        */ \
  X(dof_t1)         /* int [32]        one past the last dof of that tree (0 for lanes >= nv)     */ \
  X(dof_lim)        /* int [32]        limited-joint slot of the dof (lane = dof), -1 = none (also lanes >= nv) */ \
  X(dof_armature)   /* f32 [nv]                                                                  */ \
  X(dof_damping)    /* f32 [nv]                                                                  */ \
  X(geom_type)      /* int [ngeom]                                                               */ \
  X(geom_mb)        /* int [ngeom]     kernel body, -1 static                                    */ \
  X(geom_slot)      /* int [ngeom]     slot in the per-env dynamic geom frames, -1 static        */ \
  X(geom_size)      /* f32 [ngeom*3]                                                             */ \
  X(geom_rbound)    /* f32 [ngeom]                                                               */ \
  X(geom_pos)       /* f32 [ngeom*3]   local (dynamic) or world (static)                         */ \
  X(geom_mat)       /* f32 [ngeom*9]   static: world rotation; dynamic: unused                   */ \
  X(geom_quat)      /* f32 [ngeom*4]   dynamic: local quaternion                                 */ \
  X(geom_ray)       /* int [ngeom]     1 if visible to rays (alpha != 0)                         */ \
  X(pair_pack)      /* u32 [npair]     g1 | g2 << 12 | class << 24  (sorted by type pair)        */ \
  X(pclass)         /* f32 [nclass*12] margin, includemargin, mu, K, B, solimp[5], condim, pad   */ \
  X(bp_block)       /* [nblock*4]      pair blocks (tree x tree | tree x static geom): see BP_*  */ \
  X(bp_passmask)    /* u32 [npass*2]   blocks present in each 32-pair pass of the broad phase    */ \
  X(site_mb)        /* int [nsite]                                                               */ \
  X(site_type)      /* int [nsite]                                                               */ \
  X(site_pos)       /* f32 [nsite*3]   local (or world when static)                              */ \
  X(site_quat)      /* f32 [nsite*4]                                                             */ \
  X(site_size)      /* f32 [nsite*3]                                                             */ \
  X(sensor_type)    /* int [nsensor]                                                             */ \
  X(sensor_site)    /* int [nsensor]   site; jointpos / jointvel: qpos / dof address             */ \
  X(sensor_adr)     /* int [nsensor]                                                             */ \
  X(sensor_dim)     /* int [nsensor]                                                             */ \
  X(sensor_dtype)   /* int [nsensor]   0 real, 1 positive, 2 axis, 3 quaternion                  */ \
  X(sensor_cutoff)  /* f32 [nsensor]                                                             */ \
  X(act_dof)        /* int [nu]                                                                  */ \
  X(act_param)      /* f32 [nu*4]      gear, ctrllimited, lo, hi                                 */ \
  X(dof_actadr)     /* int [nv]        actuators acting on a dof: range in act_list              */ \
  X(dof_actnum)     /* int [nv]                                                                  */ \
  X(act_list)       /* int [nu]        actuator ids grouped by dof                               */ \
  X(probe_kind)     /* int [nprobe]    0 body xipos (kernel body), 1 geom xpos, 2 constant       */ \
  X(probe_id)       /* int [nprobe]                                                              */ \
  X(probe_const)    /* f32 [nprobe*3]  value for constant (static) probes                        */ \
  X(act_index)      /* int [n_agents*n_phys_act]                                                 */ \
  X(obs_index)      /* int [sum obs]   (kind << 24) | address                                    */ \
  X(tri_lut)        /* u32 [136]       pair p = r (r + 1) / 2 + c  ->  r | c << 8   (r >= c, r < 16)       */ \
  X(qpos0)          /* f32 [nq]                                                                  */

enum ImageField {
#define X(n) IF_##n,
  MJB_IMAGE_FIELDS(X)
#undef X
      IF_COUNT
};

// ---- per-env shared-memory scratch fields ---------------------------------------------------
#define MJB_SMEM_FIELDS(X)                                                                          \
  X(qpos) X(qvel) X(qacc) X(ctrl) X(qfrc) /* state, current accel iterate, smooth force         */ \
  X(xpos) X(xquat) X(xmat) X(xipos)       /* body frames                                         */ \
  X(cdof) X(cinert) X(cfrc) X(cvel) X(cacc) /* spatial quantities about the tree root origin     */ \
  X(gpos) X(gmat) X(spos) X(smat)         /* dynamic geom / site world frames                    */ \
  X(M) X(H)                               /* joint-space inertia, Newton Hessian / factors       */ \
  X(cand)                                 /* broadphase survivors (pair indices)                 */ \
  X(con)                                  /* contacts: dist, pos3, frame9, pair, mu, pad -> 16   */ \
  X(J)                                    /* contact Jacobians, 3 rows per contact (n, t1, t2)   */ \
  X(efcD) X(efcAref) X(efcJar) X(efcJv)   /* per-row: limits 2*nlim then 4 per contact           */ \
  X(vecA) X(vecB) X(vecC) X(vecD)         /* nv-sized temporaries (force, grad, search, spare)    */ \
  X(rk)                                   /* RK4 stage storage: q0, v0, dq, dv                    */ \
  X(sens)                                 /* sensordata                                          */

enum SmemField {
#define X(n) SF_##n,
  MJB_SMEM_FIELDS(X)
#undef X
      SF_COUNT
};

struct DevPlugin {
  int kind, act_lo, act_hi, n_obs;
  float param[4];
};

struct DevModel {
  // sizes
  int nq, nv, nu, nmb, njnt, nlim, ngeom, ngdyn, nsite, nsensor, nsensordata, npair, nclass, nlevel, nprobe;
  int maxcon, maxcand, maxefc, ldj, maxtree, nblock;
  // packing: `pack` real envs per warp (see replicate.h); the *1 sizes are those of ONE real env
  int pack, a1, t1, nq1, nv1, nu1, ns1, np1, ngeom1, maxcon1;
  int integrator, has_damping, need_acc_sensors;
  float timestep, gravity[3];
  double timestep_d;   // opt.timestep as compiled (fp64): the ant reward divides by it like the reference
  int solver_iterations, ls_iterations;
  float solver_tol;
  float reset_noise;   // 0: resets start exactly at qpos0 (reference behaviour)
  int njnt1;           // joints of one real env
  // env spec
  int n_agents, free_joint, skip_frames, max_steps, n_phys_act, act_dim;
  int obs_dim[8], obs_adr[9], agent_probe[8];
  int n_dynamics, n_rewards, n_dones, n_targets;
  DevPlugin dynamics[4], rewards[4], dones[4];
  int target_probe[16];
  unsigned long long seed;
  // layout
  int off[IF_COUNT];      // word offsets into the constant image
  int image_words;        // multiple of 4 (16 B) for the bulk copy
  int soff[SF_COUNT];     // word offsets into one env's scratch
  int env_words;          // scratch words per env (multiple of 4)
  // HBM strides
  int qpos_stride, qvel_stride, ctrl_stride, sensor_stride, act_stride, obs_stride, store_i32, store_f32;
  // MJB_SPEC_AUTORESET: the step resets the envs it finishes; bounds of the one action slot each dynamic reads (act_lo:
  // Language's utterance; the random action of the reset, mjb_reset_action).  Last, and 48 bytes in this order, so that
  // the kernels without the flag address every other field and kernel parameter with the same 16-byte alignment as before.
  float* final_obs;    // [N, A, obs_stride] (mjb_env_spec.final_obs)
  int autoreset;
  float dyn_act_low[4], dyn_act_high[4];
  // start-state pool (mjb_env_spec.start_qpos / start_qvel / n_start): rows of one real env, nq1 / nv1 floats each.
  // 32 bytes, padded for the same reason as the auto-reset fields above.
  const float* start_qpos;
  const float* start_qvel;
  int n_start;
  int start_pad[3];
  // per-env parameter table (mjb_env_spec.params, DESIGN §5e): 64 bytes, padded like the fields above.  Only batches with
  // a table set them; their kernels (PRM) keep the env's values in a scratch block of prm_n words at soff prm_soff:
  // body mass [nmb] and inertia [nmb*3] in kernel order, then dof damping [nv], actuator gear [nu], geom friction
  // [ngeom] in (virtual) MuJoCo order.  Image word offsets: prm_map (u32 [prm_n]: row offset | index << 16 | family << 28
  // | copy << 30) and prm_nominal (f32 [prm_n]).
  float* params;       // [N, n_params]
  int n_params, prm_n;
  int randomize, prm_soff, off_prm_map, off_prm_nominal;
  float prm_lo[4], prm_hi[4];
  // frame, velocity and joint sensors (DESIGN §5f): 8 bytes.  off_sens_obj: image word offset of one SO_STRIDE record per
  // sensor, present only when ext_sensors is set.
  int ext_sensors, off_sens_obj;
  // MJB_SPEC_AUTORESET: [N, qpos_stride] rows of the episodes a step ends (mjb_env_spec.final_qpos), null: not written.
  // It takes the 8 padding bytes that ended the struct, so the size and every kernel parameter offset stay as they were.
  float* final_qpos;
};
// Object record of a frame / velocity sensor: the kernel body the object rides on (-1: static) and the object's pose in
// that body's frame (in the world frame when static).  jointpos / jointvel keep their qpos / dof address in sensor_site.
enum { SO_MB = 0, SO_POS = 1, SO_QUAT = 4, SO_STRIDE = 8 };
// Image sensor_type of framex/y/zaxis on a body, xbody or geom: the evaluation pass of the other frame sensors takes them,
// the site-only path in sensors_pos does not.
enum { KSENS_OBJ_AXIS = 64 };
// offsets of the parameter families inside the PRM scratch block
template <class M> MJB_HD int prm_inertia(const M& dm) { return dm.nmb; }
template <class M> MJB_HD int prm_damping(const M& dm) { return 4 * dm.nmb; }
template <class M> MJB_HD int prm_gear(const M& dm) { return 4 * dm.nmb + dm.nv; }
template <class M> MJB_HD int prm_friction(const M& dm) { return 4 * dm.nmb + dm.nv + dm.nu; }

// The model's warp-uniform integer shape: sizes, strides, word offsets, plugin counts and flags.  Two models with the same
// shape differ only in values (floats, pointers, seed, the per-lane image tables) and can share one specialised kernel.
#define MJB_SHAPE_FIELDS(X)                                                                                                  \
  X(nq) X(nv) X(nu) X(nmb) X(njnt) X(nlim) X(ngeom) X(ngdyn) X(nsite) X(nsensor) X(nsensordata) X(npair) X(nclass)         \
  X(nlevel) X(nprobe) X(maxcon) X(maxcand) X(maxefc) X(ldj) X(maxtree) X(nblock)                                           \
  X(pack) X(a1) X(t1) X(nq1) X(nv1) X(nu1) X(ns1) X(np1) X(ngeom1) X(maxcon1) X(njnt1)                                     \
  X(integrator) X(has_damping) X(need_acc_sensors) X(solver_iterations) X(ls_iterations)                                   \
  X(n_agents) X(free_joint) X(n_phys_act) X(act_dim) X(n_dynamics) X(n_rewards) X(n_dones) X(n_targets)                   \
  X(image_words) X(env_words) X(qpos_stride) X(qvel_stride) X(ctrl_stride) X(sensor_stride) X(act_stride) X(obs_stride)    \
  X(store_i32) X(store_f32) X(autoreset) X(n_params) X(prm_n) X(prm_soff) X(off_prm_map) X(off_prm_nominal)                \
  X(ext_sensors) X(off_sens_obj)

// The step kernel reads the model through `DM`.  In the generic build DM is DevModel: every field is a load of the kernel
// parameter.  The specialised build (MJB_SPEC: one NVRTC compile per batch shape, mjb_batch.cu) includes a generated
// header that derives SpecModel from DevModel and hides each MJB_SHAPE_FIELDS member with a constant of the same name, and
// defines the image / scratch word offsets (spec_off, spec_soff): the same source then folds the shape into the code.
#if defined(MJB_SPEC)
}  // namespace mjb
#include "mjb_spec_shape.h"
namespace mjb {
typedef SpecModel DM;
#else
typedef DevModel DM;
#endif

// ---- camera rendering (render_kernel.cuh): a second, small constant table next to the image -------------
// cam record: kernel body (-1 = static: pose already in the world frame), mode (0 fixed), pos[3], quat[4],
// tan(fovy / 2), 2 pad words; then one clamped RGBA (4 floats) per geom
enum { CAM_MB = 0, CAM_MODE = 1, CAM_POS = 2, CAM_QUAT = 5, CAM_TANHALF = 9, CAM_STRIDE = 12 };
struct RenderHdr {
  int ncam, ngeom;
  int off_cam, off_rgba;   // word offsets into the table
  int words;               // multiple of 4
};
// per-env geom record the rays walk (built in shared memory after the kinematics pass)
enum { GL_POS = 0, GL_MAT = 3, GL_SIZE = 12, GL_TYPE = 15, GL_RBOUND = 16, GL_RGB = 17, GL_STRIDE = 20 };

// contact record layout inside SF_con (16 words per contact)
// (CON_DOFS: the dofs of the contact's mask as up to 16 packed bytes, ascending)
enum { CON_DIST = 0, CON_POS = 1, CON_FRAME = 4, CON_PAIR = 13, CON_MU = 14, CON_MASK = 15, CON_DOFS = 16, CON_STRIDE = 20 };
enum { LIM_LO = 0, LIM_HI, LIM_MARGIN, LIM_K, LIM_B, LIM_INVW, LIM_SOLIMP, LIM_STRIDE = 12 };
enum { PC_MARGIN = 0, PC_INCMARGIN, PC_MU, PC_K, PC_B, PC_SOLIMP, PC_CONDIM = 10, PC_STRIDE = 12 };
enum { DOF_AXIS = 0, DOF_FREE_TRANS = 1, DOF_FREE_ROT = 2 };
enum { PROBE_BODY = 0, PROBE_GEOM = 1, PROBE_CONST = 2 };
// pair block: root kernel body of tree A, root kernel body of tree B (or -1 - static geom id, or BP_ALWAYS),
// reach of A + reach of B (trees) / reach of A (static partner), largest pair margin in the block
enum { BP_ROOT_A = 0, BP_PARTNER = 1, BP_REACH = 2, BP_MARGIN = 3, BP_STRIDE = 4, BP_ALWAYS = 0x7fffffff };

}  // namespace mjb
