/*
 * mjb.h — C-ABI of the B200-native batched MuJoCoRL.step hot path.
 *
 * This is the boundary a maintainer of the reference binds instead of the `mujoco`
 * pybind module (the reference's only FFI on the step path).  Each entry point names
 * the reference call site it replaces (paths relative to the reference repo):
 *
 *   mjb_model_create      mj.MjModel.from_xml_path          MuJoCo_Gym/mujoco_parent.py:126
 *   mjb_model_dims        model.nq / nv / nu / opt.timestep  mujoco_parent.py:204-212, fps_custom_env.py:20
 *   mjb_name2id/id2name   data.body(n) / data.geom(n) / model.joint(n) named access
 *                                                            mujoco_parent.py:151,204,293,403-425,441-443,463-470
 *   mjb_batch_create      mj.MjData(model)                   mujoco_parent.py:127   (x num_envs)
 *   mjb_reset             mj_resetData + mj_forward + store wipe + timestep=0
 *                                                            mujoco_parent.py:349-350, mujoco_rl.py:312,330
 *   mjb_step              apply_action + skip_frames x mj_step + get_observations + dynamics /
 *                         reward / truncation / done loops   mujoco_parent.py:316-336,380-392,
 *                                                            mujoco_rl.py:243-289
 *   mjb_step_host         the same through HOST buffers (what one reference `env.step` call sees)
 *
 * Conventions: every function returns 0 on success or a negative MJB_ERR_* code and never
 * throws across the ABI; mjb_last_error() holds the message of the last failure on the calling
 * thread (the Python layer turns it into `Exception(msg)` like the reference's `raise Exception`).
 * A batch handle is not thread-safe.  All device work is enqueued on the stream given at
 * creation; only *_host entry points and mjb_sync synchronise.  No CPU fallback exists: batch
 * creation fails loudly without a CUDA device.
 */
#ifndef MJB_H_
#define MJB_H_

#include <stdint.h>

#include "mjb_blob.h"

#ifdef __cplusplus
extern "C" {
#endif

#define MJB_OK 0
#define MJB_ERR_PARSE -1    /* MJCF syntax / unsupported element */
#define MJB_ERR_ARG -2      /* bad argument */
#define MJB_ERR_CUDA -3     /* CUDA runtime failure (incl. no device) */
#define MJB_ERR_LIMIT -4    /* model exceeds a compiled-in kernel limit */

typedef struct mjb_model mjb_model;
typedef struct mjb_batch mjb_batch;

typedef struct mjb_dims {
  int32_t nq, nv, nu, nbody, njnt, ngeom, nsite, nsensor, nsensordata, npair;
  int32_t integrator;     /* MJB_INT_EULER / MJB_INT_RK4 */
  int32_t ncam;           /* <camera> elements (agent cameras, mujoco_parent.py:505-516) */
  double timestep;
} mjb_dims;

/* ---- model (host only, no CUDA needed) ---------------------------------------------------- */
int mjb_model_create(const char* mjcf_text, mjb_model** out);
void mjb_model_destroy(mjb_model* m);
int mjb_model_dims(const mjb_model* m, mjb_dims* out);
/* packed blob (include/mjb_blob.h); pointer stays valid until mjb_model_destroy */
const void* mjb_model_blob(const mjb_model* m, int64_t* nbytes);
/* -1 when the name does not exist (lets the caller keep the reference's body -> geom fallback) */
int mjb_name2id(const mjb_model* m, int objtype, const char* name);
const char* mjb_id2name(const mjb_model* m, int objtype, int id);
const char* mjb_last_error(void);
const char* mjb_version(void);

/* ---- per-step plugin programme (the reference's plugin lists re-expressed as data) --------- */
enum {
  MJB_DYN_LANGUAGE = 1, /* README.md:108-137: store int(action[0]); observe the first other agent's utterance */
  MJB_DYN_PICKUP = 2    /* Testing/Pick_Up_Dynamic.py:4-41 re-expressed per agent */
};
enum {
  MJB_REW_TAG_DISTANCE = 1, /* README.md:149-163: 10 * (previous distance - distance) to the drawn target */
  MJB_REW_ANT = 2           /* benchmarking/fps_gym/fps_custom_env.py:4-27 */
};
enum { MJB_DONE_DISTANCE_LE = 1 /* README.md:168-173: data_store[agent]["distance"] <= 1 */ };

#define MJB_MAX_AGENTS 8
#define MJB_MAX_PLUGINS 4
#define MJB_MAX_TARGETS 16
#define MJB_MAX_EXTRA_PROBES 48

typedef struct mjb_plugin {
  int32_t kind;      /* MJB_DYN_* / MJB_REW_* / MJB_DONE_* */
  int32_t act_lo;    /* dynamics: slice [act_lo, act_hi) of the agent's action vector (action_routing) */
  int32_t act_hi;
  int32_t n_obs;     /* dynamics: observations appended per agent */
  float param[4];    /* kind specific: threshold, scale ... */
} mjb_plugin;

/* what the Python host derives once from the MJCF + config_dict with the reference's own rules
 * (mujoco_parent.py:233-314, mujoco_rl.py:171-213,355-378) */
typedef struct mjb_env_spec {
  int32_t n_agents;
  int32_t free_joint;                 /* config "freeJoint" */
  int32_t skip_frames;                /* config "skipFrames" */
  int32_t max_steps;                  /* config "maxSteps" */
  int32_t n_phys_act;                 /* physical actions per agent (homogeneous, mujoco_rl.py:182) */
  int32_t act_dim;                    /* physical + dynamic actions per agent */
  int32_t obs_dim[MJB_MAX_AGENTS];    /* total observation length per agent (incl. dynamics) */
  int32_t agent_body[MJB_MAX_AGENTS]; /* body id of every agent */
  const int32_t* act_index;           /* [n_agents * n_phys_act]: ctrl index, or qvel dof index (freeJoint) */
  const int32_t* obs_index;           /* flat list, per agent: (kind << 24) | address; kind 0 sensordata, 1 qpos, 2 qvel */
  int32_t obs_adr[MJB_MAX_AGENTS + 1];
  int32_t n_dynamics, n_rewards, n_dones;
  mjb_plugin dynamics[MJB_MAX_PLUGINS];
  mjb_plugin rewards[MJB_MAX_PLUGINS];
  mjb_plugin dones[MJB_MAX_PLUGINS];
  int32_t n_targets;                       /* filter_by_tag("target") result, duplicates kept */
  int32_t target_objtype[MJB_MAX_TARGETS]; /* MJB_OBJ_BODY (xipos) or MJB_OBJ_GEOM (xpos) */
  int32_t target_objid[MJB_MAX_TARGETS];
  uint64_t seed;                      /* counter-based stream replacing random.randint (README.md:154) */
  int32_t solver_iterations;          /* fixed Newton iteration count per substep (0 = library default) */
  int32_t ls_iterations;              /* fixed line-search iterations (0 = default) */
  int32_t flags;                      /* MJB_SPEC_* bits */
  float reset_noise;                  /* 0 = every reset starts at qpos0 / zero velocity like the reference
                                         (mujoco_parent.py:349); > 0: hinge / slide qpos and all qvel start at
                                         +- reset_noise (uniform, counter-based stream) to decorrelate envs */
  /* extra exported positions beyond the agents and the targets (`distance` / `get_data` / `data.body(n).xipos` for
   * other objects, mujoco_parent.py:394-449): MJB_OBJ_BODY (xipos) or MJB_OBJ_GEOM (xpos) ids.  A spec with extra
   * probes is never packed (one env per warp). */
  int32_t n_extra_probes;
  int32_t extra_objtype[MJB_MAX_EXTRA_PROBES];
  int32_t extra_objid[MJB_MAX_EXTRA_PROBES];
} mjb_env_spec;

/* mjb_env_spec.flags */
enum { MJB_SPEC_NO_PACK = 1 /* one env per warp even for small models (needed by mjb_set_env_subset) */ };

/* Caller-owned device buffers (torch CUDA tensors on the Python side).  Row-major, env-major;
 * strides are in elements and come from mjb_batch_layout. Optional pointers may be NULL. */
typedef struct mjb_layout {
  int32_t num_envs;
  int32_t qpos_stride, qvel_stride, ctrl_stride, sensor_stride; /* floats per env row (16 B aligned) */
  int32_t act_stride;   /* floats per (env, agent) */
  int32_t obs_stride;   /* floats per (env, agent) */
  int32_t probe_count;  /* exported positions: agents' bodies, then targets, then extra probes */
  int32_t maxcon;       /* contact slots per env */
  int32_t store_i32, store_f32; /* per (env, agent) data_store columns */
} mjb_layout;

typedef struct mjb_buffers {
  float* qpos;       /* [N, qpos_stride] */
  float* qvel;       /* [N, qvel_stride] */
  float* ctrl;       /* [N, ctrl_stride] */
  float* warmstart;  /* [N, qvel_stride]  qacc_warmstart */
  float* sensordata; /* [N, sensor_stride] */
  float* probe;      /* [N, probe_count, 4]  xipos / geom xpos of agents and targets (pre-integration, see SURVEY 3.3) */
  float* actions;    /* [N, n_agents, act_stride] input */
  float* obs;        /* [N, n_agents, obs_stride] */
  float* reward;     /* [N, n_agents] */
  uint8_t* term;     /* [N, n_agents + 1]  last column = "__all__" */
  uint8_t* trunc;    /* [N, n_agents + 1] */
  int32_t* timestep; /* [N] */
  int32_t* store_i;  /* [N, n_agents, store_i32] */
  float* store_f;    /* [N, n_agents, store_f32] */
  int32_t* ncon;     /* [N] or NULL */
  int32_t* contact_geom; /* [N, maxcon, 2] or NULL */
  float* contact_dist;   /* [N, maxcon] or NULL */
  int32_t* niter;        /* [N] or NULL: Newton iterations of the last forward pass (diagnostic) */
  int32_t* nreset;       /* [N] or NULL: how often the env was auto-reset because its state became non-finite
                            (MuJoCo's mj_checkPos / mj_checkVel behaviour: warn and mj_resetData) */
  float* probe_quat;     /* [N, probe_count, 4] or NULL: orientation (w, x, y, z) of every exported MOVING body (xmat) /
                            geom (geom xmat) from the same forward pass as `probe`; rows of static objects are left to
                            the caller (constants).  Feeds get_data()["orientation"], mujoco_parent.py:407,419 */
  int32_t* ncon_dropped; /* [N] or NULL: cumulative count of contacts found beyond the env's `maxcon` slots and
                            therefore dropped (MuJoCo grows its arena instead); 0 = every contact was simulated */
} mjb_buffers;

/* data_store column ids */
enum { MJB_STORE_I_UTTERANCE = 0, MJB_STORE_I_HAS_UTTERANCE = 1, MJB_STORE_I_TARGET = 2, MJB_STORE_I_INVENTORY = 3,
       MJB_STORE_I_HAS_XPOS = 4, MJB_STORE_I_DRAWS = 5, MJB_STORE_I_COUNT = 8 };
/* DISTANCE64: the same distance as an fp64 value spread over two float columns (the reward / done arithmetic runs
 * in fp64 like the reference's math.dist on float64 views, mujoco_parent.py:449) */
enum { MJB_STORE_F_DISTANCE = 0, MJB_STORE_F_XPOS_BEFORE = 1, MJB_STORE_F_DISTANCE64 = 2, MJB_STORE_F_COUNT = 4 };

/* ---- batch (CUDA) ---------------------------------------------------------------------------- */
int mjb_batch_layout(const mjb_model* m, const mjb_env_spec* spec, int32_t num_envs, mjb_layout* out);
/* stream: a cudaStream_t cast to void* (NULL = default stream) */
int mjb_batch_create(const mjb_model* m, const mjb_env_spec* spec, int32_t num_envs, int32_t device, void* stream,
                     const mjb_buffers* buffers, mjb_batch** out);
void mjb_batch_destroy(mjb_batch* b);
/* reset envs whose mask byte is non-zero (NULL = all): qpos0, zero velocities, forward pass,
 * data_store wipe, timestep = 0, observations (dynamics applied once with `actions`, results discarded
 * from the store as mujoco_rl.py:322-328 does) */
int mjb_reset(mjb_batch* b, const uint8_t* mask_dev);
/* one MuJoCoRL.step for every env; reads buffers.actions, writes obs / reward / term / trunc */
int mjb_step(mjb_batch* b);
/* physics only (apply_action + skip_frames x mj_step), for stage-wise parity tests */
int mjb_physics(mjb_batch* b, int32_t skip_frames);
/* forward pass only (mj_forward): kinematics, collisions, sensors; no integration */
int mjb_forward(mjb_batch* b);
int mjb_sync(mjb_batch* b);
/* host-buffer call: H2D actions, step, D2H obs/reward/flags, synchronises.  Layouts as above.
 * When all five arrays are page-locked (cudaHostAlloc / torch pin_memory) the kernel writes obs / reward / term /
 * trunc straight into them (zero-copy) and the DEVICE copies buffers.obs / reward / term / trunc are NOT updated by
 * that call: read the results from the host arrays.  State buffers (qpos, qvel, store, timestep ...) are always
 * updated. */
int mjb_step_host(mjb_batch* b, const float* actions, float* obs, float* reward, uint8_t* term, uint8_t* trunc);
/* number of kernel launches issued so far by this handle */
int64_t mjb_launch_count(const mjb_batch* b);
/* average device time (ms) of the step kernel over the launches since the last call; uses CUDA events
 * recorded around each launch when enabled with mjb_set_timing(b, 1) */
int mjb_set_timing(mjb_batch* b, int32_t enable);
int mjb_kernel_time_ms(mjb_batch* b, double* total_ms, int64_t* launches);
/* Level variants (the reference's `xmlPath` list, mujoco_parent.py:88-91,351-356): several batch handles, one
 * per level, are created over the SAME caller-owned buffers; each then steps / resets only the envs currently
 * assigned to its level.  `env_ids_dev` lists `count` distinct env indices in [0, num_envs) (device memory,
 * must stay valid until replaced); NULL restores "all envs".  Needs a batch created with MJB_SPEC_NO_PACK.
 * A reset mask stays indexed by env id. */
int mjb_set_env_subset(mjb_batch* b, const int32_t* env_ids_dev, int32_t count);   /* (non-NULL, 0) = no env at all */
/* Agent cameras (`get_camera_data`, mujoco_parent.py:518-556): renders `ncams` fixed cameras (model camera ids,
 * host array; mjb_name2id with MJB_OBJ_CAMERA) of every env from its current qpos into
 * rgb_dev = u8 [num_envs, ncams, height, width, 3] (device), rows bottom-up as glReadPixels returns them.
 * Image formation: first geom hit per pixel, two-sided head-light shading of the geom's rgba (render_kernel.cuh);
 * the OpenGL pipeline's lights / materials / shadows are not modelled. */
int mjb_render(mjb_batch* b, const int32_t* cam_ids, int32_t ncams, int32_t width, int32_t height, uint8_t* rgb_dev);
/* launch geometry chosen at creation: CTAs, env-warps per CTA, dynamic shared memory per CTA */
int mjb_batch_geometry(const mjb_batch* b, int32_t* grid, int32_t* warps_per_cta, int64_t* smem_bytes);
/* debug builds (-DMJB_PHASE_PROF) only: reads and clears the per-phase clock-cycle counters of the step kernel
 * (step_kernel.cuh PH_*); returns the number of phases, 0 in the product build */
int mjb_phase_cycles(uint64_t* out, int32_t n);
/* counter-based draw used for target selection: exported so tests can reproduce the stream */
uint32_t mjb_draw_u32(uint64_t seed, uint32_t env, uint32_t agent, uint32_t counter);

#ifdef __cplusplus
}
#endif
#endif /* MJB_H_ */
