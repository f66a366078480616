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

#if !defined(__CUDACC_RTC__)
#include <stdint.h>
#endif

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
/* row layout of a per-env parameter table (mjb_env_spec.params) for this model: offsets (in floats) of the five fields
 * in a row, and the row length */
typedef struct mjb_param_offsets {
  int32_t body_mass, body_inertia, geom_friction, actuator_gear, dof_damping;
  int32_t n_params;
} mjb_param_offsets;
int mjb_param_layout(const mjb_model* m, mjb_param_offsets* out);
/* overwrite the fp64 field `name` (count values, the field's full length) of the model, as MuJoCo's
 * `model.body_mass[:] = x` does: nothing mj_setConst derives from it is recomputed (body / dof invweight0, subtree
 * masses ...).  `geom_friction` is the one exception: MuJoCo mixes a contact's friction from the geoms' values at
 * collision time, and this model stores that mix per collision pair (pair_friction, the elementwise max of the two
 * geoms'), so setting geom_friction mixes pair_friction again.  Batches created afterwards use the new values.
 * MJB_ERR_ARG for an unknown name, an int field or a wrong count. */
int mjb_model_set_field(mjb_model* m, const char* name, const double* values, int32_t count);

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
  /* action-space bounds of action dimension d < act_dim, the same for every agent (as action_space.sample() sees
   * them); read only with MJB_SPEC_AUTORESET, for the random action the dynamics are applied with at an auto-reset */
  float act_low[64], act_high[64];
  /* MJB_SPEC_AUTORESET (required then at mjb_batch_create, ignored otherwise): device buffer
   * [N, n_agents, obs_stride] that receives the last observation of every episode mjb_step ends; rows of other envs
   * are not written.  (A field of the spec, not of mjb_buffers, so that mjb_buffers keeps its layout.) */
  float* final_obs;
  /* start-state pool (device memory, caller-owned, must stay valid while the batch lives): rows [n_start, nq] of qpos
   * and [n_start, nv] of qvel of one real env.  n_start = 0: no pool, every reset starts from qpos0 / zero velocity.
   * With a pool, every reset that would start from qpos0 (mjb_reset, full or masked, and the auto-reset of mjb_step)
   * starts instead from pool row mjb_start_index(seed, env, ep, n_start), ep being the key reset_noise uses; the pool
   * replaces qpos0 / zero velocity and nothing else (see mjb_reset_rows).  Level variants: give every level's handle
   * the same pool.  mjb_batch_create refuses (MJB_ERR_ARG) n_start < 0 and n_start > 0 with a NULL pointer. */
  const float* start_qpos;
  const float* start_qvel;
  int32_t n_start;
  /* per-env physical parameters (device memory, caller-owned, must stay valid while the batch lives): rows
   * [N, n_params] of fp32, laid out as mjb_param_layout says, in MuJoCo id order: body_mass [nbody], body_inertia
   * [nbody, 3] (principal), geom_friction [ngeom] (sliding), actuator_gear [nu] (gear[0]), dof_damping [nv].  NULL: no
   * table, every env uses the model's values.  With a table, env n steps exactly as an env of a model whose five fields
   * hold row n would; a contact's friction is max(geom_friction[g1], geom_friction[g2]).  What MuJoCo derives from these
   * fields in mj_setConst keeps its nominal value (body / dof invweight0 and with them the contact and limit
   * regularisers, subtree masses), as after editing model.body_mass in MuJoCo without calling mj_setConst.  Entries of
   * static bodies (and of the world body) are ignored.  Rows persist: the caller may write them between launches and the
   * next launch uses them.
   * MJB_SPEC_RANDOMIZE: every reset (mjb_reset, full or masked, mjb_reset_rows and the auto-reset of mjb_step)
   * overwrites the row of every env it resets with nominal * s before the env's forward pass, s = mjb_param_scale(seed,
   * env, family, index, ep, param_lo[family], param_hi[family]) drawn per element (index: the MuJoCo body / geom /
   * actuator / dof id; a body's three inertia entries take its mass's s); families 0 body_mass + body_inertia,
   * 1 geom_friction, 2 actuator_gear, 3 dof_damping.  Entries of static bodies are not written.  Level variants: give
   * every level's handle the same table; rows hold values, not scales, so when the caller moves an env to another
   * level it writes that env's row (MuJoCoRL writes the new level's nominal values unless it randomises).  mjb_batch_create refuses (MJB_ERR_ARG) MJB_SPEC_RANDOMIZE without a table,
   * non-finite ranges, lo > hi, lo < 0 (lo <= 0 for family 0), and a table with skip_frames = 0. */
  float* params;
  float param_lo[4], param_hi[4];
} mjb_env_spec;

/* mjb_env_spec.flags */
enum {
  MJB_SPEC_NO_PACK = 1,   /* one env per warp even for small models (needed by mjb_set_env_subset) */
  MJB_SPEC_AUTORESET = 2, /* mjb_step resets every env whose step ends its episode, in the same launch (see mjb_step) */
  MJB_SPEC_RANDOMIZE = 4, /* every reset draws the env's row of spec.params (see mjb_env_spec.params) */
  MJB_SPEC_GENERIC = 8    /* mjb_step runs the generic step kernel, not the one compiled for the model's shape */
};


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
 * from the store as mujoco_rl.py:322-328 does), reward / term / trunc = 0.  Never auto-resets. */
int mjb_reset(mjb_batch* b, const uint8_t* mask_dev);
/* mjb_reset, except that every masked env starts from the qpos / qvel rows it currently holds in buffers.qpos /
 * buffers.qvel (as the caller wrote them) instead of qpos0 / zero velocity (or a pool row).  Everything else is as in
 * mjb_reset: ctrl and warm start zeroed, one forward pass, store wiped keeping its draw counters, dynamics applied once
 * with `actions` and discarded, timestep = 0, observations, reward / term / trunc = 0.  reset_noise is added on top
 * (hinge / slide qpos += noise, qvel += noise, the same draws as mjb_reset), keyed by the caller's rows.  Rows are
 * used as given, except that a free joint's quaternion is stored normalised, as every forward pass stores it. */
int mjb_reset_rows(mjb_batch* b, const uint8_t* mask_dev);
/* one MuJoCoRL.step for every env; reads buffers.actions, writes obs / reward / term / trunc.
 * With MJB_SPEC_AUTORESET, every env whose step sets term[n_agents] | trunc[n_agents] (the "__all__" columns) then
 * has its obs rows copied to spec.final_obs and is reset in the same launch, as mjb_reset with its mask byte set
 * would reset it, with two differences: the dynamics are applied with the random action of mjb_reset_action (one
 * draw per agent and action dimension, keyed by the env's rows as the finishing step left them) instead of
 * buffers.actions, and reward / term / trunc keep the values of the finishing step.  buffers.obs then holds the
 * new episode's first observation.  Refused at creation (MJB_ERR_ARG) with skip_frames = 0. */
int mjb_step(mjb_batch* b);
/* physics only (apply_action + skip_frames x mj_step), for stage-wise parity tests */
int mjb_physics(mjb_batch* b, int32_t skip_frames);
/* forward pass only (mj_forward): kinematics, collisions, sensors; no integration */
int mjb_forward(mjb_batch* b);
int mjb_sync(mjb_batch* b);
/* host-buffer call: H2D actions, step, D2H obs/reward/flags, synchronises.  Layouts as above.  MJB_ERR_ARG on a
 * batch created with MJB_SPEC_AUTORESET.
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
 * A reset mask stays indexed by env id.  MJB_ERR_ARG on a batch created with MJB_SPEC_AUTORESET (a reset there
 * cannot draw a new level). */
int mjb_set_env_subset(mjb_batch* b, const int32_t* env_ids_dev, int32_t count);   /* (non-NULL, 0) = no env at all */
/* Agent cameras (`get_camera_data`, mujoco_parent.py:518-556): renders `ncams` fixed cameras (model camera ids,
 * host array; mjb_name2id with MJB_OBJ_CAMERA) of every env from its current qpos into
 * rgb_dev = u8 [num_envs, ncams, height, width, 3] (device), rows bottom-up as glReadPixels returns them.
 * Image formation: first geom hit per pixel, two-sided head-light shading of the geom's rgba (render_kernel.cuh);
 * the OpenGL pipeline's lights / materials / shadows are not modelled. */
int mjb_render(mjb_batch* b, const int32_t* cam_ids, int32_t ncams, int32_t width, int32_t height, uint8_t* rgb_dev);
/* launch geometry chosen at creation: CTAs, env-warps per CTA, dynamic shared memory per CTA */
int mjb_batch_geometry(const mjb_batch* b, int32_t* grid, int32_t* warps_per_cta, int64_t* smem_bytes);
/* The physics step of mjb_step runs a kernel compiled at mjb_batch_create for the model's shape (sizes, strides and
 * offsets as constants; NVRTC, once per shape and process), with the same results as the generic kernel.  Without NVRTC
 * of the release that built the library, with MJB_SPEC_GENERIC, or when the compile fails, the batch runs the generic
 * kernel.  `specialised`: which one runs; `compile_ms`: NVRTC time of the shape; `reason`: why not specialised ("" if it is). */
int mjb_batch_spec_info(const mjb_batch* b, int32_t* specialised, double* compile_ms, char* reason, int32_t reason_len);
/* compile the specialised step kernel a batch of (m, spec, num_envs) would run, without a device: its cubin goes to
 * `cubin` when *cubin_bytes is large enough; *cubin_bytes returns its size */
int mjb_spec_compile(const mjb_model* m, const mjb_env_spec* spec, int32_t num_envs, double* compile_ms, void* cubin, int64_t* cubin_bytes);
/* debug builds (-DMJB_PHASE_PROF) only: reads and clears the per-phase clock-cycle counters of the step kernel
 * (step_kernel.cuh PH_*); returns the number of phases, 0 in the product build */
int mjb_phase_cycles(uint64_t* out, int32_t n);
/* counter-based draw used for target selection: exported so tests can reproduce the stream */
uint32_t mjb_draw_u32(uint64_t seed, uint32_t env, uint32_t agent, uint32_t counter);
/* the random action an auto-reset (MJB_SPEC_AUTORESET) applies the dynamics with, for action dimension `dim` of
 * `agent` in `env`:
 *   u = (mjb_draw_u32(seed ^ 0x5eedc0de, env, 0xC000 + agent * 64 + dim, ep) >> 8) * 2^-24
 *   a = low + u * (high - low)     (fp32, each operation rounded to nearest, no fused multiply-add)
 * ep = timestep ^ bits(qpos[0]) ^ (bits(qvel[0]) << 13) of the env's rows as the finishing step left them (the key
 * reset_noise uses); low / high = act_low[dim] / act_high[dim] of the spec */
float mjb_reset_action(uint64_t seed, uint32_t env, uint32_t agent, uint32_t dim, uint32_t ep, float low, float high);
/* the pool row a reset of `env` starts from (spec.n_start > 0), in [0, n_start):
 *   p = (mjb_draw_u32(seed ^ 0x5eedc0de, env, 0xD000, ep) * (uint64_t)n_start) >> 32
 * ep = the reset_noise / mjb_reset_action key of the env's rows before the reset.  Each env of a packed warp draws its
 * own row.  Returns 0 for n_start < 1. */
uint32_t mjb_start_index(uint64_t seed, uint32_t env, uint32_t ep, int32_t n_start);
/* the scale a randomising reset (MJB_SPEC_RANDOMIZE) applies to element `index` of parameter family `family` (0..3):
 *   u = (mjb_draw_u32(seed ^ 0x5eedc0de, env, 0x10000 + 0x1000 * family + index, ep) >> 8) * 2^-24
 *   s = lo + u * (hi - lo)     (fp32, each operation rounded to nearest, no fused multiply-add)
 * the new value is nominal * s (fp32).  ep = the reset_noise / mjb_reset_action key of the env's rows before the reset. */
float mjb_param_scale(uint64_t seed, uint32_t env, int32_t family, uint32_t index, uint32_t ep, float lo, float hi);

#ifdef __cplusplus
}
#endif
#endif /* MJB_H_ */
