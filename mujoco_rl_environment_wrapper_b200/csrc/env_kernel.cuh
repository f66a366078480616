// env_kernel.cuh — per-environment driver around the physics in step_kernel.cuh: state load /
// action scatter / substeps / state store, and the fused epilogue (observation gather, dynamics,
// reward, truncation, done — MuJoCo_Gym/mujoco_rl.py:243-289 and the reset path :291-331).
#pragma once
#include "step_kernel.cuh"
#if defined(MJB_HOST_EMU)
#define MJB_IMG_WAIT(c) ((void)0)
#else
#include "tma_prims.cuh"
// the model image travels into shared memory by one bulk copy per launch; an env's row loads do not need it, so the
// first env of a warp requests its rows first and waits for the image after
#define MJB_IMG_WAIT(c) do { if ((c).img_bar) mbar_wait((c).img_bar, 0); } while (0)
#endif

namespace mjb {

// MODE_RESET_ROWS: MODE_RESET with the masked envs starting from their own qpos / qvel rows (mjb_reset_rows)
enum { MODE_STEP = 0, MODE_PHYSICS = 1, MODE_FORWARD = 2, MODE_RESET = 3, MODE_RESET_ROWS = 4 };

// agent loops of run_plugins: unrolled when the bound is small (registers), rolled in the general form (code size)
#if defined(MJB_HOST_EMU)
#define MJB_AGENT_LOOP
#else
#define MJB_AGENT_LOOP _Pragma("unroll (AMAX <= 2 ? 2 : 1)")
#endif

// counter-based draw replacing `random.randint` (README.md:154, Testing/Pick_Up_Dynamic.py:28,38)
MJB_HD uint32_t draw_u32(unsigned long long seed, uint32_t env, uint32_t agent, uint32_t counter) {
  unsigned long long z = seed + 0x9E3779B97F4A7C15ull * (1ull + env) + 0xBF58476D1CE4E5B9ull * agent +
                         0x94D049BB133111EBull * counter;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z ^= z >> 31;
  return (uint32_t)(z >> 32);
}

// the random action of an auto-reset (include/mjb.h, mjb_reset_action): uniform in [low, high), keyed like reset_noise
// by how the episode ended; each operation rounded on its own, so that a float32 host evaluation gives the same bits
MJB_HD float reset_action(unsigned long long seed, uint32_t env, uint32_t agent, uint32_t dim, uint32_t ep, float low, float high) {
  const float u = (float)(draw_u32(seed ^ 0x5eedc0deULL, env, 0xC000u + agent * 64u + dim, ep) >> 8) * (1.f / 16777216.f);
#if defined(__CUDA_ARCH__)
  return __fadd_rn(low, __fmul_rn(u, high - low));
#else
  volatile float span = u * (high - low);
  return low + span;
#endif
}

// the start-state pool row of a reset (include/mjb.h, mjb_start_index), keyed like reset_noise
MJB_HD uint32_t start_index(unsigned long long seed, uint32_t env, uint32_t ep, int n_start) {
  return n_start < 1 ? 0u : (uint32_t)(((unsigned long long)draw_u32(seed ^ 0x5eedc0deULL, env, 0xD000u, ep) * (uint32_t)n_start) >> 32);
}

// the scale of a randomising reset (include/mjb.h, mjb_param_scale) for element `index` of parameter family `family`,
// keyed like reset_noise; rounded like reset_action
MJB_HD float param_scale(unsigned long long seed, uint32_t env, uint32_t family, uint32_t index, uint32_t ep, float lo, float hi) {
  const float u = (float)(draw_u32(seed ^ 0x5eedc0deULL, env, 0x10000u + 0x1000u * family + index, ep) >> 8) * (1.f / 16777216.f);
#if defined(__CUDA_ARCH__)
  return __fadd_rn(lo, __fmul_rn(u, hi - lo));
#else
  volatile float span = u * (hi - lo);
  return lo + span;
#endif
}

// Distances, the reward arithmetic and the done comparison run in fp64 on the fp32 positions (the reference computes
// math.dist on float64 numpy views, mujoco_parent.py:428-449): given identical xipos the reward, cast to fp32, and the
// done flag are those of the reference's own arithmetic.  The stored distance keeps its fp64 value in two store_f
// columns (MJB_STORE_F_DISTANCE64, +1) next to the fp32 copy that `data_store[agent]["distance"]` shows.
MJB_DEV double probe_dist(const float* probe, int a, int b) {
  const double dx = (double)probe[4 * a] - (double)probe[4 * b], dy = (double)probe[4 * a + 1] - (double)probe[4 * b + 1],
               dz = (double)probe[4 * a + 2] - (double)probe[4 * b + 2];
  // plain IEEE evaluation, no fused multiply-add: (dx*dx + dy*dy) + dz*dz, so that any fp64 host evaluation of the same
  // expression (numpy, torch) gives the same bits
#if defined(MJB_HOST_EMU)
  volatile double xx = dx * dx, yy = dy * dy, zz = dz * dz;
  return sqrt((xx + yy) + zz);
#else
  return sqrt(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
#endif
}
MJB_DEV double ld_dist(const float* sfa) {
  union { double d; float f[2]; } u;
  u.f[0] = sfa[MJB_STORE_F_DISTANCE64]; u.f[1] = sfa[MJB_STORE_F_DISTANCE64 + 1];
  return u.d;
}
MJB_DEV void st_dist(float* sfa, double d) {
  union { double d; float f[2]; } u;
  u.d = d;
  sfa[MJB_STORE_F_DISTANCE64] = u.f[0]; sfa[MJB_STORE_F_DISTANCE64 + 1] = u.f[1];
  sfa[MJB_STORE_F_DISTANCE] = (float)d;
}

// the dynamics / reward / done programme of one env, executed by one lane in the reference's order
// (dynamic outer, agent inner; then reward fn outer, agent inner; truncation; done fns with early exit)
// `obs` / `rew` / `term` / `trunc` are the env's own result rows ([A, obs_stride], [A], [A + 1], [A + 1]; global or
// shared memory), `ctrl` the env's ctrl row (read by the ant reward), `probe` its exported positions.
// AMAX bounds the agent loops at compile time: with a small AMAX (the tile kernel uses 2) the per-agent accumulators
// live in registers and the loops unroll; MJB_MAX_AGENTS is the general form.
// A reset zeroes rew / term / trunc unless `keep_flags` (auto-reset: they stay those of the step that ended the episode).
// Returns whether the step ended the episode (term[A] | trunc[A]); false for a reset.
template <int AMAX>
MJB_DEV bool run_plugins(const DM& dm, const float* ctrl, float* obs, float* rew, uint8_t* term, uint8_t* trunc, int env, int copy,
                         bool is_reset, const float* probe, int* si, float* sf, const float* act, int* ts_io, const double* dtab = nullptr,
                         bool keep_flags = false) {
  // `env` is the REAL environment, `copy` its slot inside the (possibly packed) virtual env of this warp
  const int A = dm.a1, ab = copy * dm.a1, tb = copy * dm.t1, n_targets = dm.t1;
  // agent - target distance: from the table the warp filled lane-parallel (dist_table), or evaluated here
  auto pdist = [&](int a, int t) { return dtab ? dtab[a * n_targets + t] : probe_dist(probe, dm.agent_probe[ab + a], dm.target_probe[tb + t]); };
  double reward[AMAX];
  bool done[AMAX];
  int opos[AMAX];
  if (is_reset)  // data_store = {agent: {}} (mujoco_rl.py:312); the draw counter is not part of the store
    MJB_AGENT_LOOP
    for (int a = 0; a < AMAX; a++) if (a < A) {
      MJB_NOUNROLL
      for (int k = 0; k < dm.store_i32; k++) if (k != MJB_STORE_I_DRAWS) si[a * dm.store_i32 + k] = 0;
      MJB_NOUNROLL
      for (int k = 0; k < dm.store_f32; k++) sf[a * dm.store_f32 + k] = 0.f;
    }
  MJB_AGENT_LOOP
  for (int a = 0; a < AMAX; a++) if (a < A) { reward[a] = 0.0; done[a] = false; opos[a] = dm.obs_adr[ab + a + 1] - dm.obs_adr[ab + a]; }
  MJB_NOUNROLL
  for (int p = 0; p < dm.n_dynamics; p++) {
    const DevPlugin& dyn = dm.dynamics[p];
    MJB_AGENT_LOOP
    for (int a = 0; a < AMAX; a++) if (a < A) {
      int* sia = si + a * dm.store_i32;
      float* sfa = sf + a * dm.store_f32;
      float* oa = obs + a * dm.obs_stride;
      if (dyn.kind == MJB_DYN_LANGUAGE) {
        int utt = (int)act[a * dm.act_stride + dyn.act_lo];  // int(): truncation toward zero
        sia[MJB_STORE_I_UTTERANCE] = utt; sia[MJB_STORE_I_HAS_UTTERANCE] = 1;
        int other = a == 0 ? 1 : 0;
        float val = 0.f;
        if (other < A && si[other * dm.store_i32 + MJB_STORE_I_HAS_UTTERANCE]) val = (float)si[other * dm.store_i32 + MJB_STORE_I_UTTERANCE];
        oa[opos[a]++] = val;
      } else if (dyn.kind == MJB_DYN_PICKUP) {
        int tgt = sia[MJB_STORE_I_TARGET];
        if (tgt == 0 && n_targets > 0) {
          tgt = 1 + (int)(draw_u32(dm.seed, env, a, sia[MJB_STORE_I_DRAWS]++) % (uint32_t)n_targets);
          sia[MJB_STORE_I_TARGET] = tgt;
        }
        if (tgt > 0) {
          const double d = pdist(a, tgt - 1);
          if (d < (double)dyn.param[0]) {
            sia[MJB_STORE_I_INVENTORY] ^= 1;
            reward[a] += 1.0;
            tgt = 1 + (int)(draw_u32(dm.seed, env, a, sia[MJB_STORE_I_DRAWS]++) % (uint32_t)n_targets);
            sia[MJB_STORE_I_TARGET] = tgt;
            st_dist(sfa, pdist(a, tgt - 1));
          }
          const float* tp = probe + 4 * dm.target_probe[tb + tgt - 1];
          oa[opos[a]] = tp[0]; oa[opos[a] + 1] = tp[1]; oa[opos[a] + 2] = tp[2];
        } else {
          oa[opos[a]] = 0.f; oa[opos[a] + 1] = 0.f; oa[opos[a] + 2] = 0.f;
        }
        oa[opos[a] + 3] = (float)sia[MJB_STORE_I_INVENTORY];
        opos[a] += 4;
      }
    }
  }
  if (is_reset) {
    // everything the dynamics wrote is discarded (mujoco_rl.py:326-328); rewards / dones are not run
    MJB_AGENT_LOOP
    for (int a = 0; a < AMAX; a++) if (a < A) {
      MJB_NOUNROLL
      for (int k = 0; k < dm.store_i32; k++) if (k != MJB_STORE_I_DRAWS) si[a * dm.store_i32 + k] = 0;
      MJB_NOUNROLL
      for (int k = 0; k < dm.store_f32; k++) sf[a * dm.store_f32 + k] = 0.f;
      if (!keep_flags) { rew[a] = 0.f; term[a] = 0; trunc[a] = 0; }
    }
    if (!keep_flags) { term[A] = 0; trunc[A] = 0; }
    *ts_io = 0;
    return false;
  }
  MJB_NOUNROLL
  for (int p = 0; p < dm.n_rewards; p++) {
    const DevPlugin& rf = dm.rewards[p];
    MJB_AGENT_LOOP
    for (int a = 0; a < AMAX; a++) if (a < A) {
      int* sia = si + a * dm.store_i32;
      float* sfa = sf + a * dm.store_f32;
      if (rf.kind == MJB_REW_TAG_DISTANCE) {
        int tgt = sia[MJB_STORE_I_TARGET];
        if (n_targets <= 0) continue;
        if (tgt == 0) {
          tgt = 1 + (int)(draw_u32(dm.seed, env, a, sia[MJB_STORE_I_DRAWS]++) % (uint32_t)n_targets);
          sia[MJB_STORE_I_TARGET] = tgt;
          st_dist(sfa, pdist(a, tgt - 1));
        } else {
          const double d = pdist(a, tgt - 1);
          reward[a] += (ld_dist(sfa) - d) * (double)rf.param[0];
          st_dist(sfa, d);
        }
      } else if (rf.kind == MJB_REW_ANT) {
        float x_after = probe[4 * dm.agent_probe[ab + a]];
        if (!sia[MJB_STORE_I_HAS_XPOS]) {
          sia[MJB_STORE_I_HAS_XPOS] = 1;
        } else {
          double cc = 0.0;
          MJB_NOUNROLL
          for (int u = 0; u < dm.nu1; u++) cc += (double)ctrl[u] * (double)ctrl[u];
          // contact cost term: cfrc_ext is zero on these models (no force / acc sensors, SURVEY Q11); the Python
          // layer refuses to fuse this reward for models with accelerometers, where MuJoCo fills cfrc_ext
          reward[a] += ((double)x_after - (double)sfa[MJB_STORE_F_XPOS_BEFORE]) / dm.timestep_d - 0.5 * cc;
        }
        sfa[MJB_STORE_F_XPOS_BEFORE] = x_after;
      }
    }
  }
  int ts = *ts_io;
  uint8_t tr = ts >= dm.max_steps ? 1 : 0;
  MJB_NOUNROLL
  for (int a = 0; a <= A; a++) trunc[a] = tr;
  bool all = false;
  MJB_NOUNROLL
  for (int p = 0; p < dm.n_dones && !all; p++) {
    const DevPlugin& df = dm.dones[p];
    MJB_AGENT_LOOP
    for (int a = 0; a < AMAX; a++) if (a < A)
      if (df.kind == MJB_DONE_DISTANCE_LE) done[a] = done[a] || (ld_dist(sf + a * dm.store_f32) <= (double)df.param[0]);
    MJB_AGENT_LOOP
    for (int a = 0; a < AMAX; a++) if (a < A) all = all || done[a];
  }
  MJB_AGENT_LOOP
  for (int a = 0; a < AMAX; a++) if (a < A) { rew[a] = (float)reward[a]; term[a] = done[a] ? 1 : 0; }
  term[A] = all ? 1 : 0;
  *ts_io = ts + 1;
  return all || tr;
}

// element i of a virtual per-copy array -> (copy, element); no division in the unpacked case
MJB_DEV void split_copy(int i, int n1, int K, int& k, int& j) {
  if (K == 1) { k = 0; j = i; }
  else { k = i / n1; j = i - k * n1; }
}

// whole per-env pipeline.  Every lane of the warp calls this with the same arguments.  `venv` is the virtual
// environment of this warp: dm.pack real environments (venv * pack + copy) presented to the physics as one
// model with `pack` independent copies (csrc/replicate.h); pack == 1 is the plain case.  Virtual state index i
// of a per-copy array of length n1 maps to copy i / n1, element i % n1 of that real env's HBM row.
// Auto-reset (MJB_SPEC_AUTORESET): after a step, the copies whose episode it ended run this body once more, in
// MODE_RESET with `upd` = those copies, exactly as a masked reset of them would (same call sites: one forward pass in
// the code, see DESIGN §4).  Start states (DESIGN §5d): a reset's fresh copies load the start-state pool row they draw
// (dm.n_start > 0) or, in MODE_RESET_ROWS, their own rows, instead of qpos0 / zero velocity.
// EXT = false compiles auto-reset and start states out (the device kernels of batches and launches that use neither);
// with EXT = true they follow dm.autoreset, dm.n_start and the mode.
// PRM (batches with a parameter table, DESIGN §5e): every copy loads its row of dm.params into the scratch block the
// physics reads; the fresh copies of a reset with dm.randomize draw the row instead and store it back.
template <bool PHYS, bool PACKED, bool EXT = true, bool PRM = false>
MJB_DEV void run_env(const Ctx& c_in, const mjb_buffers& B, int venv, int num_envs, int mode_in, int skip_frames,
                     const uint8_t* reset_mask) {
  uint32_t fin = 0;   // 0: the pass the launch asked for; else the auto-reset pass over these copies (the step pass finished them)
pass:
  const bool auto_pass = fin != 0;
  const bool own_rows = EXT && mode_in == MODE_RESET_ROWS;
  const int mode = (auto_pass || own_rows) ? (int)MODE_RESET : mode_in;
  Ctx c = c_in;
  float* probe = c.probe;
  const DM& dm = *c.dm;
  const int lane = c.lane, K = PACKED ? dm.pack : 1, e0 = venv * K;   // K == 1 folds all copy arithmetic away
  c.probe_quat = (!PACKED && B.probe_quat) ? B.probe_quat + (size_t)e0 * dm.np1 * 4 : nullptr;
  // which copies hold a real env, and which of them this launch updates
  uint32_t live = 0, upd = 0;
  for (int k = 0; k < K; k++)
    if (e0 + k < num_envs) {
      live |= 1u << k;
      if (!(mode == MODE_RESET && reset_mask && !reset_mask[e0 + k])) upd |= 1u << k;
    }
  if (auto_pass) {
    upd = fin;
    c.cta_threads = 0;   // no CTA-level alignment in forward(): the other warps do not run this pass
  }
  if (!upd) return;
  // the loads below read the image only for copies that start from qpos0 or hold no env
  if (mode == MODE_RESET || live != (K >= 32 ? 0xffffffffu : (1u << K) - 1u)) MJB_IMG_WAIT(c);
  float *qpos = SF(qpos), *qvel = SF(qvel), *qacc = SF(qacc), *ctrl = SF(ctrl), *sens = SF(sens);
  auto fresh = [&](int k) { return mode == MODE_RESET && ((upd >> k) & 1u); };   // copy starts from qpos0 (or a start state)
  auto has = [&](int k) { return ((live >> k) & 1u) != 0; };
  // key of a reset's draws: how the previous episode ended (its rows as the last step left them)
  auto reset_key = [&](uint32_t env) {
    return (uint32_t)B.timestep[env] ^ MJB_F2U(B.qpos[(size_t)env * dm.qpos_stride]) ^ (MJB_F2U(B.qvel[(size_t)env * dm.qvel_stride]) << 13);
  };
  // start states: fresh copies load their own rows (own_rows) or the pool row pr[k] they draw, before any row is stored
  const bool pool = EXT && mode == MODE_RESET && !own_rows && dm.n_start > 0, from_start = own_rows || pool;
  uint32_t pr[MJB_MAX_PACK] = {0, 0, 0, 0};
  if (pool) {
#pragma unroll
    for (int k = 0; k < MJB_MAX_PACK; k++)
      if (k < K && fresh(k)) pr[k] = start_index(dm.seed, (uint32_t)(e0 + k), reset_key((uint32_t)(e0 + k)), dm.n_start);
  }
  auto pool_row = [&](const float* base, int n1, int k) {   // constant indices into pr: it stays in registers
    return base + (size_t)(K == 1 || k == 0 ? pr[0] : k == 1 ? pr[1] : k == 2 ? pr[2] : pr[3]) * n1;
  };
  MJB_NOUNROLL
  for (int i = lane; i < dm.nq; i += 32) {
    int k, j;
    split_copy(i, dm.nq1, K, k, j);
    if (from_start && fresh(k)) MJB_G2S(&qpos[i], pool ? pool_row(dm.start_qpos, dm.nq1, k) + j : &B.qpos[(size_t)(e0 + k) * dm.qpos_stride + j]);
    else if (fresh(k) || !has(k)) qpos[i] = CF(qpos0)[i];
    else MJB_G2S(&qpos[i], &B.qpos[(size_t)(e0 + k) * dm.qpos_stride + j]);
  }
  MJB_NOUNROLL
  for (int i = lane; i < dm.nv; i += 32) {
    int k, j;
    split_copy(i, dm.nv1, K, k, j);
    bool z = fresh(k) || !has(k);
    if (from_start && fresh(k)) {
      MJB_G2S(&qvel[i], pool ? pool_row(dm.start_qvel, dm.nv1, k) + j : &B.qvel[(size_t)(e0 + k) * dm.qvel_stride + j]);
      qacc[i] = 0.f;
    } else if (z) { qvel[i] = 0.f; qacc[i] = 0.f; }
    else {
      MJB_G2S(&qvel[i], &B.qvel[(size_t)(e0 + k) * dm.qvel_stride + j]);
      MJB_G2S(&qacc[i], &B.warmstart[(size_t)(e0 + k) * dm.qvel_stride + j]);
    }
  }
  MJB_NOUNROLL
  for (int i = lane; i < dm.nu; i += 32) {
    int k, j;
    split_copy(i, dm.nu1, K, k, j);
    if (fresh(k) || !has(k)) ctrl[i] = 0.f;
    else MJB_G2S(&ctrl[i], &B.ctrl[(size_t)(e0 + k) * dm.ctrl_stride + j]);
  }
  MJB_NOUNROLL
  for (int i = lane; i < dm.nsensordata; i += 32) {
    int k, j;
    split_copy(i, dm.ns1, K, k, j);
    if (fresh(k) || !has(k)) sens[i] = 0.f;
    else MJB_G2S(&sens[i], &B.sensordata[(size_t)(e0 + k) * dm.sensor_stride + j]);
  }
  // exported positions: virtual probe order is [agents of every copy ..., targets of every copy ...]
  auto probe_slot = [&](int p, int& k, int& p1) {
    if (K == 1) { k = 0; p1 = p; }
    else if (p < K * dm.a1) { k = p / dm.a1; p1 = p - k * dm.a1; }
    else { int q = p - K * dm.a1; k = q / dm.t1; p1 = dm.a1 + (q - k * dm.t1); }
  };
  MJB_NOUNROLL
  for (int i = lane; i < 4 * dm.nprobe; i += 32) {
    int k, p1;
    probe_slot(i >> 2, k, p1);
    if (has(k)) MJB_G2S(&probe[i], &B.probe[((size_t)(e0 + k) * dm.np1 + p1) * 4 + (i & 3)]);
    else probe[i] = 0.f;
  }
  // unpacked case: fetch the plugin store rows, dynamic actions and step counter of the env now, so that their
  // global-memory latency overlaps the state loads / the physics; consumed by the epilogue
  const bool epi = (mode == MODE_STEP || mode == MODE_RESET);
  int pre_si[2] = {0, 0}, pre_ts = 0;
  float pre_sf = 0.f, pre_act[2] = {0.f, 0.f};
  if (epi && K == 1) {
    const int* gsi = B.store_i + (size_t)e0 * dm.a1 * dm.store_i32;
    const float* gsf = B.store_f + (size_t)e0 * dm.a1 * dm.store_f32;
    const float* gact = B.actions + (size_t)e0 * dm.a1 * dm.act_stride;
    for (int r = 0; r < 2; r++) {
      int i = lane + 32 * r;
      if (i < dm.a1 * dm.store_i32) pre_si[r] = gsi[i];
      if (i < dm.a1 * dm.act_stride) pre_act[r] = gact[i];
    }
    if (lane < dm.a1 * dm.store_f32) pre_sf = gsf[lane];
    if (lane == 0) pre_ts = B.timestep[e0];
  }
  MJB_IMG_WAIT(c);
  if (PRM) {
    // the env's parameters (the map and the nominal values are image words)
    float* prm = c.s + dm.prm_soff;
    const uint32_t* map = c.img + dm.off_prm_map;
    const float* nominal = (const float*)(c.img + dm.off_prm_nominal);
    MJB_NOUNROLL
    for (int i = lane; i < dm.prm_n; i += 32) {
      const uint32_t e = map[i];
      const int k = (int)(e >> 30), off = (int)(e & 0xffffu);
      float* row = dm.params + (size_t)(e0 + k) * dm.n_params;
      if (!has(k)) prm[i] = nominal[i];
      else if (dm.randomize && fresh(k)) {
        const uint32_t f = (e >> 28) & 3u;
        const float s = param_scale(dm.seed, (uint32_t)(e0 + k), f, (e >> 16) & 0xfffu, reset_key((uint32_t)(e0 + k)), dm.prm_lo[f], dm.prm_hi[f]);
        prm[i] = nominal[i] * s;
        row[off] = prm[i];
      } else MJB_G2S(&prm[i], &row[off]);
    }
  }
  MJB_G2S_WAIT();
  if (MJB_UNLIKELY(mode == MODE_RESET && dm.reset_noise > 0.f)) {
    // optional decorrelated starts (off by default: the reference always restarts at qpos0).  The draw is keyed by
    // (seed, env, joint / dof) and by how the previous episode ended, so that it differs from reset to reset.
    MJB_SYNC();
    MJB_NOUNROLL
    for (int j = lane; j < dm.njnt; j += 32) {
      const int k = K == 1 ? 0 : j / dm.njnt1;
      if (!fresh(k) || !has(k) || CI(jnt_type)[j] == MJB_JNT_FREE) continue;
      const uint32_t env = (uint32_t)(e0 + k);
      const uint32_t ep = reset_key(env);
      const float u = (float)(draw_u32(dm.seed ^ 0x5eedc0deULL, env, 0x4000u + (uint32_t)(j - k * dm.njnt1), ep) >> 8) * (1.f / 16777216.f);
      qpos[CI(jnt_qposadr)[j]] += dm.reset_noise * (2.f * u - 1.f);
    }
    MJB_NOUNROLL
    for (int i = lane; i < dm.nv; i += 32) {
      int k, j;
      split_copy(i, dm.nv1, K, k, j);
      if (!fresh(k) || !has(k)) continue;
      const uint32_t env = (uint32_t)(e0 + k);
      const uint32_t ep = reset_key(env);
      const float u = (float)(draw_u32(dm.seed ^ 0x5eedc0deULL, env, 0x8000u + (uint32_t)j, ep) >> 8) * (1.f / 16777216.f);
      const float d = dm.reset_noise * (2.f * u - 1.f);
      qvel[i] = EXT ? qvel[i] + d : d;   // start velocity + noise (0 + d == d: the same bits without a start state)
    }
  }
  MJB_SYNC();
  if (mode == MODE_STEP || mode == MODE_PHYSICS) {
    // apply_action (mujoco_parent.py:316-332): overwrite qvel (freeJoint) or ctrl
    const int n_act = dm.n_agents * dm.n_phys_act;
    const bool from_regs = K == 1 && epi && dm.a1 * dm.act_stride <= 64;   // the action rows were prefetched above
    MJB_NOUNROLL
    for (int i0 = 0; i0 < n_act; i0 += 32) {
      const int i = i0 + lane;
      const bool on = i < n_act;
      int av = on ? i / dm.n_phys_act : 0, k, a1;
      split_copy(av, dm.a1, K, k, a1);
      const int off = a1 * dm.act_stride + (on ? i - av * dm.n_phys_act : 0);
      float v;
      if (from_regs) {
        const float lo = MJB_SHFL(pre_act[0], off & 31), hi = MJB_SHFL(pre_act[1], off & 31);
        v = off < 32 ? lo : hi;
      } else {
        v = (on && has(k)) ? B.actions[(size_t)(e0 + k) * dm.a1 * dm.act_stride + off] : 0.f;
      }
      if (on && has(k)) {
        int idx = CI(act_index)[i];
        if (dm.free_joint) qvel[idx] = v; else ctrl[idx] = v;
      }
    }
    MJB_SYNC();
  }
  MJB_PH(c, PH_LOAD);
  int ncon = -1;
  // mj_forward (reset / forward modes) is one pass of the same loop body without integration
  const bool integrate = !(mode == MODE_FORWARD || mode == MODE_RESET);
  const int passes = integrate ? skip_frames : 1;
  int niter = 0;
  if (PHYS) {
    int dropped[MJB_MAX_PACK] = {0, 0, 0, 0};
    MJB_NOUNROLL
    for (int f = 0; f < passes; f++) ncon = substep<PRM>(c, f == passes - 1, integrate, &niter, dropped);
    if (B.ncon_dropped && lane == 0) {   // cumulative per real env: stays 0 while no contact was ever dropped
#pragma unroll
      for (int k = 0; k < MJB_MAX_PACK; k++)
        if (k < K && dropped[k] && ((upd >> k) & 1u)) B.ncon_dropped[e0 + k] += dropped[k];
    }
    if (integrate) {
      // MuJoCo's mj_checkPos / mj_checkVel: a non-finite or absurd state resets that env (here: that copy)
      MJB_NOUNROLL
      for (int k = 0; k < K; k++) {
        bool bad = false;
        for (int j = lane; j < dm.nq1; j += 32) { float x = qpos[k * dm.nq1 + j]; bad |= !(fabsf(x) < 1e10f); }
        for (int j = lane; j < dm.nv1; j += 32) { float x = qvel[k * dm.nv1 + j]; bad |= !(fabsf(x) < 1e10f); }
        if (MJB_UNLIKELY(MJB_BALLOT(bad))) {   // warp-uniform
          for (int j = lane; j < dm.nq1; j += 32) qpos[k * dm.nq1 + j] = CF(qpos0)[k * dm.nq1 + j];
          for (int j = lane; j < dm.nv1; j += 32) { qvel[k * dm.nv1 + j] = 0.f; qacc[k * dm.nv1 + j] = 0.f; }
          if (B.nreset && lane == 0 && ((upd >> k) & 1u)) B.nreset[e0 + k] += 1;
        }
      }
      MJB_SYNC();
    }
  }
  MJB_PH(c, PH_INTEGRATE);
  if (ncon >= 0 && (B.ncon || B.contact_geom) && K == 1) {
    const uint32_t* pairs = CU(pair_pack);
    if (B.ncon && lane == 0) B.ncon[e0] = ncon;
    if (B.niter && lane == 0) B.niter[e0] = niter;
    if (B.contact_geom) {
      MJB_NOUNROLL
      for (int k = lane; k < dm.maxcon; k += 32) {
        int g1 = -1, g2 = -1;
        float dist = 0.f;
        if (k < ncon) {
          const float* r = SF(con) + CON_STRIDE * k;
          uint32_t pk = pairs[((const int*)r)[CON_PAIR]];
          g1 = pk & 0xfff; g2 = (pk >> 12) & 0xfff; dist = r[CON_DIST];
        }
        B.contact_geom[((size_t)e0 * dm.maxcon + k) * 2] = g1;
        B.contact_geom[((size_t)e0 * dm.maxcon + k) * 2 + 1] = g2;
        if (B.contact_dist) B.contact_dist[(size_t)e0 * dm.maxcon + k] = dist;
      }
    }
  } else if (ncon >= 0 && (B.ncon || B.contact_geom)) {
    // packed: contact records per real env; a contact belongs to the copy its first geom lives in
    const uint32_t* pairs = CU(pair_pack);
    MJB_NOUNROLL
    for (int k = lane; k < K; k += 32) {
      if (!((upd >> k) & 1u)) continue;
      int n = 0;
      MJB_NOUNROLL
      for (int i = 0; i < ncon; i++) {
        const float* r = SF(con) + CON_STRIDE * i;
        uint32_t pk = pairs[((const int*)r)[CON_PAIR]];
        int g1 = pk & 0xfff, g2 = (pk >> 12) & 0xfff;
        if (g1 / dm.ngeom1 != k) continue;
        if (n < dm.maxcon1 && B.contact_geom) {
          size_t o = (size_t)(e0 + k) * dm.maxcon1 + n;
          B.contact_geom[2 * o] = g1 - k * dm.ngeom1; B.contact_geom[2 * o + 1] = g2 - k * dm.ngeom1;
          if (B.contact_dist) B.contact_dist[o] = r[CON_DIST];
        }
        n++;
      }
      if (B.contact_geom)
        for (int i = n; i < dm.maxcon1; i++) {
          size_t o = (size_t)(e0 + k) * dm.maxcon1 + i;
          B.contact_geom[2 * o] = -1; B.contact_geom[2 * o + 1] = -1;
          if (B.contact_dist) B.contact_dist[o] = 0.f;
        }
      if (B.ncon) B.ncon[e0 + k] = n < dm.maxcon1 ? n : dm.maxcon1;
      if (B.niter) B.niter[e0 + k] = niter;
    }
  }
  // auto-reset pass, lane k < K: the key of copy k's reset draws, read before the stores below overwrite its rows
  const uint32_t ep_k = (auto_pass && lane < K && ((upd >> lane) & 1u)) ? reset_key((uint32_t)(e0 + lane)) : 0u;
  MJB_SYNC();
  auto writes = [&](int k) { return ((upd >> k) & 1u) != 0; };
  uint32_t ended = 0;   // copies whose episode this step ended (auto-reset)
  MJB_NOUNROLL
  for (int i = lane; i < dm.nq; i += 32) {
    int k, j;
    split_copy(i, dm.nq1, K, k, j);
    if (writes(k)) B.qpos[(size_t)(e0 + k) * dm.qpos_stride + j] = qpos[i];
  }
  MJB_NOUNROLL
  for (int i = lane; i < dm.nv; i += 32) {
    int k, j;
    split_copy(i, dm.nv1, K, k, j);
    if (writes(k)) { B.qvel[(size_t)(e0 + k) * dm.qvel_stride + j] = qvel[i]; B.warmstart[(size_t)(e0 + k) * dm.qvel_stride + j] = qacc[i]; }
  }
  MJB_NOUNROLL
  for (int i = lane; i < dm.nu; i += 32) {
    int k, j;
    split_copy(i, dm.nu1, K, k, j);
    if (writes(k)) B.ctrl[(size_t)(e0 + k) * dm.ctrl_stride + j] = ctrl[i];
  }
  MJB_NOUNROLL
  for (int i = lane; i < dm.nsensordata; i += 32) {
    int k, j;
    split_copy(i, dm.ns1, K, k, j);
    if (writes(k)) B.sensordata[(size_t)(e0 + k) * dm.sensor_stride + j] = sens[i];
  }
  MJB_NOUNROLL
  for (int i = lane; i < 4 * dm.nprobe; i += 32) {
    int k, p1;
    probe_slot(i >> 2, k, p1);
    if (writes(k)) B.probe[((size_t)(e0 + k) * dm.np1 + p1) * 4 + (i & 3)] = probe[i];
  }
  MJB_PH(c, PH_STORE);
  if (mode != MODE_STEP && mode != MODE_RESET) return;
  // ---- epilogue: get_observations (mujoco_parent.py:380-392): sensordata(t) ++ qpos(t+h) ++ qvel(t+h)
  MJB_NOUNROLL
  for (int av = 0; av < dm.n_agents; av++) {
    int k, a1;
    split_copy(av, dm.a1, K, k, a1);
    if (!writes(k)) continue;
    float* oa = B.obs + ((size_t)(e0 + k) * dm.a1 + a1) * dm.obs_stride;
    int n = dm.obs_adr[av + 1] - dm.obs_adr[av];
    MJB_NOUNROLL
    for (int i = lane; i < n; i += 32) {
      int e = CI(obs_index)[dm.obs_adr[av] + i], kind = e >> 24, adr = e & 0xffffff;
      oa[i] = kind == 0 ? sens[adr] : (kind == 1 ? qpos[adr] : qvel[adr]);
    }
  }
  MJB_PH(c, PH_EPI_OBS);
  // plugins per real env: its store rows, dynamic actions and step counter are staged in shared memory (the
  // contact Jacobian scratch is dead by now) so that one lane can run the reference-order programme on them
  int* s_si = (int*)SF(J);
  float* s_sf = SF(J) + MJB_MAX_AGENTS * MJB_STORE_I_COUNT;
  float* s_act = s_sf + MJB_MAX_AGENTS * MJB_STORE_F_COUNT;
  int* s_ts = (int*)(s_act + 64);
  double* s_dtab = (double*)(s_ts + 4);   // [a1, t1] agent - target distances of the copy being processed
  MJB_NOUNROLL
  for (int k = 0; k < K; k++) {
    if (!writes(k)) continue;
    const int env = e0 + k, A1 = dm.a1;
    int* gsi = B.store_i + (size_t)env * A1 * dm.store_i32;
    float* gsf = B.store_f + (size_t)env * A1 * dm.store_f32;
    const float* gact = B.actions + (size_t)env * A1 * dm.act_stride;
    MJB_SYNC();
    if (K == 1) {
      for (int r = 0; r < 2; r++) {
        int i = lane + 32 * r;
        if (i < A1 * dm.store_i32) s_si[i] = pre_si[r];
        if (i < A1 * dm.act_stride) s_act[i] = pre_act[r];
      }
      if (lane < A1 * dm.store_f32) s_sf[lane] = pre_sf;
      if (lane == 0) *s_ts = pre_ts;
    } else {
      for (int i = lane; i < A1 * dm.store_i32; i += 32) s_si[i] = gsi[i];
      for (int i = lane; i < A1 * dm.act_stride; i += 32) s_act[i] = gact[i];
      if (lane < A1 * dm.store_f32) s_sf[lane] = gsf[lane];
      if (lane == 0) *s_ts = B.timestep[env];
    }
    // every agent - target distance of this env, one pair per lane (fp64: run_plugins then only looks them up)
    MJB_NOUNROLL
    for (int i = lane; i < A1 * dm.t1; i += 32) {
      const int a = i / dm.t1, t = i - a * dm.t1;
      s_dtab[i] = probe_dist(probe, dm.agent_probe[k * A1 + a], dm.target_probe[k * dm.t1 + t]);
    }
    MJB_SYNC();
    MJB_PH(c, PH_EPI_STAGE);
    const uint32_t ep = auto_pass ? MJB_SHFL(ep_k, k) : 0u;
    bool last_step = false;   // lane 0: this step ended the copy's episode
    if (lane == 0) {
      // auto-reset: the dynamics see a random action (mjb_reset_action) in the one slot each of them reads
      if (auto_pass) {
        MJB_NOUNROLL
        for (int a = 0; a < A1; a++) {
          MJB_NOUNROLL
          for (int p = 0; p < dm.n_dynamics; p++) {
            const DevPlugin& dyn = dm.dynamics[p];
            if (dyn.act_hi > dyn.act_lo)
              s_act[a * dm.act_stride + dyn.act_lo] = reset_action(dm.seed, (uint32_t)env, (uint32_t)a, (uint32_t)dyn.act_lo, ep,
                                                                   dm.dyn_act_low[p], dm.dyn_act_high[p]);
          }
        }
      }
      // up to two agents (every level of the reference): the per-agent accumulators of the programme live in registers
      if (MJB_LIKELY(A1 <= 2))
        last_step = run_plugins<2>(dm, SF(ctrl) + k * dm.nu1, B.obs + (size_t)env * A1 * dm.obs_stride, B.reward + (size_t)env * A1, B.term + (size_t)env * (A1 + 1),
                                   B.trunc + (size_t)env * (A1 + 1), env, k, mode == MODE_RESET, probe, s_si, s_sf, s_act, s_ts, s_dtab, auto_pass);
      else
        last_step = run_plugins<MJB_MAX_AGENTS>(dm, SF(ctrl) + k * dm.nu1, B.obs + (size_t)env * A1 * dm.obs_stride, B.reward + (size_t)env * A1,
                                                B.term + (size_t)env * (A1 + 1), B.trunc + (size_t)env * (A1 + 1), env, k, mode == MODE_RESET, probe, s_si,
                                                s_sf, s_act, s_ts, s_dtab, auto_pass);
    }
    MJB_SYNC();
    MJB_PH(c, PH_EPI_PLUG);
    for (int i = lane; i < A1 * dm.store_i32; i += 32) gsi[i] = s_si[i];
    if (lane < A1 * dm.store_f32) gsf[lane] = s_sf[lane];
    if (lane == 0) B.timestep[env] = *s_ts;
    // (the physics-free step never auto-resets: batch creation refuses skipFrames = 0 with the flag)
    if (EXT && PHYS && mode == MODE_STEP && dm.autoreset && MJB_SHFL((int)last_step, 0)) {
      // the episode's last observation, complete with lane 0's plugin columns (ordered by the MJB_SYNC above)
      ended |= 1u << k;
      const size_t o = (size_t)env * A1 * dm.obs_stride;
      MJB_NOUNROLL
      for (int i = lane; i < A1 * dm.obs_stride; i += 32) dm.final_obs[o + i] = B.obs[o + i];
    }
  }
  MJB_PH(c, PH_EPILOGUE);
  if (MJB_UNLIKELY(ended)) {
    // the reset pass re-reads the rows the step pass stored: the warp barrier orders the lanes' global stores before it
    MJB_SYNC();
    fin = ended;
    goto pass;
  }
}

#if !defined(MJB_HOST_EMU)
#ifndef MJB_MAX_THREADS
#define MJB_MAX_THREADS 512
#endif

// One CTA per SM, `warps` environments in flight per CTA; each warp walks the env index space with a grid-wide
// stride (envs are independent: the warps only meet at the staging of the model image and at the alignment points).
// `active` envs are walked starting at `env_base` (range launches of the host-buffer step) or through `env_ids`
// (the env ids of one level: mjb_set_env_subset).  EXT: the step resets the envs it finishes (MJB_SPEC_AUTORESET) and
// resets start from start states (pool or the caller's rows), a separate instantiation so that batches and launches that
// use neither run exactly the code they ran before.  PRM: the batch has a per-env parameter table (DESIGN §5e); only
// instantiated with EXT, which covers every launch of such a batch.
template <bool PHYS, bool PACKED, bool EXT = false, bool PRM = false>
__global__ void __launch_bounds__(PHYS ? MJB_MAX_THREADS : 512, PHYS ? 1 : 4) k_env(const __grid_constant__ DM dm, const uint32_t* __restrict__ image, const mjb_buffers B,
                      int num_envs, int mode, int skip_frames, const uint8_t* __restrict__ mask,
                      const int* __restrict__ env_ids, int active, int env_base) {
  extern __shared__ __align__(128) uint32_t smem[];
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem);
  uint32_t* img = smem + 4;  // 16 B after the barrier
  const int warps = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    mbar_init(bar, 1);
    mbar_fence_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t bytes = (uint32_t)dm.image_words * 4u;
    mbar_expect_tx(bar, bytes);
    bulk_g2s(img, image, bytes, bar);
  }
  float* scratch = reinterpret_cast<float*>(img + dm.image_words) + (size_t)warp * (dm.env_words + 4 * ((dm.nprobe + 3) & ~3));
  float* probe = scratch + dm.env_words;
  Ctx c{&dm, img, scratch, lane, probe, 0};
#if defined(MJB_PHASE_PROF)
  long long t_last = clock64();
  c.t_last = &t_last;
#endif
  // Lock-step rounds: every env-warp of the CTA takes one env per round, so the warps walk through the (large) step
  // code together and share instruction-cache lines (measured 2x at 65536 envs against a grid-wide work counter).
  // The physics step re-aligns the busy env-warps right after the Newton solve (step_kernel.cuh, forward): they leave
  // it together and stay together through the tail of the step and the head of the next env, so there is no barrier
  // at the round boundary.  The physics-free step has no alignment point inside and re-aligns at the end of each round.
  const int stride = gridDim.x * warps;
  const int pack = PACKED ? dm.pack : 1;
  const int nvirt = (active + pack - 1) / pack;   // virtual envs: `pack` real envs share a warp (active = envs this launch walks)
  const int rounds = (nvirt - blockIdx.x * warps + stride - 1) / stride;
  int env = blockIdx.x * warps + warp;
  for (int r = 0; r < rounds; r++) {
    if (PHYS) {
      int busy = nvirt - (blockIdx.x * warps + r * stride);  // env-warps of this CTA with work in this round
      // (a masked reset lets warps skip their env, so intra-step alignment is off for it)
      c.cta_threads = (mask == nullptr ? 32 : 0) * (busy > warps ? warps : (busy < 0 ? 0 : busy));
    }
    c.img_bar = r == 0 ? bar : nullptr;
    if (env < nvirt) run_env<PHYS, PACKED, EXT, PRM>(c, B, env_ids ? env_ids[env] : env + env_base, num_envs, mode, skip_frames, mask);
    if (r == 0) mbar_wait(bar, 0);   // warps that had nothing to do in the first round (or returned early) have not waited yet
    if (!PHYS) __syncthreads();
    MJB_PH(c, PH_BARRIER);
    env += stride;
  }
}
#endif

}  // namespace mjb
