// mjb_batch.cu — CUDA half of the C-ABI (include/mjb.h): the persistent warp-per-env kernel and the
// batch handle.  sm_100a only; there is no CPU fallback (creation fails without a device).
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/mjb.h"
#include "dev_model_build.h"
#include "env_kernel.cuh"
#include "render_kernel.cuh"
#include "tma_prims.cuh"
#include "lite_kernel.cuh"
#include "mjb_internal.h"
#include "spec_jit.h"

struct mjb_batch {
  mjb::PackedModel packed;   // K real envs per warp (K = 1: plain)
  mjb::DevImage img;
  mjb::DevImage lite;     // skipFrames = 0 only: state-rows-only scratch layout for the step kernel
  bool has_lite = false;
  int lite_warps = 0, lite_grid = 0;
  size_t lite_smem = 0;
  mjb::LiteLayout tile{};   // skipFrames = 0: tile kernel geometry
  int tile_grid = 0;
  size_t tile_smem = 0;
  int* d_lite_tab = nullptr;   // the tile kernel's index tables (lite_tables())
  mjb::DevModel* d_lite_dm = nullptr;   // ... and its DevModel header, padded to 16 bytes
  mjb_buffers B;
  // MODE_STEP of the physics step: the kernel compiled for this batch's shape (spec_jit.h), null: the generic k_env
  cudaKernel_t spec_kern = nullptr;
  std::string spec_why;      // why there is none
  double spec_ms = 0;        // NVRTC compile time of this shape (once per process: later batches find it in the cache)
  int num_envs = 0, device = 0, warps = 0, grid = 0;
  size_t smem_bytes = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t stream2 = nullptr;            // host-buffer step: second half of the envs (copy / compute overlap)
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  uint32_t* d_image = nullptr;
  mjb::DevImage rimg;     // camera rendering: one-env-per-CTA image + camera table (models with cameras only)
  uint32_t *d_rimage = nullptr, *d_rtab = nullptr;
  const int* subset = nullptr;      // the env ids of this handle's level (null: all envs)
  int subset_count = -1;
  int64_t launches = 0;
  bool timing = false;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> events;
  // pinned staging for the host-buffer entry point
  float *h_act = nullptr, *h_obs = nullptr, *h_rew = nullptr;
  uint8_t *h_term = nullptr, *h_trunc = nullptr;
  const void* pin_cache[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
};

namespace {
#define CUDA_TRY(expr)                                                                      \
  do {                                                                                      \
    cudaError_t e_ = (expr);                                                                \
    if (e_ != cudaSuccess) {                                                                \
      mjb::set_error(std::string(#expr) + ": " + cudaGetErrorString(e_));                   \
      return MJB_ERR_CUDA;                                                                  \
    }                                                                                       \
  } while (0)

// `base` / `count` (in envs, multiples of the pack factor) restrict the launch to a contiguous env range
int launch(mjb_batch* b, int mode, int skip_frames, const uint8_t* mask, cudaStream_t stream = nullptr, int base = 0, int count = -1,
           const mjb_buffers* out_buffers = nullptr) {
  if (b->subset && b->subset_count == 0) return MJB_OK;   // no env on this level right now
  if (!stream) stream = b->stream;
  const int active = b->subset ? b->subset_count : (count >= 0 ? count : b->num_envs);
  const mjb_buffers& B = out_buffers ? *out_buffers : b->B;   // the host-buffer step redirects the result arrays
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (b->timing) {
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    CUDA_TRY(cudaEventRecord(e0, stream));
  }
  if (mode == mjb::MODE_STEP && b->has_lite && !b->subset) {
    // no physics in the step: the bandwidth-shaped tile kernel (lite_kernel.cuh) over the contiguous env range
    const int ntiles = (active + b->tile.tile - 1) / b->tile.tile;
    const mjb::LiteLayout& T = b->tile;
    mjb::LiteIssue I{};
    int k = 0;
    auto row = [&](const void* basep, int words, int off_words) {
      if (words <= 0) return;
      I.c[k].base = (const char*)basep; I.c[k].row_bytes = 4u * words; I.c[k].fixed = 0; I.c[k].dst_off = 4u * off_words; k++;
      I.sum_row_bytes += 4u * words;
    };
    auto fixed = [&](const void* basep, int bytes, int off_words) {
      I.c[k].base = (const char*)basep; I.c[k].row_bytes = 0; I.c[k].fixed = bytes; I.c[k].dst_off = 4u * off_words; k++;
      I.first_bytes += bytes;
    };
    row(B.qpos, T.qs, T.o_qpos); row(B.qvel, T.vs, T.o_qvel); row(B.actions, T.as, T.o_act);
    row(B.store_i, T.sis, T.o_si); row(B.store_f, T.sfs, T.o_sf);
    if (T.use_ctrl) row(B.ctrl, T.cs, T.o_ctrl);
    if (T.use_sens) row(B.sensordata, T.ss, T.o_sens);
    if (T.use_probe) row(B.probe, T.ps, T.o_probe);
    fixed(b->d_lite_tab, 4 * T.table_words, T.o_gather);
    fixed(b->d_lite_dm, T.dm_bytes, T.o_dm);
    I.ncopy = k; I.tile = T.tile; I.active = active; I.env_base = base; I.profile = T.profile;
    mjb::k_lite<<<std::min(ntiles, b->tile_grid), LITE_THREADS, b->tile_smem, stream>>>(I, B, T);
  } else if (mode == mjb::MODE_STEP && b->has_lite) {
    // an env-id list (level variants) is not a contiguous range: the warp-per-env form of the same step
    mjb::k_env<false, false><<<b->lite_grid, b->lite_warps * 32, b->lite_smem, stream>>>(b->lite.dm, b->d_image, B, b->num_envs, mode,
                                                                                   skip_frames, mask, b->subset, active, base);
  } else {
    const bool ext = b->img.dm.autoreset || mode == mjb::MODE_RESET_ROWS || (mode == mjb::MODE_RESET && b->img.dm.n_start > 0);
    auto kern = b->img.dm.prm_n > 0 ? (b->img.dm.pack > 1 ? mjb::k_env<true, true, true, true> : mjb::k_env<true, false, true, true>)
              : ext ? (b->img.dm.pack > 1 ? mjb::k_env<true, true, true> : mjb::k_env<true, false, true>)
                    : (b->img.dm.pack > 1 ? mjb::k_env<true, true> : mjb::k_env<true, false>);
    const int pack = b->img.dm.pack;
    const int need = ((active + pack - 1) / pack + b->warps - 1) / b->warps;
    const int grid = std::min(b->grid, std::max(1, need)), env_base = base / pack;
    if (mode == mjb::MODE_STEP && b->spec_kern) {
      // the same instantiation as `kern`, compiled for this shape (the generic kernels give the same bits: spec_jit.h)
      const int* env_ids = b->subset;
      void* args[] = {(void*)&b->img.dm, (void*)&b->d_image, (void*)&B, (void*)&b->num_envs, (void*)&mode, (void*)&skip_frames,
                      (void*)&mask, (void*)&env_ids, (void*)&active, (void*)&env_base};
      CUDA_TRY(cudaLaunchKernel((const void*)b->spec_kern, dim3(grid), dim3(b->warps * 32), args, b->smem_bytes, stream));
    } else {
      kern<<<grid, b->warps * 32, b->smem_bytes, stream>>>(b->img.dm, b->d_image, B, b->num_envs, mode, skip_frames, mask, b->subset,
                                                           active, env_base);
    }
  }
  CUDA_TRY(cudaGetLastError());
  if (b->timing) {
    CUDA_TRY(cudaEventRecord(e1, stream));
    b->events.emplace_back(e0, e1);
  }
  b->launches++;
  return MJB_OK;
}
}  // namespace

extern "C" {

uint32_t mjb_draw_u32(uint64_t seed, uint32_t env, uint32_t agent, uint32_t counter) {
  return mjb::draw_u32(seed, env, agent, counter);
}

float mjb_reset_action(uint64_t seed, uint32_t env, uint32_t agent, uint32_t dim, uint32_t ep, float low, float high) {
  return mjb::reset_action(seed, env, agent, dim, ep, low, high);
}

uint32_t mjb_start_index(uint64_t seed, uint32_t env, uint32_t ep, int32_t n_start) {
  return mjb::start_index(seed, env, ep, n_start);
}

float mjb_param_scale(uint64_t seed, uint32_t env, int32_t family, uint32_t index, uint32_t ep, float lo, float hi) {
  return mjb::param_scale(seed, env, (uint32_t)family, index, ep, lo, hi);
}

int mjb_batch_layout(const mjb_model* m, const mjb_env_spec* spec, int32_t num_envs, mjb_layout* out) {
  if (!m || !spec || !out || num_envs < 1) { mjb::set_error("mjb_batch_layout: bad argument"); return MJB_ERR_ARG; }
  if (const char* e = mjb::param_spec_error(*spec)) { mjb::set_error(std::string("mjb_batch_layout: ") + e); return MJB_ERR_ARG; }
  try {
    mjb::ModelView mv(m->host.blob.data());
    mjb::DevImage img;
    mjb::build_dev_model(mv, *spec, img);
    mjb::fill_layout(img.dm, num_envs, *out);
    return MJB_OK;
  } catch (const std::exception& e) {
    mjb::set_error(e.what());
    return MJB_ERR_LIMIT;
  }
}

int mjb_batch_create(const mjb_model* m, const mjb_env_spec* spec, int32_t num_envs, int32_t device, void* stream,
                     const mjb_buffers* buffers, mjb_batch** out) {
  if (!m || !spec || !buffers || !out || num_envs < 1) { mjb::set_error("mjb_batch_create: bad argument"); return MJB_ERR_ARG; }
  *out = nullptr;
  if (spec->flags & MJB_SPEC_AUTORESET) {
    if (spec->skip_frames == 0) {
      mjb::set_error("mjb_batch_create: MJB_SPEC_AUTORESET needs skip_frames >= 1 (the physics-free step has no forward pass to reset with)");
      return MJB_ERR_ARG;
    }
    if (!spec->final_obs) { mjb::set_error("mjb_batch_create: MJB_SPEC_AUTORESET needs spec.final_obs"); return MJB_ERR_ARG; }
    for (int d = 0; d < spec->act_dim && d < 64; d++)
      if (!(spec->act_low[d] <= spec->act_high[d]) || !std::isfinite(spec->act_low[d]) || !std::isfinite(spec->act_high[d])) {
        mjb::set_error("mjb_batch_create: MJB_SPEC_AUTORESET needs finite act_low <= act_high");
        return MJB_ERR_ARG;
      }
  }
  if (spec->n_start < 0) { mjb::set_error("mjb_batch_create: spec.n_start < 0"); return MJB_ERR_ARG; }
  if (spec->n_start > 0 && (!spec->start_qpos || !spec->start_qvel)) {
    mjb::set_error("mjb_batch_create: spec.n_start > 0 needs spec.start_qpos and spec.start_qvel");
    return MJB_ERR_ARG;
  }
  if (const char* e = mjb::param_spec_error(*spec)) { mjb::set_error(std::string("mjb_batch_create: ") + e); return MJB_ERR_ARG; }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) {
    mjb::set_error("mjb_batch_create: no CUDA device (the step path has no CPU fallback)");
    return MJB_ERR_CUDA;
  }
  mjb_batch* b = new mjb_batch();
  try {
    const int K = mjb::choose_pack(m->host, *spec, num_envs);
    mjb::make_packed(m->host, *spec, K, b->packed);
    mjb::ModelView mv(K > 1 ? b->packed.rep.blob.data() : m->host.blob.data());
    mjb::build_dev_model(mv, b->packed.vspec, b->img, false, K);
    mjb::ModelView mv1(m->host.blob.data());
    if (mv1.ncam > 0) mjb::build_dev_model(mv1, *spec, b->rimg, false, 1);
  } catch (const std::exception& e) {
    mjb::set_error(e.what());
    delete b;
    return MJB_ERR_LIMIT;
  }
  b->B = *buffers;
  b->num_envs = num_envs; b->device = device; b->stream = (cudaStream_t)stream;
  const mjb::DevModel& dm = b->img.dm;
  for (const void* p : {(const void*)b->B.qpos, (const void*)b->B.qvel, (const void*)b->B.ctrl, (const void*)b->B.warmstart,
                        (const void*)b->B.sensordata, (const void*)b->B.probe, (const void*)b->B.actions, (const void*)b->B.obs,
                        (const void*)b->B.reward, (const void*)b->B.term, (const void*)b->B.trunc, (const void*)b->B.timestep,
                        (const void*)b->B.store_i, (const void*)b->B.store_f})
    if (!p) { mjb::set_error("mjb_batch_create: a required buffer is NULL"); delete b; return MJB_ERR_ARG; }
  auto fail = [&](int rc) { mjb_batch_destroy(b); return rc; };
  if (cudaSetDevice(device) != cudaSuccess) { mjb::set_error("cudaSetDevice failed"); return fail(MJB_ERR_CUDA); }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { mjb::set_error("cudaGetDeviceProperties failed"); return fail(MJB_ERR_CUDA); }
  size_t max_smem = prop.sharedMemPerBlockOptin;
  size_t fixed = 16 + (size_t)dm.image_words * 4;
  size_t per_env = ((size_t)dm.env_words + 4 * ((dm.nprobe + 3) & ~3)) * 4;
  size_t cta_budget = std::min(max_smem, prop.sharedMemPerMultiprocessor - 1024);
  int warps = cta_budget > fixed ? (int)((cta_budget - fixed) / per_env) : 0;
  int cap = std::min(MJB_MAX_THREADS / 32, mjb::env_int("MJB_WARPS", MJB_MAX_THREADS / 32));
  if (warps > cap) warps = cap;
  if (warps < 1) { mjb::set_error("model needs more shared memory per environment than one SM has"); return fail(MJB_ERR_LIMIT); }
  // even out the rounds: the fewest warps per CTA that keeps the same number of passes over the envs
  int sms = prop.multiProcessorCount;
  const int nvirt = (num_envs + dm.pack - 1) / dm.pack;
  int rounds = (nvirt + sms * warps - 1) / (sms * warps);
  int even = (nvirt + sms * rounds - 1) / (sms * rounds);
  if (even < warps) warps = even < 1 ? 1 : even;
  b->warps = warps;
  b->grid = (nvirt + warps - 1) / warps;
  if (b->grid > sms) b->grid = sms;
  b->smem_bytes = fixed + per_env * warps;
  // The limit is an attribute of the kernel on the device, shared by every batch: it is only ever raised, so that a batch
  // created later with less shared memory per CTA (one without a parameter table, a smaller model) leaves the launches
  // of the earlier ones valid.
  static std::mutex smem_attr_mu;
  static std::map<int, size_t> smem_attr;
  std::lock_guard<std::mutex> smem_attr_lock(smem_attr_mu);
  if (b->smem_bytes > smem_attr[device] && (cudaFuncSetAttribute(mjb::k_env<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->smem_bytes) != cudaSuccess ||
      cudaFuncSetAttribute(mjb::k_env<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->smem_bytes) != cudaSuccess ||
      cudaFuncSetAttribute(mjb::k_env<true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->smem_bytes) != cudaSuccess ||
      cudaFuncSetAttribute(mjb::k_env<true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->smem_bytes) != cudaSuccess ||
      cudaFuncSetAttribute(mjb::k_env<true, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->smem_bytes) != cudaSuccess ||
      cudaFuncSetAttribute(mjb::k_env<true, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->smem_bytes) != cudaSuccess)) {
    mjb::set_error(std::string("cudaFuncSetAttribute(max dynamic smem) failed: ") + cudaGetErrorString(cudaGetLastError()));
    return fail(MJB_ERR_CUDA);
  }
  smem_attr[device] = std::max(smem_attr[device], b->smem_bytes);
  if (spec->flags & MJB_SPEC_GENERIC) b->spec_why = "MJB_SPEC_GENERIC";
  else if (spec->skip_frames == 0) b->spec_why = "skip_frames = 0 (the physics-free step)";
  else {
    mjb::SpecKernel* sk = mjb::spec_compile(dm);
    b->spec_kern = mjb::spec_kernel(sk, device, b->smem_bytes, b->spec_why);
    b->spec_ms = sk->compile_ms;
  }
  if (spec->skip_frames == 0) {
    try {
      mjb::ModelView mv(m->host.blob.data());
      mjb::build_dev_model(mv, *spec, b->lite, /*lite=*/true);
    } catch (const std::exception& e) { mjb::set_error(e.what()); return fail(MJB_ERR_LIMIT); }
    size_t lite_env = ((size_t)b->lite.dm.env_words + 4 * ((b->lite.dm.nprobe + 3) & ~3)) * 4;
    b->lite_warps = 16;
    b->lite_smem = fixed + lite_env * b->lite_warps;
    int per_sm = 1;
    if (cudaFuncSetAttribute(mjb::k_env<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->lite_smem) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mjb::k_env<false, false>, b->lite_warps * 32, b->lite_smem) != cudaSuccess || per_sm < 1) {
      mjb::set_error("lite step kernel configuration failed");
      return fail(MJB_ERR_CUDA);
    }
    b->lite_grid = std::min((num_envs + b->lite_warps - 1) / b->lite_warps, prop.multiProcessorCount * per_sm);
    b->has_lite = true;
    // tile kernel: the largest tile of 64 / 32 / 16 envs whose rows fit 48 KB, so that several CTAs share an SM and
    // keep enough bytes in flight for HBM
    int tile = std::max(16, mjb::env_int("MJB_LITE_TILE", 64) / 16 * 16);
    for (;;) {
      b->tile = mjb::make_lite_layout(b->lite.dm, tile);
      b->tile.profile = mjb::env_int("MJB_LITE_PROFILE", 0);
      b->tile_smem = 16 + (size_t)b->tile.words * 4;
      if (b->tile_smem <= 48 * 1024 || tile <= 16) break;
      tile /= 2;
    }
    int tile_per_sm = 1;
    if (b->tile_smem > max_smem || cudaFuncSetAttribute(mjb::k_lite, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)b->tile_smem) != cudaSuccess ||
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&tile_per_sm, mjb::k_lite, LITE_THREADS, b->tile_smem) != cudaSuccess || tile_per_sm < 1) {
      mjb::set_error("tile step kernel configuration failed (rows of one env too large for shared memory)");
      return fail(MJB_ERR_CUDA);
    }
    b->tile_grid = prop.multiProcessorCount * tile_per_sm;
    {
      std::vector<int> tab = mjb::lite_tables(b->lite.dm, b->tile, b->img.words.data());
      std::vector<char> hdr(b->tile.dm_bytes, 0);
      memcpy(hdr.data(), &b->lite.dm, sizeof(mjb::DevModel));
      if (cudaMalloc(&b->d_lite_tab, tab.size() * 4) != cudaSuccess ||
          cudaMemcpy(b->d_lite_tab, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice) != cudaSuccess ||
          cudaMalloc(&b->d_lite_dm, hdr.size()) != cudaSuccess ||
          cudaMemcpy(b->d_lite_dm, hdr.data(), hdr.size(), cudaMemcpyHostToDevice) != cudaSuccess) {
        mjb::set_error("tile kernel table upload failed");
        return fail(MJB_ERR_CUDA);
      }
    }
  }
  if (cudaMalloc(&b->d_image, (size_t)dm.image_words * 4) != cudaSuccess ||
      cudaMemcpy(b->d_image, b->img.words.data(), (size_t)dm.image_words * 4, cudaMemcpyHostToDevice) != cudaSuccess) {
    mjb::set_error("device image upload failed");
    return fail(MJB_ERR_CUDA);
  }
  if (cudaStreamCreateWithFlags(&b->stream2, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&b->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&b->ev_join, cudaEventDisableTiming) != cudaSuccess) {
    mjb::set_error("mjb_batch_create: stream / event creation failed");
    return fail(MJB_ERR_CUDA);
  }
  const int A = dm.a1;
  if (cudaMallocHost(&b->h_act, sizeof(float) * (size_t)num_envs * A * dm.act_stride + 16) != cudaSuccess ||
      cudaMallocHost(&b->h_obs, sizeof(float) * (size_t)num_envs * A * dm.obs_stride + 16) != cudaSuccess ||
      cudaMallocHost(&b->h_rew, sizeof(float) * (size_t)num_envs * A + 16) != cudaSuccess ||
      cudaMallocHost(&b->h_term, (size_t)num_envs * (A + 1) + 16) != cudaSuccess ||
      cudaMallocHost(&b->h_trunc, (size_t)num_envs * (A + 1) + 16) != cudaSuccess) {
    mjb::set_error("pinned staging allocation failed");
    return fail(MJB_ERR_CUDA);
  }
  *out = b;
  return MJB_OK;
}

void mjb_batch_destroy(mjb_batch* b) {
  if (!b) return;
  for (auto& ev : b->events) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
  if (b->d_image) cudaFree(b->d_image);
  if (b->stream2) cudaStreamDestroy(b->stream2);
  for (cudaEvent_t e : {b->ev_fork, b->ev_join}) if (e) cudaEventDestroy(e);
  if (b->d_rimage) cudaFree(b->d_rimage);
  if (b->d_rtab) cudaFree(b->d_rtab);
  if (b->d_lite_tab) cudaFree(b->d_lite_tab);
  if (b->d_lite_dm) cudaFree(b->d_lite_dm);
  if (b->h_act) cudaFreeHost(b->h_act);
  if (b->h_obs) cudaFreeHost(b->h_obs);
  if (b->h_rew) cudaFreeHost(b->h_rew);
  if (b->h_term) cudaFreeHost(b->h_term);
  if (b->h_trunc) cudaFreeHost(b->h_trunc);
  delete b;
}

int mjb_reset(mjb_batch* b, const uint8_t* mask_dev) {
  if (!b) { mjb::set_error("mjb_reset: null batch"); return MJB_ERR_ARG; }
  return launch(b, mjb::MODE_RESET, 0, mask_dev);
}
int mjb_reset_rows(mjb_batch* b, const uint8_t* mask_dev) {
  if (!b) { mjb::set_error("mjb_reset_rows: null batch"); return MJB_ERR_ARG; }
  return launch(b, mjb::MODE_RESET_ROWS, 0, mask_dev);
}
int mjb_step(mjb_batch* b) {
  if (!b) { mjb::set_error("mjb_step: null batch"); return MJB_ERR_ARG; }
  return launch(b, mjb::MODE_STEP, b->img.dm.skip_frames, nullptr);
}
int mjb_physics(mjb_batch* b, int32_t skip_frames) {
  if (!b || skip_frames < 0) { mjb::set_error("mjb_physics: bad argument"); return MJB_ERR_ARG; }
  return launch(b, mjb::MODE_PHYSICS, skip_frames, nullptr);
}
int mjb_forward(mjb_batch* b) {
  if (!b) { mjb::set_error("mjb_forward: null batch"); return MJB_ERR_ARG; }
  return launch(b, mjb::MODE_FORWARD, 0, nullptr);
}
int mjb_sync(mjb_batch* b) {
  if (!b) { mjb::set_error("mjb_sync: null batch"); return MJB_ERR_ARG; }
  CUDA_TRY(cudaStreamSynchronize(b->stream));
  return MJB_OK;
}

int mjb_step_host(mjb_batch* b, const float* actions, float* obs, float* reward, uint8_t* term, uint8_t* trunc) {
  if (!b || !actions || !obs || !reward || !term || !trunc) { mjb::set_error("mjb_step_host: null argument"); return MJB_ERR_ARG; }
  if (b->img.dm.autoreset) { mjb::set_error("mjb_step_host: not available on a batch created with MJB_SPEC_AUTORESET"); return MJB_ERR_ARG; }
  const mjb::DevModel& dm = b->img.dm;
  const size_t N = b->num_envs, A = dm.a1;   // agents of ONE real env (the image may pack several envs per warp)
  const size_t nb_act = sizeof(float) * N * A * dm.act_stride, nb_obs = sizeof(float) * N * A * dm.obs_stride;
  const size_t nb_rew = sizeof(float) * N * A, nb_flag = N * (A + 1);
  // page-locked caller buffers are copied directly; pageable ones go through the pinned staging area
  auto pinned = [&](const void* p) {
    if (p == b->pin_cache[0] || p == b->pin_cache[1] || p == b->pin_cache[2] || p == b->pin_cache[3] || p == b->pin_cache[4]) return true;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
  };
  bool direct = pinned(actions) && pinned(obs) && pinned(reward) && pinned(term) && pinned(trunc);
  if (direct) {
    b->pin_cache[0] = actions; b->pin_cache[1] = obs; b->pin_cache[2] = reward; b->pin_cache[3] = term; b->pin_cache[4] = trunc;
  }
  // Page-locked result arrays are written by the kernel itself (zero-copy: pinned host memory is device-addressable,
  // the stores are posted PCIe writes that overlap the rest of the step), so no device-to-host copy follows the
  // kernel.  The actions still go up by copy engine, in two halves on two streams so that the second half's upload
  // overlaps the first half's compute.  Same results (envs are independent).
  if (direct && !b->subset) {
    mjb_buffers Bh = b->B;
    void *d_obs = nullptr, *d_rew = nullptr, *d_term = nullptr, *d_trunc = nullptr;
    if (cudaHostGetDevicePointer(&d_obs, obs, 0) == cudaSuccess && cudaHostGetDevicePointer(&d_rew, reward, 0) == cudaSuccess &&
        cudaHostGetDevicePointer(&d_term, term, 0) == cudaSuccess && cudaHostGetDevicePointer(&d_trunc, trunc, 0) == cudaSuccess) {
      Bh.obs = (float*)d_obs; Bh.reward = (float*)d_rew; Bh.term = (uint8_t*)d_term; Bh.trunc = (uint8_t*)d_trunc;
      const size_t act_row = sizeof(float) * A * dm.act_stride;
      const int pack = dm.pack;
      const int half = (int)((N / 2 + pack - 1) / pack * pack);
      if (N >= (size_t)(4 * b->warps) && half > 0 && (size_t)half < N) {
        CUDA_TRY(cudaEventRecord(b->ev_fork, b->stream));
        CUDA_TRY(cudaStreamWaitEvent(b->stream2, b->ev_fork, 0));
        CUDA_TRY(cudaMemcpyAsync(b->B.actions, actions, act_row * half, cudaMemcpyHostToDevice, b->stream));
        CUDA_TRY(cudaMemcpyAsync((char*)b->B.actions + act_row * half, (const char*)actions + act_row * half, act_row * (N - half),
                                 cudaMemcpyHostToDevice, b->stream2));
        int rc = launch(b, mjb::MODE_STEP, dm.skip_frames, nullptr, b->stream, 0, half, &Bh);
        if (rc != MJB_OK) return rc;
        rc = launch(b, mjb::MODE_STEP, dm.skip_frames, nullptr, b->stream2, half, (int)N - half, &Bh);
        if (rc != MJB_OK) return rc;
        CUDA_TRY(cudaEventRecord(b->ev_join, b->stream2));
        CUDA_TRY(cudaStreamWaitEvent(b->stream, b->ev_join, 0));
      } else {
        CUDA_TRY(cudaMemcpyAsync(b->B.actions, actions, nb_act, cudaMemcpyHostToDevice, b->stream));
        int rc = launch(b, mjb::MODE_STEP, dm.skip_frames, nullptr, b->stream, 0, -1, &Bh);
        if (rc != MJB_OK) return rc;
      }
      CUDA_TRY(cudaStreamSynchronize(b->stream));
      return MJB_OK;
    }
    // not device-addressable after all (e.g. an address remembered as page-locked was freed and re-used by pageable
    // memory): forget what was remembered and take the staged path for this call
    cudaGetLastError();
    for (auto& p : b->pin_cache) p = nullptr;
    direct = false;
  }
  // Pageable arrays, a level subset, or arrays not device-addressable: upload the actions, step, copy the results back
  // (page-locked arrays directly, others through the pinned staging area).
  if (!direct) memcpy(b->h_act, actions, nb_act);
  CUDA_TRY(cudaMemcpyAsync(b->B.actions, direct ? actions : b->h_act, nb_act, cudaMemcpyHostToDevice, b->stream));
  int rc = launch(b, mjb::MODE_STEP, dm.skip_frames, nullptr);
  if (rc != MJB_OK) return rc;
  CUDA_TRY(cudaMemcpyAsync(direct ? obs : b->h_obs, b->B.obs, nb_obs, cudaMemcpyDeviceToHost, b->stream));
  CUDA_TRY(cudaMemcpyAsync(direct ? reward : b->h_rew, b->B.reward, nb_rew, cudaMemcpyDeviceToHost, b->stream));
  CUDA_TRY(cudaMemcpyAsync(direct ? term : b->h_term, b->B.term, nb_flag, cudaMemcpyDeviceToHost, b->stream));
  CUDA_TRY(cudaMemcpyAsync(direct ? trunc : b->h_trunc, b->B.trunc, nb_flag, cudaMemcpyDeviceToHost, b->stream));
  CUDA_TRY(cudaStreamSynchronize(b->stream));
  if (!direct) {
    memcpy(obs, b->h_obs, nb_obs);
    memcpy(reward, b->h_rew, nb_rew);
    memcpy(term, b->h_term, nb_flag);
    memcpy(trunc, b->h_trunc, nb_flag);
  }
  return MJB_OK;
}

int64_t mjb_launch_count(const mjb_batch* b) { return b ? b->launches : 0; }

int mjb_set_timing(mjb_batch* b, int32_t enable) {
  if (!b) { mjb::set_error("mjb_set_timing: null batch"); return MJB_ERR_ARG; }
  b->timing = enable != 0;
  return MJB_OK;
}

int mjb_kernel_time_ms(mjb_batch* b, double* total_ms, int64_t* launches) {
  if (!b || !total_ms || !launches) { mjb::set_error("mjb_kernel_time_ms: null argument"); return MJB_ERR_ARG; }
  CUDA_TRY(cudaStreamSynchronize(b->stream));
  double tot = 0;
  for (auto& ev : b->events) {
    float ms = 0;
    CUDA_TRY(cudaEventElapsedTime(&ms, ev.first, ev.second));
    tot += ms;
    cudaEventDestroy(ev.first); cudaEventDestroy(ev.second);
  }
  *total_ms = tot; *launches = (int64_t)b->events.size();
  b->events.clear();
  return MJB_OK;
}

int mjb_render(mjb_batch* b, const int32_t* cam_ids, int32_t ncams, int32_t width, int32_t height, uint8_t* rgb_dev) {
  if (!b || !cam_ids || !rgb_dev) { mjb::set_error("mjb_render: null argument"); return MJB_ERR_ARG; }
  mjb_render_args a{};
  a.cam_ids = cam_ids; a.ncams = ncams; a.width = width; a.height = height; a.rgb = rgb_dev;
  return mjb_render_ex(b, &a);
}

int mjb_render_ex(mjb_batch* b, const mjb_render_args* args) {
  if (!b || !args || !args->cam_ids) { mjb::set_error("mjb_render: null argument"); return MJB_ERR_ARG; }
  const mjb_render_args& a = *args;
  const int32_t ncams = a.ncams, width = a.width, height = a.height;
  if (!a.rgb && !a.depth && !a.segmentation) { mjb::set_error("mjb_render_ex: rgb, depth and segmentation are all NULL"); return MJB_ERR_ARG; }
  const float* qpos = (a.qpos == nullptr || a.qpos == b->B.qpos) ? b->B.qpos : a.qpos;
  if (qpos != b->B.qpos && (qpos != b->img.dm.final_qpos || !b->img.dm.final_qpos)) {
    mjb::set_error(b->img.dm.final_qpos ? "mjb_render_ex: qpos must be NULL, buffers.qpos or the batch's spec.final_qpos"
                                        : "mjb_render_ex: qpos must be NULL or buffers.qpos (the batch has no spec.final_qpos)");
    return MJB_ERR_ARG;
  }
  const mjb::RenderHdr& rh = b->rimg.rhdr;
  if (rh.ncam == 0) { mjb::set_error("mjb_render: the model has no <camera>"); return MJB_ERR_ARG; }
  if (ncams < 1 || ncams > RENDER_MAX_CAMS || width < 1 || height < 1 || width > 4096 || height > 4096) {
    mjb::set_error("mjb_render: 1.." + std::to_string(RENDER_MAX_CAMS) + " cameras, 1..4096 pixels per side");
    return MJB_ERR_ARG;
  }
  mjb::RenderCams cams{};
  cams.n = ncams;
  for (int k = 0; k < ncams; k++) {
    if (a.cam_ids[k] < 0 || a.cam_ids[k] >= rh.ncam) { mjb::set_error("mjb_render: camera id out of range"); return MJB_ERR_ARG; }
    if (b->rimg.render[rh.off_cam + a.cam_ids[k] * mjb::CAM_STRIDE + mjb::CAM_MODE] != 0) {
      mjb::set_error("mjb_render: only mode=\"fixed\" cameras can be rendered");
      return MJB_ERR_ARG;
    }
    cams.id[k] = a.cam_ids[k];
  }
  CUDA_TRY(cudaSetDevice(b->device));
  const mjb::DevModel& dm = b->rimg.dm;
  const size_t smem = ((size_t)dm.image_words + dm.env_words + rh.words + (size_t)dm.ngeom * mjb::GL_STRIDE + 12 * RENDER_MAX_CAMS) * 4 +
                      (size_t)RENDER_TILE_BATCH * ((dm.ngeom + 2) & ~1) * 2;
  if (!b->d_rimage) {
    CUDA_TRY(cudaMalloc(&b->d_rimage, b->rimg.words.size() * 4));
    CUDA_TRY(cudaMalloc(&b->d_rtab, b->rimg.render.size() * 4));
    CUDA_TRY(cudaMemcpy(b->d_rimage, b->rimg.words.data(), b->rimg.words.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(b->d_rtab, b->rimg.render.data(), b->rimg.render.size() * 4, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaFuncSetAttribute(mjb::k_render<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CUDA_TRY(cudaFuncSetAttribute(mjb::k_render<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  }
  int sms = 148;
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, b->device);
  const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(8, (200 * 1024) / (smem + 1024)));
  const int grid = std::min(b->num_envs, sms * per_sm);
  // depth or segmentation requested: the instantiation that keeps each pixel's hit (the colour-only one runs without it)
  auto kern = (a.depth || a.segmentation) ? mjb::k_render<true> : mjb::k_render<false>;
  kern<<<grid, 256, smem, b->stream>>>(dm, b->d_rimage, rh, b->d_rtab, qpos, a.mask, b->num_envs, cams, width, height, a.rgb, a.depth,
                                       a.segmentation);
  CUDA_TRY(cudaGetLastError());
  b->launches++;
  return MJB_OK;
}

int mjb_set_env_subset(mjb_batch* b, const int32_t* env_ids_dev, int32_t count) {
  if (!b) { mjb::set_error("mjb_set_env_subset: null batch"); return MJB_ERR_ARG; }
  if (b->img.dm.autoreset) {
    mjb::set_error("mjb_set_env_subset: level variants cannot auto-reset (a reset draws the env's level on the host)");
    return MJB_ERR_ARG;
  }
  if (!env_ids_dev) { b->subset = nullptr; b->subset_count = -1; return MJB_OK; }
  if (count < 0 || count > b->num_envs) { mjb::set_error("mjb_set_env_subset: count out of range"); return MJB_ERR_ARG; }
  if (b->img.dm.pack != 1) {
    mjb::set_error("mjb_set_env_subset: the batch packs several envs per warp; create it with MJB_SPEC_NO_PACK");
    return MJB_ERR_ARG;
  }
  b->subset = env_ids_dev; b->subset_count = count;
  return MJB_OK;
}

/* debug build (-DMJB_PHASE_PROF) only: read (and clear) the per-phase cycle counters; returns the number of phases, 0 in
   the product build */
int mjb_phase_cycles(uint64_t* out, int32_t n) {
#if defined(MJB_PHASE_PROF)
  unsigned long long h[32];
  if (cudaMemcpyFromSymbol(h, mjb::g_phase_cycles, sizeof(h)) != cudaSuccess) return -1;
  for (int i = 0; i < n && i < 32; i++) out[i] = h[i];
  memset(h, 0, sizeof(h));
  cudaMemcpyToSymbol(mjb::g_phase_cycles, h, sizeof(h));
  return mjb::PH_COUNT;
#else
  (void)out; (void)n;
  return 0;
#endif
}

int mjb_batch_spec_info(const mjb_batch* b, int32_t* specialised, double* compile_ms, char* reason, int32_t reason_len) {
  if (!b) return MJB_ERR_ARG;
  if (specialised) *specialised = b->spec_kern ? 1 : 0;
  if (compile_ms) *compile_ms = b->spec_ms;
  if (reason && reason_len > 0) snprintf(reason, (size_t)reason_len, "%s", b->spec_why.c_str());
  return MJB_OK;
}

int mjb_spec_compile(const mjb_model* m, const mjb_env_spec* spec, int32_t num_envs, double* compile_ms, void* cubin, int64_t* cubin_bytes) {
  if (!m || !spec || num_envs < 1 || !cubin_bytes) { mjb::set_error("mjb_spec_compile: bad argument"); return MJB_ERR_ARG; }
  mjb::DevImage img;
  try {
    mjb::PackedModel packed;
    const int K = mjb::choose_pack(m->host, *spec, num_envs);
    mjb::make_packed(m->host, *spec, K, packed);
    mjb::ModelView mv(K > 1 ? packed.rep.blob.data() : m->host.blob.data());
    mjb::build_dev_model(mv, packed.vspec, img, false, K);
  } catch (const std::exception& e) {
    mjb::set_error(e.what());
    return MJB_ERR_LIMIT;
  }
  const mjb::SpecKernel* sk = mjb::spec_compile(img.dm);
  if (!sk->why.empty()) { mjb::set_error("mjb_spec_compile: " + sk->why); return MJB_ERR_CUDA; }
  if (compile_ms) *compile_ms = sk->compile_ms;
  if (cubin && *cubin_bytes >= (int64_t)sk->cubin.size()) memcpy(cubin, sk->cubin.data(), sk->cubin.size());
  *cubin_bytes = (int64_t)sk->cubin.size();
  return MJB_OK;
}

/* query of the launch geometry, for bench / docs */
int mjb_batch_geometry(const mjb_batch* b, int32_t* grid, int32_t* warps_per_cta, int64_t* smem_bytes) {
  if (!b) return MJB_ERR_ARG;
  if (grid) *grid = b->grid;
  if (warps_per_cta) *warps_per_cta = b->warps;
  if (smem_bytes) *smem_bytes = (int64_t)b->smem_bytes;
  return MJB_OK;
}

}  // extern "C"
