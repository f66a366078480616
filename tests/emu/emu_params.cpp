// emu_params.cpp — host build of the device step code on the SIMT emulator, with the kernels a batch with a per-env
// parameter table runs (test tooling only; tests/test_model_params.py).  Same entry point as emu_lib.cpp's emu_run: a
// spec with `params` set runs run_env<..., PRM = true> (the instantiation k_env<..., true, true> of mjb_batch.cu), any
// other spec the plain one.
#define MJB_HOST_EMU 1
#include <cstring>
#include <string>
#include <vector>

#include "../../mujoco_rl_environment_wrapper_b200/csrc/dev_model_build.h"
#include "../../mujoco_rl_environment_wrapper_b200/csrc/env_kernel.cuh"

static std::string g_err;

extern "C" {

const char* emu_last_error() { return g_err.c_str(); }

// the refusal mjb_batch_create gives for the spec's parameter-table fields ("" = accepted)
const char* emu_param_spec_error(const mjb_env_spec* spec) {
  const char* e = mjb::param_spec_error(*spec);
  return e ? e : "";
}

int emu_run(const void* blob, const mjb_env_spec* spec, int num_envs, const mjb_buffers* B, int mode, int skip_frames,
            const uint8_t* mask, int reverse) {
  try {
    mjb::HostModel host;
    {
      const mjb_blob_header* h = (const mjb_blob_header*)blob;
      const mjb_blob_field* f = (const mjb_blob_field*)((const char*)blob + sizeof(mjb_blob_header));
      for (int i = 0; i < h->nfields; i++) {
        std::string name(f[i].name);
        const char* p = (const char*)blob + f[i].offset;
        if (f[i].dtype == MJB_DTYPE_I32) host.I(name).assign((const int32_t*)p, (const int32_t*)p + f[i].count);
        else host.F(name).assign((const double*)p, (const double*)p + f[i].count);
      }
      host.pack();
    }
    const int K = mjb::choose_pack(host, *spec, num_envs);
    mjb::PackedModel packed;
    mjb::make_packed(host, *spec, K, packed);
    mjb::ModelView mv(K > 1 ? (const void*)packed.rep.blob.data() : blob);
    mjb::DevImage img;
    mjb::build_dev_model(mv, packed.vspec, img, false, K);
    std::vector<float> scratch(img.dm.env_words + 64, 0.f), probe(4 * img.dm.nprobe + 4, 0.f);
    const int nvirt = (num_envs + K - 1) / K;
    for (int env = 0; env < nvirt; env++) {
      simt::run_warp([&]() {
        mjb::Ctx c{&img.dm, img.words.data(), scratch.data(), simt::lane(), probe.data(), 0};
        if (img.dm.prm_n > 0) mjb::run_env<true, true, true, true>(c, *B, env, num_envs, mode, skip_frames, mask);
        else mjb::run_env<true, true>(c, *B, env, num_envs, mode, skip_frames, mask);
      }, reverse != 0);
    }
    return 0;
  } catch (const std::exception& e) { g_err = e.what(); return -1; }
}

}  // extern "C"
