// mjb_model.cpp — host-only half of the C-ABI (include/mjb.h): MJCF -> model handle,
// dims, blob access and name lookups.  No CUDA in this translation unit.
#include <algorithm>
#include <cstring>
#include <string>

#include "../../include/mjb.h"
#include "host_model.h"
#include "mjb_internal.h"

namespace mjb {
thread_local std::string g_last_error;
void set_error(const std::string& s) { g_last_error = s; }
}  // namespace mjb

extern "C" {

const char* mjb_last_error(void) { return mjb::g_last_error.c_str(); }
const char* mjb_version(void) { return "mjb 0.1 (sm_100a)"; }

int mjb_model_create(const char* mjcf_text, mjb_model** out) {
  if (!mjcf_text || !out) { mjb::set_error("mjb_model_create: null argument"); return MJB_ERR_ARG; }
  *out = nullptr;
  try {
    mjb_model* m = new mjb_model();
    try {
      mjb::compile_mjcf(mjcf_text, m->host);
    } catch (...) {
      delete m;
      throw;
    }
    *out = m;
    return MJB_OK;
  } catch (const std::exception& e) {
    mjb::set_error(e.what());
    return MJB_ERR_PARSE;
  }
}

void mjb_model_destroy(mjb_model* m) { delete m; }

int mjb_model_dims(const mjb_model* m, mjb_dims* out) {
  if (!m || !out) { mjb::set_error("mjb_model_dims: null argument"); return MJB_ERR_ARG; }
  try {
    const mjb::HostModel& h = m->host;
    memset(out, 0, sizeof(*out));
    out->nq = h.get_int("nq"); out->nv = h.get_int("nv"); out->nu = h.get_int("nu");
    out->nbody = h.get_int("nbody"); out->njnt = h.get_int("njnt"); out->ngeom = h.get_int("ngeom");
    out->nsite = h.get_int("nsite"); out->nsensor = h.get_int("nsensor");
    out->nsensordata = h.get_int("nsensordata"); out->npair = h.get_int("npair");
    out->integrator = h.get_int("opt_integrator"); out->ncam = h.get_int("ncam");
    out->timestep = h.Fv("opt_timestep")[0];
    return MJB_OK;
  } catch (const std::exception& e) {
    mjb::set_error(e.what());
    return MJB_ERR_ARG;
  }
}

const void* mjb_model_blob(const mjb_model* m, int64_t* nbytes) {
  if (!m) return nullptr;
  if (nbytes) *nbytes = (int64_t)m->host.blob.size();
  return m->host.blob.data();
}

int mjb_name2id(const mjb_model* m, int objtype, const char* name) {
  if (!m || !name || !*name) return -1;
  auto it = m->host.names.find(objtype);
  if (it == m->host.names.end()) return -1;
  for (size_t i = 0; i < it->second.size(); i++)
    if (it->second[i] == name) return (int)i;
  return -1;
}

int mjb_param_layout(const mjb_model* m, mjb_param_offsets* out) {
  if (!m || !out) { mjb::set_error("mjb_param_layout: null argument"); return MJB_ERR_ARG; }
  const mjb::HostModel& h = m->host;
  const int nbody = h.get_int("nbody"), ngeom = h.get_int("ngeom"), nu = h.get_int("nu"), nv = h.get_int("nv");
  out->body_mass = 0;
  out->body_inertia = nbody;
  out->geom_friction = 4 * nbody;
  out->actuator_gear = 4 * nbody + ngeom;
  out->dof_damping = 4 * nbody + ngeom + nu;
  out->n_params = 4 * nbody + ngeom + nu + nv;
  return MJB_OK;
}

int mjb_model_set_field(mjb_model* m, const char* name, const double* values, int32_t count) {
  if (!m || !name || (!values && count > 0)) { mjb::set_error("mjb_model_set_field: null argument"); return MJB_ERR_ARG; }
  auto it = m->host.f64.find(name);
  if (it == m->host.f64.end()) {
    mjb::set_error(std::string("mjb_model_set_field: no fp64 field named '") + name + "'");
    return MJB_ERR_ARG;
  }
  if (count != (int32_t)it->second.size()) {
    mjb::set_error(std::string("mjb_model_set_field: '") + name + "' has " + std::to_string(it->second.size()) + " values, got " +
                   std::to_string(count));
    return MJB_ERR_ARG;
  }
  it->second.assign(values, values + count);
  if (std::string(name) == "geom_friction") {
    // MuJoCo mixes friction per contact from the geoms' values; here the compiler stores the mix per collision pair
    // (mjcf_compile.cpp): mix it again so that the edit reaches the contacts as it does in MuJoCo
    const std::vector<int32_t>&g1 = m->host.Iv("pair_geom1"), &g2 = m->host.Iv("pair_geom2");
    std::vector<double>& pf = m->host.f64["pair_friction"];
    for (size_t k = 0; k < g1.size(); k++)
      for (int i = 0; i < 3; i++) pf[3 * k + i] = std::max(it->second[3 * g1[k] + i], it->second[3 * g2[k] + i]);
  }
  m->host.pack();
  return MJB_OK;
}

const char* mjb_id2name(const mjb_model* m, int objtype, int id) {
  if (!m) return nullptr;
  auto it = m->host.names.find(objtype);
  if (it == m->host.names.end() || id < 0 || id >= (int)it->second.size()) return nullptr;
  return it->second[id].c_str();
}

}  // extern "C"
