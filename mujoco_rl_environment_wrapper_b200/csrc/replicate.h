// replicate.h — K-fold replication of a compiled model (host side).
//
// Small models leave most of a warp idle: an ant has 14 dofs / 13 moving bodies for 32 lanes.  Because the
// step kernel already handles several independent kinematic trees in one env at no extra cost (every phase
// is lane-parallel over bodies / dofs / pairs and the solver factors per tree block), K real environments
// can share one warp by presenting them to the kernel as ONE virtual environment whose model is the original
// repeated K times (separate trees, no collision pairs across copies).  This file builds that virtual model
// from the compiled one by replicating every per-object array and remapping the indices it holds.  The HBM
// buffers keep their per-real-env layout; env_kernel.cuh maps (virtual env, copy) -> real env on load/store.
#pragma once
#include <string>
#include <vector>

#include "host_model.h"

namespace mjb {

inline void replicate_model(const HostModel& src, int K, HostModel& dst) {
  const int nq = src.get_int("nq"), nv = src.get_int("nv"), nu = src.get_int("nu"), nbody = src.get_int("nbody"),
            njnt = src.get_int("njnt"), ngeom = src.get_int("ngeom"), nsite = src.get_int("nsite"),
            nsensor = src.get_int("nsensor"), nsensordata = src.get_int("nsensordata"), npair = src.get_int("npair"),
            ntree = src.get_int("ntree");
  (void)nu; (void)npair;
  const std::vector<int32_t>& sensor_objtype = src.Iv("sensor_objtype");
  auto bmap = [&](int b, int c) { return b <= 0 ? b : 1 + c * (nbody - 1) + (b - 1); };
  auto off = [](int v, int add) { return v < 0 ? v : v + add; };
  dst = HostModel();
  for (const std::string& name : src.order) {
    const bool is_int = src.i32.count(name) > 0;
    // scalars
    if (name == "nq" || name == "nv" || name == "nu" || name == "njnt" || name == "ngeom" || name == "nsite" ||
        name == "nsensor" || name == "nsensordata" || name == "npair" || name == "ntree" || name == "ncam") {
      dst.set_int(name, src.get_int(name) * K);
      continue;
    }
    if (name == "nbody") { dst.set_int(name, 1 + K * (nbody - 1)); continue; }
    if (name == "maxdepth" || name.rfind("opt_", 0) == 0) {
      if (is_int) dst.I(name) = src.Iv(name); else dst.F(name) = src.Fv(name);
      continue;
    }
    const bool body = name.rfind("body_", 0) == 0;
    if (is_int) {
      const std::vector<int32_t>& v = src.Iv(name);
      std::vector<int32_t>& o = dst.I(name);
      size_t count = body ? (size_t)nbody : 0;
      size_t stride = body && count ? v.size() / count : 0;
      if (body) o.insert(o.end(), v.begin(), v.begin() + stride);  // world body once
      for (int c = 0; c < K; c++) {
        size_t i0 = body ? stride : 0;
        for (size_t i = i0; i < v.size(); i++) {
          int x = v[i];
          if (name == "body_parentid" || name == "body_rootid" || name == "body_weldid" || name == "jnt_bodyid" ||
              name == "dof_bodyid" || name == "geom_bodyid" || name == "site_bodyid" || name == "cam_bodyid") x = bmap(x, c);
          else if (name == "body_jntadr" || name == "dof_jntid" || name == "actuator_trnid") x = off(x, c * njnt);
          else if (name == "body_dofadr" || name == "jnt_dofadr" || name == "dof_parentid") x = off(x, c * nv);
          else if (name == "body_geomadr" || name == "pair_geom1" || name == "pair_geom2") x = off(x, c * ngeom);
          else if (name == "body_treeid") x = off(x, c * ntree);
          else if (name == "jnt_qposadr") x = off(x, c * nq);
          else if (name == "sensor_objid") {   // numbered in its object type's id space
            const int ot = sensor_objtype[(i - i0) % nsensor];
            x = ot == MJB_OBJ_BODY || ot == MJB_OBJ_XBODY ? bmap(x, c)
                : off(x, c * (ot == MJB_OBJ_GEOM ? ngeom : ot == MJB_OBJ_JOINT ? njnt : nsite));
          }
          else if (name == "sensor_adr") x = off(x, c * nsensordata);
          o.push_back(x);
        }
      }
    } else {
      const std::vector<double>& v = src.Fv(name);
      std::vector<double>& o = dst.F(name);
      size_t count = body ? (size_t)nbody : 0;
      size_t stride = body && count ? v.size() / count : 0;
      if (body) o.insert(o.end(), v.begin(), v.begin() + stride);
      for (int c = 0; c < K; c++) o.insert(o.end(), v.begin() + (body ? stride : 0), v.end());
    }
  }
  dst.pack();
}

}  // namespace mjb
