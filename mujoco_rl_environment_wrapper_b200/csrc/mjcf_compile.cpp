// mjcf_compile.cpp — MJCF text -> compiled model (HostModel / packed blob).
//
// Replaces the reference's `mj.MjModel.from_xml_path` (MuJoCo_Gym/mujoco_parent.py:126)
// for the MJCF subset used by the reference's levels (SURVEY.md A.2):
//   <compiler angle eulerseq>, <option timestep integrator gravity iterations tolerance impratio>,
//   one unnamed <default> (joint / geom / site / motor), <worldbody> with nested <body>,
//   <geom plane|sphere|capsule|box>, <joint free|hinge|slide>, <site>, <sensor touch|
//   accelerometer|rangefinder|framexaxis|frameyaxis|framezaxis|gyro|velocimeter|jointpos|jointvel|
//   framepos|framequat|framelinvel|frameangvel>, <actuator><motor>.
// The derived constants follow MuJoCo's documented compiler behaviour (inertia from
// geoms, fromto -> pos/quat/size, degrees -> radians, qpos0, bounding radii, static
// collision filters, body/dof invweight0).  MuJoCo's source is not part of the
// reference tree, so those rules are restated from its public documentation.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <sstream>

#include "hmath.h"
#include "host_kin.h"
#include "host_model.h"
#include "model_view.h"
#include "xml_mini.h"

namespace mjb {
namespace {

const double kPi = 3.14159265358979323846;

std::vector<double> parse_nums(const std::string& s) {
  std::vector<double> out;
  const char* p = s.c_str();
  char* e;
  for (;;) {
    while (*p == ' ' || *p == '\t' || *p == '\n' || *p == '\r' || *p == ',') p++;
    if (!*p) break;
    double v = strtod(p, &e);
    if (e == p) throw std::runtime_error("MJCF: cannot parse number in '" + s + "'");
    out.push_back(v);
    p = e;
  }
  return out;
}

struct Attrs {
  // merged attribute lookup: element first, then the default class
  const XmlNode* el;
  const XmlNode* def;
  const std::string* get(const char* k) const {
    const std::string* v = el ? el->attr(k) : nullptr;
    if (!v && def) v = def->attr(k);
    return v;
  }
  bool has(const char* k) const { return get(k) != nullptr; }
  std::string str(const char* k, const std::string& d) const {
    const std::string* v = get(k);
    return v ? *v : d;
  }
  double num(const char* k, double d) const {
    const std::string* v = get(k);
    if (!v) return d;
    auto n = parse_nums(*v);
    if (n.empty()) throw std::runtime_error(std::string("MJCF: empty numeric attribute ") + k);
    return n[0];
  }
  std::vector<double> vec(const char* k, size_t n, const std::vector<double>& d, bool allow_short = false) const {
    const std::string* v = get(k);
    if (!v) return d;
    auto x = parse_nums(*v);
    if (x.size() < n) {
      if (!allow_short) throw std::runtime_error(std::string("MJCF: attribute ") + k + " needs " + std::to_string(n) + " numbers");
      std::vector<double> r = d;
      for (size_t i = 0; i < x.size(); i++) r[i] = x[i];
      return r;
    }
    x.resize(n);
    return x;
  }
  bool flag(const char* k, bool d) const {
    const std::string* v = get(k);
    if (!v) return d;
    if (*v == "true") return true;
    if (*v == "false") return false;
    if (*v == "auto") return d;
    throw std::runtime_error(std::string("MJCF: attribute ") + k + " must be true/false");
  }
};

struct CompilerOpts {
  bool degree = true;
  std::string eulerseq = "xyz";
};

Quat euler2quat(const std::vector<double>& e, const CompilerOpts& co) {
  Quat q;
  for (int i = 0; i < 3; i++) {
    double a = co.degree ? e[i] * kPi / 180.0 : e[i];
    char c = co.eulerseq[i];
    V3 ax;
    char lc = (char)tolower(c);
    ax[lc == 'x' ? 0 : (lc == 'y' ? 1 : 2)] = 1;
    Quat r = qaxisangle(ax, a);
    // lower-case: intrinsic (rotating frame) -> post-multiply; upper-case: extrinsic -> pre-multiply
    q = (c == lc) ? qmul(q, r) : qmul(r, q);
  }
  return qnormalized(q);
}

// orientation of an element from quat / euler / axisangle / zaxis (first one present wins)
Quat read_orientation(const Attrs& a, const CompilerOpts& co) {
  if (a.el && a.el->attr("quat")) {
    auto v = parse_nums(*a.el->attr("quat"));
    if (v.size() != 4) throw std::runtime_error("MJCF: quat needs 4 numbers");
    return qnormalized(Quat{v[0], v[1], v[2], v[3]});
  }
  if (a.el && a.el->attr("euler")) {
    auto v = parse_nums(*a.el->attr("euler"));
    if (v.size() != 3) throw std::runtime_error("MJCF: euler needs 3 numbers");
    return euler2quat(v, co);
  }
  if (a.el && a.el->attr("axisangle")) {
    auto v = parse_nums(*a.el->attr("axisangle"));
    if (v.size() != 4) throw std::runtime_error("MJCF: axisangle needs 4 numbers");
    double ang = co.degree ? v[3] * kPi / 180.0 : v[3];
    return qnormalized(qaxisangle(normalized(V3(v[0], v[1], v[2])), ang));
  }
  if (a.el && a.el->attr("xyaxes")) {
    auto v = parse_nums(*a.el->attr("xyaxes"));
    if (v.size() != 6) throw std::runtime_error("MJCF: xyaxes needs 6 numbers");
    V3 x = normalized(V3(v[0], v[1], v[2])), y(v[3], v[4], v[5]);
    y = normalized(y - x * dot(x, y));
    V3 z = cross(x, y);
    M3 R;
    for (int r = 0; r < 3; r++) { R(r, 0) = x[r]; R(r, 1) = y[r]; R(r, 2) = z[r]; }
    return qnormalized(m2q(R));
  }
  if (a.el && a.el->attr("zaxis")) {
    auto v = parse_nums(*a.el->attr("zaxis"));
    if (v.size() != 3) throw std::runtime_error("MJCF: zaxis needs 3 numbers");
    V3 z = normalized(V3(v[0], v[1], v[2]));
    V3 ax = cross(V3(0, 0, 1), z);
    double s = norm(ax), ang = std::atan2(s, z.z);
    if (s < 1e-10) ax = V3(1, 0, 0); else ax = ax * (1.0 / s);
    return qnormalized(qaxisangle(ax, ang));
  }
  return Quat();
}

// quaternion rotating +z onto `vec`
Quat z2quat(V3 vec) {
  V3 z = normalized(vec);
  V3 ax = cross(V3(0, 0, 1), z);
  double s = norm(ax), ang = std::atan2(s, z.z);
  if (s < 1e-10) ax = V3(1, 0, 0); else ax = ax * (1.0 / s);
  return qnormalized(qaxisangle(ax, ang));
}

struct Builder {
  HostModel& M;
  CompilerOpts co;
  const XmlNode *def_joint = nullptr, *def_geom = nullptr, *def_site = nullptr, *def_motor = nullptr;
  // growing per-object arrays
  std::vector<int32_t> body_parentid, body_jntnum, body_jntadr, body_geomnum, body_geomadr;
  std::vector<double> body_pos, body_quat;
  std::vector<std::string> body_name, jnt_name, geom_name, site_name, sensor_name, act_name;
  std::vector<int32_t> jnt_type, jnt_bodyid, jnt_limited;
  std::vector<double> jnt_pos, jnt_axis, jnt_range, jnt_margin, jnt_solref, jnt_solimp, jnt_armature, jnt_damping, jnt_ref;
  std::vector<int32_t> geom_type, geom_bodyid, geom_contype, geom_conaffinity, geom_condim;
  std::vector<double> geom_size, geom_pos, geom_quat, geom_friction, geom_margin, geom_gap, geom_solmix, geom_solref,
      geom_solimp, geom_rgba, geom_density, geom_massattr;
  std::vector<int32_t> site_bodyid, site_type;
  std::vector<double> site_pos, site_quat, site_size;
  std::vector<int32_t> cam_bodyid, cam_mode;
  std::vector<double> cam_pos, cam_quat, cam_fovy;
  std::vector<std::string> cam_name;

  explicit Builder(HostModel& m) : M(m) {}

  int geom_type_code(const std::string& t) {
    if (t == "plane") return MJB_GEOM_PLANE;
    if (t == "sphere") return MJB_GEOM_SPHERE;
    if (t == "capsule") return MJB_GEOM_CAPSULE;
    if (t == "box") return MJB_GEOM_BOX;
    throw std::runtime_error("MJCF: unsupported geom type '" + t + "' (supported: plane, sphere, capsule, box)");
  }

  void add_geom(const XmlNode* g, int body) {
    Attrs a{g, def_geom};
    int type = geom_type_code(a.str("type", "sphere"));
    std::vector<double> size = a.vec("size", 3, {0, 0, 0}, true);
    V3 pos(0, 0, 0);
    Quat quat;
    if (g->attr("fromto")) {
      if (type != MJB_GEOM_CAPSULE && type != MJB_GEOM_BOX)
        throw std::runtime_error("MJCF: fromto is only supported for capsule/box geoms");
      auto ft = parse_nums(*g->attr("fromto"));
      if (ft.size() != 6) throw std::runtime_error("MJCF: fromto needs 6 numbers");
      V3 p0(ft[0], ft[1], ft[2]), p1(ft[3], ft[4], ft[5]);
      pos = (p0 + p1) * 0.5;
      V3 d = p1 - p0;
      double len = norm(d);
      if (len < 1e-12) throw std::runtime_error("MJCF: fromto has zero length");
      quat = z2quat(d);
      if (type == MJB_GEOM_CAPSULE) size[1] = len * 0.5; else size[2] = len * 0.5;
    } else {
      auto p = a.vec("pos", 3, {0, 0, 0});
      pos = V3(p[0], p[1], p[2]);
      quat = read_orientation(a, co);
    }
    if (type == MJB_GEOM_SPHERE && size[0] <= 0) throw std::runtime_error("MJCF: sphere needs size > 0");
    if (type == MJB_GEOM_CAPSULE && (size[0] <= 0 || size[1] <= 0)) throw std::runtime_error("MJCF: capsule needs radius and half-length");
    if (type == MJB_GEOM_BOX && (size[0] <= 0 || size[1] <= 0 || size[2] <= 0)) throw std::runtime_error("MJCF: box needs 3 positive half-sizes");
    geom_type.push_back(type);
    geom_bodyid.push_back(body);
    geom_contype.push_back((int)a.num("contype", 1));
    geom_conaffinity.push_back((int)a.num("conaffinity", 1));
    geom_condim.push_back((int)a.num("condim", 3));
    for (int i = 0; i < 3; i++) geom_size.push_back(size[i]);
    for (int i = 0; i < 3; i++) geom_pos.push_back(pos[i]);
    geom_quat.insert(geom_quat.end(), {quat.w, quat.x, quat.y, quat.z});
    auto fr = a.vec("friction", 3, {1, 0.005, 0.0001}, true);
    geom_friction.insert(geom_friction.end(), fr.begin(), fr.end());
    geom_margin.push_back(a.num("margin", 0));
    geom_gap.push_back(a.num("gap", 0));
    geom_solmix.push_back(a.num("solmix", 1));
    auto sr = a.vec("solref", 2, {0.02, 1});
    geom_solref.insert(geom_solref.end(), sr.begin(), sr.end());
    auto si = a.vec("solimp", 5, {0.9, 0.95, 0.001, 0.5, 2}, true);
    geom_solimp.insert(geom_solimp.end(), si.begin(), si.end());
    auto rgba = a.vec("rgba", 4, {0.5, 0.5, 0.5, 1});
    geom_rgba.insert(geom_rgba.end(), rgba.begin(), rgba.end());
    geom_density.push_back(a.num("density", 1000));
    geom_massattr.push_back(g->attr("mass") ? a.num("mass", -1) : -1);
    geom_name.push_back(a.el->attr("name") ? *a.el->attr("name") : "");
  }

  void add_joint(const XmlNode* j, int body) {
    Attrs a{j, def_joint};
    std::string t = a.str("type", "hinge");
    int type;
    if (t == "free") type = MJB_JNT_FREE;
    else if (t == "hinge") type = MJB_JNT_HINGE;
    else if (t == "slide") type = MJB_JNT_SLIDE;
    else throw std::runtime_error("MJCF: unsupported joint type '" + t + "' (supported: free, hinge, slide)");
    jnt_type.push_back(type);
    jnt_bodyid.push_back(body);
    auto p = a.vec("pos", 3, {0, 0, 0});
    auto ax = a.vec("axis", 3, {0, 0, 1});
    V3 axis = normalized(V3(ax[0], ax[1], ax[2]));
    if (type == MJB_JNT_FREE) { p = {0, 0, 0}; axis = V3(0, 0, 1); }
    jnt_pos.insert(jnt_pos.end(), p.begin(), p.end());
    jnt_axis.insert(jnt_axis.end(), {axis.x, axis.y, axis.z});
    bool has_range = a.has("range");
    auto rg = a.vec("range", 2, {0, 0});
    if (co.degree && type == MJB_JNT_HINGE) { rg[0] *= kPi / 180.0; rg[1] *= kPi / 180.0; }
    // limited: explicit true/false, "auto" -> range present (MuJoCo autolimits)
    bool limited = false;
    const std::string* lim = a.get("limited");
    if (lim) limited = (*lim == "true") || (*lim == "auto" && has_range);
    if (type == MJB_JNT_FREE) limited = false;
    jnt_limited.push_back(limited ? 1 : 0);
    jnt_range.insert(jnt_range.end(), rg.begin(), rg.end());
    jnt_margin.push_back(a.num("margin", 0));
    auto sr = a.vec("solreflimit", 2, {0.02, 1});
    jnt_solref.insert(jnt_solref.end(), sr.begin(), sr.end());
    auto si = a.vec("solimplimit", 5, {0.9, 0.95, 0.001, 0.5, 2}, true);
    jnt_solimp.insert(jnt_solimp.end(), si.begin(), si.end());
    jnt_armature.push_back(a.num("armature", 0));
    jnt_damping.push_back(a.num("damping", 0));
    double ref = a.num("ref", 0);
    if (co.degree && type == MJB_JNT_HINGE) ref *= kPi / 180.0;
    jnt_ref.push_back(ref);
    jnt_name.push_back(j->attr("name") ? *j->attr("name") : "");
  }

  void add_site(const XmlNode* s, int body) {
    Attrs a{s, def_site};
    std::string t = a.str("type", "sphere");
    int type = t == "sphere" ? MJB_GEOM_SPHERE : (t == "capsule" ? MJB_GEOM_CAPSULE : (t == "box" ? MJB_GEOM_BOX : -1));
    if (type < 0) throw std::runtime_error("MJCF: unsupported site type '" + t + "'");
    site_type.push_back(type);
    site_bodyid.push_back(body);
    auto p = a.vec("pos", 3, {0, 0, 0});
    site_pos.insert(site_pos.end(), p.begin(), p.end());
    Quat q = read_orientation(a, co);
    site_quat.insert(site_quat.end(), {q.w, q.x, q.y, q.z});
    auto sz = a.vec("size", 3, {0.005, 0.005, 0.005}, true);
    site_size.insert(site_size.end(), sz.begin(), sz.end());
    site_name.push_back(s->attr("name") ? *s->attr("name") : "");
  }

  // <camera>: body-fixed frame looking along its -z with +y up (MuJoCo's convention); other modes keep their
  // mode id so that a render request for them can be refused
  void add_camera(const XmlNode* s, int body) {
    Attrs a{s, nullptr};
    std::string mode = a.str("mode", "fixed");
    cam_mode.push_back(mode == "fixed" ? 0 : 1);
    cam_bodyid.push_back(body);
    auto p = a.vec("pos", 3, {0, 0, 0});
    cam_pos.insert(cam_pos.end(), p.begin(), p.end());
    Quat q = read_orientation(a, co);
    cam_quat.insert(cam_quat.end(), {q.w, q.x, q.y, q.z});
    cam_fovy.push_back(a.num("fovy", 45.0));
    cam_name.push_back(s->attr("name") ? *s->attr("name") : "");
  }

  // depth-first, pre-order: a body gets its id before its children (MuJoCo's numbering)
  void add_body(const XmlNode* b, int parent) {
    int id = (int)body_parentid.size();
    body_parentid.push_back(parent);
    Attrs a{b, nullptr};
    auto p = a.vec("pos", 3, {0, 0, 0});
    body_pos.insert(body_pos.end(), p.begin(), p.end());
    Quat q = read_orientation(a, co);
    body_quat.insert(body_quat.end(), {q.w, q.x, q.y, q.z});
    body_name.push_back(b->attr("name") ? *b->attr("name") : "");
    body_jntadr.push_back((int)jnt_type.size());
    body_geomadr.push_back((int)geom_type.size());
    int nj = 0, ng = 0;
    for (auto& c : b->children) {
      if (c->tag == "joint") { add_joint(c.get(), id); nj++; }
      else if (c->tag == "freejoint") {
        XmlNode tmp; tmp.tag = "joint"; tmp.attrs = c->attrs; tmp.attrs.emplace_back("type", "free");
        const XmlNode* keep = def_joint; def_joint = nullptr;  // freejoint ignores joint defaults
        add_joint(&tmp, id); def_joint = keep; nj++;
      }
      else if (c->tag == "geom") { add_geom(c.get(), id); ng++; }
      else if (c->tag == "site") add_site(c.get(), id);
      else if (c->tag == "camera") add_camera(c.get(), id);
    }
    body_jntnum.push_back(nj);
    body_geomnum.push_back(ng);
    if (nj == 0) body_jntadr[id] = -1;
    if (ng == 0) body_geomadr[id] = -1;
    for (auto& c : b->children)
      if (c->tag == "body") add_body(c.get(), id);
  }
};

int find_name(const std::vector<std::string>& v, const std::string& n) {
  if (n.empty()) return -1;
  for (size_t i = 0; i < v.size(); i++)
    if (v[i] == n) return (int)i;
  return -1;
}

void geom_mass_inertia(int type, const double* size, double density, double massattr, double& mass, double inertia[3]) {
  double vol = 0;
  if (type == MJB_GEOM_SPHERE) vol = 4.0 / 3.0 * kPi * size[0] * size[0] * size[0];
  else if (type == MJB_GEOM_CAPSULE) {
    double h = 2 * size[1], r = size[0];
    vol = kPi * (r * r * h + 4.0 / 3.0 * r * r * r);
  } else if (type == MJB_GEOM_BOX) vol = 8 * size[0] * size[1] * size[2];
  mass = massattr >= 0 ? massattr : density * vol;
  inertia[0] = inertia[1] = inertia[2] = 0;
  if (type == MJB_GEOM_SPHERE) {
    inertia[0] = inertia[1] = inertia[2] = 2.0 * mass * size[0] * size[0] / 5.0;
  } else if (type == MJB_GEOM_CAPSULE) {
    double h = 2 * size[1], r = size[0];
    double sphere_mass = mass * 4 * r / (4 * r + 3 * h);
    double cyl_mass = mass - sphere_mass;
    inertia[0] = inertia[1] = cyl_mass * (3 * r * r + h * h) / 12.0;
    inertia[2] = cyl_mass * r * r / 2.0;
    double si = 2 * sphere_mass * r * r / 5.0;
    inertia[0] += si + sphere_mass * h * (3 * r + 2 * h) / 8.0;
    inertia[1] += si + sphere_mass * h * (3 * r + 2 * h) / 8.0;
    inertia[2] += si;
  } else if (type == MJB_GEOM_BOX) {
    inertia[0] = mass * (size[1] * size[1] + size[2] * size[2]) / 3.0;
    inertia[1] = mass * (size[0] * size[0] + size[2] * size[2]) / 3.0;
    inertia[2] = mass * (size[0] * size[0] + size[1] * size[1]) / 3.0;
  }
}

}  // namespace

void compile_mjcf(const std::string& xml_text, HostModel& M) {
  XmlParser parser(xml_text);
  std::unique_ptr<XmlNode> root = parser.parse();
  if (root->tag != "mujoco") throw std::runtime_error("MJCF: root element must be <mujoco>");
  Builder B(M);

  if (const XmlNode* c = root->child("compiler")) {
    if (const std::string* a = c->attr("angle")) {
      if (*a == "radian") B.co.degree = false;
      else if (*a != "degree") throw std::runtime_error("MJCF: compiler angle must be degree or radian");
    }
    if (const std::string* a = c->attr("eulerseq")) {
      if (a->size() != 3) throw std::runtime_error("MJCF: eulerseq needs 3 characters");
      B.co.eulerseq = *a;
    }
    if (const std::string* a = c->attr("coordinate"))
      if (*a != "local") throw std::runtime_error("MJCF: only coordinate=local is supported");
  }
  double timestep = 0.002, impratio = 1, tolerance = 1e-8;
  int integrator = MJB_INT_EULER, iterations = 100;
  std::vector<double> gravity = {0, 0, -9.81};
  if (const XmlNode* o = root->child("option")) {
    Attrs a{o, nullptr};
    timestep = a.num("timestep", timestep);
    impratio = a.num("impratio", impratio);
    tolerance = a.num("tolerance", tolerance);
    iterations = (int)a.num("iterations", iterations);
    gravity = a.vec("gravity", 3, gravity);
    std::string in = a.str("integrator", "Euler");
    if (in == "Euler") integrator = MJB_INT_EULER;
    else if (in == "RK4") integrator = MJB_INT_RK4;
    else throw std::runtime_error("MJCF: unsupported integrator '" + in + "' (supported: Euler, RK4)");
    std::string cone = a.str("cone", "pyramidal");
    if (cone != "pyramidal") throw std::runtime_error("MJCF: only cone=pyramidal is supported");
  }
  if (const XmlNode* d = root->child("default")) {
    B.def_joint = d->child("joint");
    B.def_geom = d->child("geom");
    B.def_site = d->child("site");
    B.def_motor = d->child("motor");
    if (d->child("default")) throw std::runtime_error("MJCF: nested default classes are not supported");
  }

  const XmlNode* wb = root->child("worldbody");
  if (!wb) throw std::runtime_error("MJCF: missing <worldbody>");
  // world body = id 0
  B.body_parentid.push_back(0);
  B.body_pos.insert(B.body_pos.end(), {0, 0, 0});
  B.body_quat.insert(B.body_quat.end(), {1, 0, 0, 0});
  B.body_name.push_back("world");
  B.body_jntadr.push_back(-1);
  B.body_jntnum.push_back(0);
  B.body_geomadr.push_back((int)B.geom_type.size());
  int ng0 = 0;
  for (auto& c : wb->children) {
    if (c->tag == "geom") { B.add_geom(c.get(), 0); ng0++; }
    else if (c->tag == "site") B.add_site(c.get(), 0);
    else if (c->tag == "camera") B.add_camera(c.get(), 0);
    else if (c->tag == "joint" || c->tag == "freejoint") throw std::runtime_error("MJCF: joints are not allowed in the world body");
  }
  B.body_geomnum.push_back(ng0);
  if (ng0 == 0) B.body_geomadr[0] = -1;
  for (auto& c : wb->children)
    if (c->tag == "body") B.add_body(c.get(), 0);

  const int nbody = (int)B.body_parentid.size(), njnt = (int)B.jnt_type.size(), ngeom = (int)B.geom_type.size(),
            nsite = (int)B.site_type.size();

  // geoms were appended body by body in pre-order EXCEPT that a body's geoms are added before its
  // children, which is exactly body-id order -> geom ids are already grouped by body.

  // ---- joints -> qpos / dof layout
  std::vector<int32_t> jnt_qposadr(njnt), jnt_dofadr(njnt);
  int nq = 0, nv = 0;
  for (int j = 0; j < njnt; j++) {
    jnt_qposadr[j] = nq; jnt_dofadr[j] = nv;
    if (B.jnt_type[j] == MJB_JNT_FREE) {
      int b = B.jnt_bodyid[j];
      if (B.body_parentid[b] != 0 || B.body_jntnum[b] != 1)
        throw std::runtime_error("MJCF: a free joint must be the only joint of a top-level body");
      nq += 7; nv += 6;
    } else { nq += 1; nv += 1; }
  }
  std::vector<double> qpos0(nq, 0.0);
  std::vector<int32_t> dof_bodyid(nv), dof_jntid(nv), dof_parentid(nv);
  std::vector<double> dof_armature(nv), dof_damping(nv);
  std::vector<int32_t> body_dofnum(nbody, 0), body_dofadr(nbody, -1), body_rootid(nbody, 0), body_weldid(nbody, 0),
      body_depth(nbody, 0), body_treeid(nbody, -1);
  std::vector<int> body_lastdof(nbody, -1);  // last dof of the nearest moving ancestor-or-self
  int ntree = 0, maxdepth = 0;
  for (int b = 1; b < nbody; b++) {
    int p = B.body_parentid[b];
    body_rootid[b] = (p == 0) ? b : body_rootid[p];
    body_weldid[b] = (B.body_jntnum[b] == 0) ? body_weldid[p] : b;
    body_depth[b] = (p == 0) ? 1 : body_depth[p] + 1;
    maxdepth = std::max(maxdepth, body_depth[b]);
    int last = body_lastdof[p];
    if (B.body_jntnum[b] > 0) body_dofadr[b] = jnt_dofadr[B.body_jntadr[b]];
    for (int j = B.body_jntadr[b]; j >= 0 && j < B.body_jntadr[b] + B.body_jntnum[b]; j++) {
      int nd = B.jnt_type[j] == MJB_JNT_FREE ? 6 : 1;
      for (int i = 0; i < nd; i++) {
        int d = jnt_dofadr[j] + i;
        dof_bodyid[d] = b; dof_jntid[d] = j; dof_parentid[d] = last;
        dof_armature[d] = B.jnt_armature[j]; dof_damping[d] = B.jnt_damping[j];
        last = d;
      }
      body_dofnum[b] += nd;
      if (B.jnt_type[j] == MJB_JNT_FREE) {
        int qa = jnt_qposadr[j];
        for (int i = 0; i < 3; i++) qpos0[qa + i] = B.body_pos[3 * b + i];
        for (int i = 0; i < 4; i++) qpos0[qa + 3 + i] = B.body_quat[4 * b + i];
      } else {
        qpos0[jnt_qposadr[j]] = B.jnt_ref[j];
      }
    }
    body_lastdof[b] = last;
    // kinematic tree id: trees are rooted at top-level bodies that (or whose descendants) move
    if (p == 0) body_treeid[b] = -2;  // resolved below
    else body_treeid[b] = body_treeid[p];
  }
  // assign tree ids to top-level subtrees that contain at least one dof
  {
    std::vector<int> sub_has_dof(nbody, 0);
    for (int b = nbody - 1; b >= 1; b--) {
      if (body_dofnum[b] > 0) sub_has_dof[b] = 1;
      if (sub_has_dof[b]) sub_has_dof[B.body_parentid[b]] = 1;
    }
    std::vector<int> root_tree(nbody, -1);
    for (int b = 1; b < nbody; b++)
      if (B.body_parentid[b] == 0 && sub_has_dof[b]) root_tree[b] = ntree++;
    for (int b = 1; b < nbody; b++) body_treeid[b] = root_tree[body_rootid[b]];
  }

  // ---- body inertial properties from geoms (inertiafromgeom)
  std::vector<double> body_mass(nbody, 0.0), body_inertia(3 * nbody, 0.0), body_ipos(3 * nbody, 0.0),
      body_iquat(4 * nbody, 0.0), body_subtreemass(nbody, 0.0), geom_rbound(ngeom, 0.0);
  for (int b = 0; b < nbody; b++) body_iquat[4 * b] = 1;
  for (int g = 0; g < ngeom; g++) {
    const double* s = &B.geom_size[3 * g];
    switch (B.geom_type[g]) {
      case MJB_GEOM_SPHERE: geom_rbound[g] = s[0]; break;
      case MJB_GEOM_CAPSULE: geom_rbound[g] = s[0] + s[1]; break;
      case MJB_GEOM_BOX: geom_rbound[g] = std::sqrt(s[0] * s[0] + s[1] * s[1] + s[2] * s[2]); break;
      default: geom_rbound[g] = 0; break;
    }
  }
  for (int b = 1; b < nbody; b++) {
    int ga = B.body_geomadr[b], gn = B.body_geomnum[b];
    if (gn <= 0) continue;
    double mtot = 0;
    V3 com;
    std::vector<double> gm(gn);
    std::vector<double> gi(3 * gn);
    for (int k = 0; k < gn; k++) {
      int g = ga + k;
      geom_mass_inertia(B.geom_type[g], &B.geom_size[3 * g], B.geom_density[g], B.geom_massattr[g], gm[k], &gi[3 * k]);
      mtot += gm[k];
      com = com + V3(B.geom_pos[3 * g], B.geom_pos[3 * g + 1], B.geom_pos[3 * g + 2]) * gm[k];
    }
    if (mtot <= 0) continue;
    com = com * (1.0 / mtot);
    body_mass[b] = mtot;
    for (int i = 0; i < 3; i++) body_ipos[3 * b + i] = com[i];
    if (gn == 1) {
      // single geom: inertial frame = geom frame (no eigen-decomposition needed)
      for (int i = 0; i < 4; i++) body_iquat[4 * b + i] = B.geom_quat[4 * ga + i];
      for (int i = 0; i < 3; i++) body_inertia[3 * b + i] = gi[i];
    } else {
      M3 T;
      for (int i = 0; i < 9; i++) T.m[i] = 0;
      for (int k = 0; k < gn; k++) {
        int g = ga + k;
        M3 R = q2m(Quat{B.geom_quat[4 * g], B.geom_quat[4 * g + 1], B.geom_quat[4 * g + 2], B.geom_quat[4 * g + 3]});
        V3 d = V3(B.geom_pos[3 * g], B.geom_pos[3 * g + 1], B.geom_pos[3 * g + 2]) - com;
        for (int r = 0; r < 3; r++)
          for (int c = 0; c < 3; c++) {
            double s = 0;
            for (int a2 = 0; a2 < 3; a2++) s += R(r, a2) * gi[3 * k + a2] * R(c, a2);
            s += gm[k] * ((r == c ? dot(d, d) : 0.0) - d[r] * d[c]);
            T(r, c) += s;
          }
      }
      double ev[3];
      M3 V;
      eig3(T, ev, V);
      Quat q = m2q(V);
      body_iquat[4 * b] = q.w; body_iquat[4 * b + 1] = q.x; body_iquat[4 * b + 2] = q.y; body_iquat[4 * b + 3] = q.z;
      for (int i = 0; i < 3; i++) body_inertia[3 * b + i] = ev[i];
    }
  }
  for (int b = nbody - 1; b >= 1; b--) {
    body_subtreemass[b] += body_mass[b];
    body_subtreemass[B.body_parentid[b]] += body_subtreemass[b];
  }
  for (int b = 1; b < nbody; b++)
    if (body_dofnum[b] > 0 && body_subtreemass[b] <= 0)
      throw std::runtime_error("MJCF: moving body '" + B.body_name[b] + "' has no mass");

  // ---- sensors
  std::vector<int32_t> sensor_type, sensor_objtype, sensor_objid, sensor_adr, sensor_dim, sensor_datatype;
  std::vector<double> sensor_cutoff;
  int nsensordata = 0;
  if (const XmlNode* sn = root->child("sensor")) {
    for (auto& s : sn->children) {
      const std::string what = "MJCF: sensor <" + s->tag + (s->attr("name") ? " name='" + *s->attr("name") + "'" : std::string()) + ">";
      auto fail = [&](const std::string& why) { throw std::runtime_error(what + ": " + why); };
      int type, dim, datatype = MJB_DATA_REAL;
      // attribute naming the object: "site", "joint" or "objname" (with "objtype")
      enum { BY_SITE, BY_JOINT, BY_FRAME } by = BY_SITE;
      if (s->tag == "touch") { type = MJB_SENS_TOUCH; dim = 1; datatype = MJB_DATA_POSITIVE; }
      else if (s->tag == "accelerometer") { type = MJB_SENS_ACCELEROMETER; dim = 3; }
      else if (s->tag == "velocimeter") { type = MJB_SENS_VELOCIMETER; dim = 3; }
      else if (s->tag == "gyro") { type = MJB_SENS_GYRO; dim = 3; }
      else if (s->tag == "rangefinder") { type = MJB_SENS_RANGEFINDER; dim = 1; datatype = MJB_DATA_POSITIVE; }
      else if (s->tag == "jointpos") { type = MJB_SENS_JOINTPOS; dim = 1; by = BY_JOINT; }
      else if (s->tag == "jointvel") { type = MJB_SENS_JOINTVEL; dim = 1; by = BY_JOINT; }
      else if (s->tag == "framepos") { type = MJB_SENS_FRAMEPOS; dim = 3; by = BY_FRAME; }
      else if (s->tag == "framequat") { type = MJB_SENS_FRAMEQUAT; dim = 4; datatype = MJB_DATA_QUATERNION; by = BY_FRAME; }
      else if (s->tag == "framexaxis") { type = MJB_SENS_FRAMEXAXIS; dim = 3; datatype = MJB_DATA_AXIS; by = BY_FRAME; }
      else if (s->tag == "frameyaxis") { type = MJB_SENS_FRAMEYAXIS; dim = 3; datatype = MJB_DATA_AXIS; by = BY_FRAME; }
      else if (s->tag == "framezaxis") { type = MJB_SENS_FRAMEZAXIS; dim = 3; datatype = MJB_DATA_AXIS; by = BY_FRAME; }
      else if (s->tag == "framelinvel") { type = MJB_SENS_FRAMELINVEL; dim = 3; by = BY_FRAME; }
      else if (s->tag == "frameangvel") { type = MJB_SENS_FRAMEANGVEL; dim = 3; by = BY_FRAME; }
      else throw std::runtime_error("MJCF: unsupported sensor <" + s->tag + ">");
      if (s->attr("reftype") || s->attr("refname")) fail("reftype / refname are not supported");
      int objtype = MJB_OBJ_SITE, objid = -1;
      std::string objname;
      if (by == BY_FRAME) {
        const std::string* ot = s->attr("objtype");
        if (!ot) fail("needs objtype");
        if (!s->attr("objname")) fail("needs objname");
        objname = *s->attr("objname");
        if (*ot == "site") { objtype = MJB_OBJ_SITE; objid = find_name(B.site_name, objname); }
        else if (*ot == "body" || *ot == "xbody") {
          objtype = *ot == "body" ? MJB_OBJ_BODY : MJB_OBJ_XBODY;
          objid = find_name(B.body_name, objname);
        } else if (*ot == "geom") { objtype = MJB_OBJ_GEOM; objid = find_name(B.geom_name, objname); }
        else fail("objtype '" + *ot + "' is not supported (supported: site, body, xbody, geom)");
      } else if (by == BY_JOINT) {
        if (!s->attr("joint")) fail("needs a joint");
        objname = *s->attr("joint");
        objtype = MJB_OBJ_JOINT;
        objid = find_name(B.jnt_name, objname);
        if (objid >= 0 && B.jnt_type[objid] == MJB_JNT_FREE) fail("joint '" + objname + "' is a free joint (supported: hinge, slide)");
      } else {
        if (!s->attr("site")) fail("needs a site");
        objname = *s->attr("site");
        objid = find_name(B.site_name, objname);
      }
      if (objid < 0) fail("refers to unknown object '" + objname + "'");
      Attrs a{s.get(), nullptr};
      sensor_type.push_back(type); sensor_objtype.push_back(objtype); sensor_objid.push_back(objid);
      sensor_adr.push_back(nsensordata); sensor_dim.push_back(dim); sensor_datatype.push_back(datatype);
      sensor_cutoff.push_back(a.num("cutoff", 0));
      B.sensor_name.push_back(s->attr("name") ? *s->attr("name") : "");
      nsensordata += dim;
    }
  }
  const int nsensor = (int)sensor_type.size();

  // ---- actuators (motors on joints)
  std::vector<int32_t> actuator_trnid, actuator_ctrllimited;
  std::vector<double> actuator_gear, actuator_ctrlrange;
  if (const XmlNode* an = root->child("actuator")) {
    for (auto& mtr : an->children) {
      if (mtr->tag != "motor") throw std::runtime_error("MJCF: unsupported actuator <" + mtr->tag + "> (supported: motor)");
      Attrs a{mtr.get(), B.def_motor};
      const std::string* jn = mtr->attr("joint");
      if (!jn) throw std::runtime_error("MJCF: motor needs a joint");
      int jid = find_name(B.jnt_name, *jn);
      if (jid < 0) throw std::runtime_error("MJCF: motor refers to unknown joint '" + *jn + "'");
      if (B.jnt_type[jid] == MJB_JNT_FREE) throw std::runtime_error("MJCF: motors on free joints are not supported");
      actuator_trnid.push_back(jid);
      auto cr = a.vec("ctrlrange", 2, {0, 0});
      bool has_range = a.has("ctrlrange");
      bool lim = false;
      const std::string* cl = a.get("ctrllimited");
      if (cl) lim = (*cl == "true") || (*cl == "auto" && has_range);
      actuator_ctrllimited.push_back(lim ? 1 : 0);
      actuator_ctrlrange.insert(actuator_ctrlrange.end(), cr.begin(), cr.end());
      auto gear = a.vec("gear", 1, {1}, true);
      actuator_gear.push_back(gear[0]);
      B.act_name.push_back(mtr->attr("name") ? *mtr->attr("name") : "");
    }
  }
  const int nu = (int)actuator_trnid.size();

  // ---- static collision pair table.  Filters (MuJoCo documented rules):
  //   (contype1 & conaffinity2) || (contype2 & conaffinity1); not the same weld body; not
  //   weld-parent / weld-child unless one of them is welded to the world.
  struct Pair { int b1, b2, g1, g2; };
  std::vector<Pair> pairs;
  for (int g1 = 0; g1 < ngeom; g1++)
    for (int g2 = g1 + 1; g2 < ngeom; g2++) {
      int b1 = B.geom_bodyid[g1], b2 = B.geom_bodyid[g2];
      int w1 = body_weldid[b1], w2 = body_weldid[b2];
      if (w1 == w2) continue;
      if (!((B.geom_contype[g1] & B.geom_conaffinity[g2]) || (B.geom_contype[g2] & B.geom_conaffinity[g1]))) continue;
      int wp1 = body_weldid[B.body_parentid[w1]], wp2 = body_weldid[B.body_parentid[w2]];
      if (w1 != 0 && w2 != 0 && (w1 == wp2 || w2 == wp1)) continue;
      if (B.geom_type[g1] == MJB_GEOM_PLANE && B.geom_type[g2] == MJB_GEOM_PLANE) continue;
      Pair p{std::min(b1, b2), std::max(b1, b2), g1, g2};
      if (B.geom_type[g1] > B.geom_type[g2]) std::swap(p.g1, p.g2);
      pairs.push_back(p);
    }
  std::stable_sort(pairs.begin(), pairs.end(), [](const Pair& x, const Pair& y) {
    if (x.b1 != y.b1) return x.b1 < y.b1;
    return x.b2 < y.b2;
  });
  const int npair = (int)pairs.size();
  std::vector<int32_t> pair_geom1(npair), pair_geom2(npair), pair_condim(npair);
  std::vector<double> pair_margin(npair), pair_includemargin(npair), pair_friction(3 * npair), pair_solref(2 * npair),
      pair_solimp(5 * npair);
  for (int k = 0; k < npair; k++) {
    int g1 = pairs[k].g1, g2 = pairs[k].g2;
    pair_geom1[k] = g1; pair_geom2[k] = g2;
    pair_condim[k] = std::max(B.geom_condim[g1], B.geom_condim[g2]);
    if (pair_condim[k] != 3 && pair_condim[k] != 1)
      throw std::runtime_error("MJCF: only condim 1 and 3 contacts are supported");
    double margin = std::max(B.geom_margin[g1], B.geom_margin[g2]);
    double gap = std::max(B.geom_gap[g1], B.geom_gap[g2]);
    pair_margin[k] = margin; pair_includemargin[k] = margin - gap;
    for (int i = 0; i < 3; i++) pair_friction[3 * k + i] = std::max(B.geom_friction[3 * g1 + i], B.geom_friction[3 * g2 + i]);
    double s1 = B.geom_solmix[g1], s2 = B.geom_solmix[g2];
    double mix = (s1 >= 1e-15 && s2 >= 1e-15) ? s1 / (s1 + s2) : (s1 < 1e-15 && s2 < 1e-15 ? 0.5 : (s1 < 1e-15 ? 0.0 : 1.0));
    if (B.geom_solref[2 * g1] > 0 && B.geom_solref[2 * g2] > 0)
      for (int i = 0; i < 2; i++) pair_solref[2 * k + i] = mix * B.geom_solref[2 * g1 + i] + (1 - mix) * B.geom_solref[2 * g2 + i];
    else
      for (int i = 0; i < 2; i++) pair_solref[2 * k + i] = std::min(B.geom_solref[2 * g1 + i], B.geom_solref[2 * g2 + i]);
    for (int i = 0; i < 5; i++) pair_solimp[5 * k + i] = mix * B.geom_solimp[5 * g1 + i] + (1 - mix) * B.geom_solimp[5 * g2 + i];
  }

  // ---- fill the model
  M.set_int("nq", nq); M.set_int("nv", nv); M.set_int("nu", nu); M.set_int("nbody", nbody); M.set_int("njnt", njnt);
  M.set_int("ngeom", ngeom); M.set_int("nsite", nsite); M.set_int("nsensor", nsensor);
  M.set_int("nsensordata", nsensordata); M.set_int("npair", npair); M.set_int("opt_integrator", integrator);
  M.set_int("ntree", ntree); M.set_int("maxdepth", maxdepth); M.set_int("opt_iterations", iterations);
  M.set_f64("opt_timestep", timestep); M.set_f64("opt_impratio", impratio); M.set_f64("opt_tolerance", tolerance);
  M.F("opt_gravity") = gravity;
  M.I("body_parentid") = B.body_parentid; M.I("body_rootid") = body_rootid; M.I("body_weldid") = body_weldid;
  M.I("body_jntnum") = B.body_jntnum; M.I("body_jntadr") = B.body_jntadr; M.I("body_dofnum") = body_dofnum;
  M.I("body_dofadr") = body_dofadr; M.I("body_geomnum") = B.body_geomnum; M.I("body_geomadr") = B.body_geomadr;
  M.I("body_depth") = body_depth; M.I("body_treeid") = body_treeid;
  M.F("body_pos") = B.body_pos; M.F("body_quat") = B.body_quat; M.F("body_ipos") = body_ipos;
  M.F("body_iquat") = body_iquat; M.F("body_mass") = body_mass; M.F("body_inertia") = body_inertia;
  M.F("body_subtreemass") = body_subtreemass;
  M.I("jnt_type") = B.jnt_type; M.I("jnt_bodyid") = B.jnt_bodyid; M.I("jnt_qposadr") = jnt_qposadr;
  M.I("jnt_dofadr") = jnt_dofadr; M.I("jnt_limited") = B.jnt_limited;
  M.F("jnt_pos") = B.jnt_pos; M.F("jnt_axis") = B.jnt_axis; M.F("jnt_range") = B.jnt_range;
  M.F("jnt_margin") = B.jnt_margin; M.F("jnt_solref") = B.jnt_solref; M.F("jnt_solimp") = B.jnt_solimp;
  M.I("dof_bodyid") = dof_bodyid; M.I("dof_jntid") = dof_jntid; M.I("dof_parentid") = dof_parentid;
  M.F("dof_armature") = dof_armature; M.F("dof_damping") = dof_damping;
  M.I("geom_type") = B.geom_type; M.I("geom_bodyid") = B.geom_bodyid; M.I("geom_contype") = B.geom_contype;
  M.I("geom_conaffinity") = B.geom_conaffinity; M.I("geom_condim") = B.geom_condim;
  M.F("geom_size") = B.geom_size; M.F("geom_pos") = B.geom_pos; M.F("geom_quat") = B.geom_quat;
  M.F("geom_friction") = B.geom_friction; M.F("geom_margin") = B.geom_margin; M.F("geom_gap") = B.geom_gap;
  M.F("geom_solmix") = B.geom_solmix; M.F("geom_solref") = B.geom_solref; M.F("geom_solimp") = B.geom_solimp;
  M.F("geom_rbound") = geom_rbound; M.F("geom_rgba") = B.geom_rgba;
  M.I("site_bodyid") = B.site_bodyid; M.I("site_type") = B.site_type;
  M.F("site_pos") = B.site_pos; M.F("site_quat") = B.site_quat; M.F("site_size") = B.site_size;
  M.I("sensor_type") = sensor_type; M.I("sensor_objtype") = sensor_objtype; M.I("sensor_objid") = sensor_objid;
  M.I("sensor_adr") = sensor_adr; M.I("sensor_dim") = sensor_dim; M.I("sensor_datatype") = sensor_datatype;
  M.F("sensor_cutoff") = sensor_cutoff;
  M.I("actuator_trnid") = actuator_trnid; M.I("actuator_ctrllimited") = actuator_ctrllimited;
  M.F("actuator_gear") = actuator_gear; M.F("actuator_ctrlrange") = actuator_ctrlrange;
  M.I("pair_geom1") = pair_geom1; M.I("pair_geom2") = pair_geom2; M.I("pair_condim") = pair_condim;
  M.F("pair_margin") = pair_margin; M.F("pair_includemargin") = pair_includemargin;
  M.F("pair_friction") = pair_friction; M.F("pair_solref") = pair_solref; M.F("pair_solimp") = pair_solimp;
  M.F("qpos0") = qpos0;
  M.set_int("ncam", (int)B.cam_bodyid.size());
  M.I("cam_bodyid") = B.cam_bodyid; M.I("cam_mode") = B.cam_mode;
  M.F("cam_pos") = B.cam_pos; M.F("cam_quat") = B.cam_quat; M.F("cam_fovy") = B.cam_fovy;
  M.names[MJB_OBJ_CAMERA] = B.cam_name;
  M.names[MJB_OBJ_BODY] = B.body_name; M.names[MJB_OBJ_JOINT] = B.jnt_name; M.names[MJB_OBJ_GEOM] = B.geom_name;
  M.names[MJB_OBJ_SITE] = B.site_name; M.names[MJB_OBJ_SENSOR] = B.sensor_name; M.names[MJB_OBJ_ACTUATOR] = B.act_name;

  // ---- qpos0-dependent constants: body_invweight0 / dof_invweight0 (MuJoCo's set-constants pass)
  M.pack();
  std::vector<double> body_invweight0(2 * nbody, 0.0), dof_invweight0(nv, 0.0);
  if (nv > 0) {
    ModelView mv(M.blob.data(), /*need_invweight=*/false);
    HostKin kin;
    host_fk(mv, qpos0.data(), kin);
    std::vector<double> Mm;
    host_mass_matrix(mv, kin, Mm);
    std::vector<double> L = Mm;
    if (!host_cholesky(L, nv)) throw std::runtime_error("MJCF: mass matrix at qpos0 is not positive definite");
    // Minv columns
    std::vector<double> Minv((size_t)nv * nv, 0.0), col(nv);
    for (int c = 0; c < nv; c++) {
      std::fill(col.begin(), col.end(), 0.0);
      col[c] = 1;
      host_chol_solve(L, nv, col.data());
      for (int r = 0; r < nv; r++) Minv[(size_t)r * nv + c] = col[r];
    }
    std::vector<double> jp, jr;
    for (int b = 1; b < nbody; b++) {
      if (body_mass[b] < 1e-15 || body_treeid[b] < 0) continue;
      host_jac(mv, kin, b, kin.xipos[b], jp, jr);
      double tran = 0, rot = 0;
      for (int r = 0; r < 3; r++)
        for (int i = 0; i < nv; i++)
          for (int j = 0; j < nv; j++) {
            tran += jp[r * nv + i] * Minv[(size_t)i * nv + j] * jp[r * nv + j];
            rot += jr[r * nv + i] * Minv[(size_t)i * nv + j] * jr[r * nv + j];
          }
      body_invweight0[2 * b] = std::max(1e-15, tran / 3);
      body_invweight0[2 * b + 1] = std::max(1e-15, rot / 3);
    }
    for (int j = 0; j < njnt; j++) {
      int da = jnt_dofadr[j];
      if (B.jnt_type[j] == MJB_JNT_FREE) {
        double t = 0, r = 0;
        for (int i = 0; i < 3; i++) { t += Minv[(size_t)(da + i) * nv + da + i]; r += Minv[(size_t)(da + 3 + i) * nv + da + 3 + i]; }
        for (int i = 0; i < 3; i++) { dof_invweight0[da + i] = t / 3; dof_invweight0[da + 3 + i] = r / 3; }
      } else {
        dof_invweight0[da] = Minv[(size_t)da * nv + da];
      }
    }
  }
  M.F("body_invweight0") = body_invweight0;
  M.F("dof_invweight0") = dof_invweight0;
  M.pack();
}

}  // namespace mjb
