// Host-side MJCF reader + planar flattener (see mjcf_flatten.h).
#include "mjcf_flatten.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <memory>
#include <sstream>
#include <vector>

#include "planar_engine.cuh"

namespace cassie {
namespace {

// ------------------------------------------------------------------ tolerant XML subset
// The reference model files are not well-formed (comments closed by '--->',
// cassie2d_stiff.xml:69,73), so this is a small hand parser: elements, attributes in single
// or double quotes, comments, self-closing tags.  No entities, no CDATA, no text nodes.
struct XmlNode {
  std::string tag;
  std::map<std::string, std::string> attr;
  std::vector<std::unique_ptr<XmlNode>> kids;
  const XmlNode* child(const char* t) const {
    for (auto& k : kids) if (k->tag == t) return k.get();
    return nullptr;
  }
  bool has(const char* a) const { return attr.count(a) > 0; }
  std::string get(const char* a, const std::string& d = "") const {
    auto it = attr.find(a);
    return it == attr.end() ? d : it->second;
  }
};

struct XmlParser {
  const std::string& s;
  size_t i = 0;
  std::string err;
  explicit XmlParser(const std::string& str) : s(str) {}
  void skip_ws() { while (i < s.size() && isspace((unsigned char)s[i])) i++; }
  bool skip_misc() {  // whitespace, comments, <?...?>, <!DOCTYPE>
    for (;;) {
      skip_ws();
      if (s.compare(i, 4, "<!--") == 0) {
        size_t e = s.find("-->", i + 4);
        if (e == std::string::npos) { err = "unterminated comment"; return false; }
        i = e + 3;
      } else if (s.compare(i, 2, "<?") == 0) {
        size_t e = s.find("?>", i);
        if (e == std::string::npos) { err = "unterminated <?"; return false; }
        i = e + 2;
      } else if (s.compare(i, 2, "<!") == 0) {
        size_t e = s.find('>', i);
        if (e == std::string::npos) { err = "unterminated <!"; return false; }
        i = e + 1;
      } else
        return true;
    }
  }
  std::unique_ptr<XmlNode> element() {
    if (!skip_misc()) return nullptr;
    if (i >= s.size() || s[i] != '<') { err = "expected '<' at offset " + std::to_string(i); return nullptr; }
    i++;
    auto n = std::make_unique<XmlNode>();
    while (i < s.size() && (isalnum((unsigned char)s[i]) || s[i] == '_' || s[i] == '-' || s[i] == ':')) n->tag += s[i++];
    if (n->tag.empty()) { err = "empty tag at offset " + std::to_string(i); return nullptr; }
    for (;;) {
      skip_ws();
      if (i >= s.size()) { err = "eof in tag <" + n->tag; return nullptr; }
      if (s[i] == '/') {
        if (i + 1 < s.size() && s[i + 1] == '>') { i += 2; return n; }
        err = "stray '/' in <" + n->tag; return nullptr;
      }
      if (s[i] == '>') { i++; break; }
      std::string key;
      while (i < s.size() && s[i] != '=' && !isspace((unsigned char)s[i]) && s[i] != '>' && s[i] != '/') key += s[i++];
      skip_ws();
      if (i >= s.size() || s[i] != '=') { err = "attribute '" + key + "' without value in <" + n->tag; return nullptr; }
      i++;
      skip_ws();
      if (i >= s.size() || (s[i] != '\'' && s[i] != '"')) { err = "unquoted attribute '" + key + "'"; return nullptr; }
      const char qc = s[i++];
      size_t e = s.find(qc, i);
      if (e == std::string::npos) { err = "unterminated attribute '" + key + "'"; return nullptr; }
      n->attr[key] = s.substr(i, e - i);
      i = e + 1;
    }
    for (;;) {  // children until the closing tag
      if (!skip_misc()) return nullptr;
      if (i >= s.size()) { err = "eof inside <" + n->tag + ">"; return nullptr; }
      if (s.compare(i, 2, "</") == 0) {
        size_t e = s.find('>', i);
        if (e == std::string::npos) { err = "unterminated closing tag"; return nullptr; }
        i = e + 1;
        return n;
      }
      if (s[i] != '<') {  // text content: ignore
        while (i < s.size() && s[i] != '<') i++;
        continue;
      }
      auto k = element();
      if (!k) return nullptr;
      n->kids.push_back(std::move(k));
    }
  }
};

bool parse_doubles(const std::string& str, int n, double* out) {
  std::istringstream is(str);
  for (int i = 0; i < n; i++)
    if (!(is >> out[i])) return false;
  return true;
}

// ------------------------------------------------------------------ 3-D intermediate model
struct V3 { double x = 0, y = 0, z = 0; };
struct M3 { double m[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}; };
V3 operator+(V3 a, V3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
V3 operator-(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
V3 operator*(double s, V3 a) { return {s * a.x, s * a.y, s * a.z}; }
double dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
V3 cross(V3 a, V3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
V3 normalized(V3 a) { double n = std::sqrt(dot(a, a)); return (1.0 / n) * a; }
V3 mul(const M3& A, V3 v) {
  return {A.m[0] * v.x + A.m[1] * v.y + A.m[2] * v.z, A.m[3] * v.x + A.m[4] * v.y + A.m[5] * v.z,
          A.m[6] * v.x + A.m[7] * v.y + A.m[8] * v.z};
}
V3 tmul(const M3& A, V3 v) {
  return {A.m[0] * v.x + A.m[3] * v.y + A.m[6] * v.z, A.m[1] * v.x + A.m[4] * v.y + A.m[7] * v.z,
          A.m[2] * v.x + A.m[5] * v.y + A.m[8] * v.z};
}
M3 mul(const M3& A, const M3& B) {
  M3 R;
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++)
      R.m[3 * i + j] = A.m[3 * i] * B.m[j] + A.m[3 * i + 1] * B.m[3 + j] + A.m[3 * i + 2] * B.m[6 + j];
  return R;
}
M3 transpose(const M3& A) {
  M3 R;
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) R.m[3 * i + j] = A.m[3 * j + i];
  return R;
}
M3 from_columns(V3 x, V3 y, V3 z) {
  M3 R;
  R.m[0] = x.x; R.m[3] = x.y; R.m[6] = x.z;
  R.m[1] = y.x; R.m[4] = y.y; R.m[7] = y.z;
  R.m[2] = z.x; R.m[5] = z.y; R.m[8] = z.z;
  return R;
}
M3 axis_angle(V3 a, double ang) {
  const double c = std::cos(ang), s = std::sin(ang), t = 1 - c;
  M3 R;
  R.m[0] = t * a.x * a.x + c;       R.m[1] = t * a.x * a.y - s * a.z; R.m[2] = t * a.x * a.z + s * a.y;
  R.m[3] = t * a.x * a.y + s * a.z; R.m[4] = t * a.y * a.y + c;       R.m[5] = t * a.y * a.z - s * a.x;
  R.m[6] = t * a.x * a.z - s * a.y; R.m[7] = t * a.y * a.z + s * a.x; R.m[8] = t * a.z * a.z + c;
  return R;
}

struct Joint3 {
  std::string name;
  bool hinge = true, limited = false, free = false;
  V3 axis{0, 0, 1}, pos;
  double ref = 0, lo = 0, hi = 0, damping = 0, armature = 0;
  double solref[2] = {0.02, 1}, solimp[5] = {0.9, 0.95, 0.001, 0.5, 2};
};
struct Geom3 {
  int type = 0;  // 0 plane 2 sphere 3 capsule
  V3 pos, from, to;
  double radius = 0;
  int contype = 1, conaffinity = 1, condim = 3;
  double friction[3] = {1, 0.005, 0.0001}, solref[2] = {0.02, 1}, solimp[5] = {0.9, 0.95, 0.001, 0.5, 2};
};
struct Site3 { std::string name; V3 pos; };
struct Body3 {
  std::string name;
  int parent = 0;
  V3 pos, ipos;
  M3 mat;
  double mass = 0, I[6] = {0, 0, 0, 0, 0, 0};
  std::vector<Joint3> joints;
  std::vector<Geom3> geoms;
  std::vector<Site3> sites;
};
struct Connect3 { int b1 = 0, b2 = 0; V3 anchor; double solref[2] = {0.02, 1}, solimp[5] = {0.9, 0.95, 0.001, 0.5, 2}; };
struct Motor3 { std::string joint; double gear = 1, lo = 0, hi = 0; bool limited = false; };
struct Model3 {
  std::vector<Body3> bodies;  // [0] = world
  std::vector<Connect3> connects;
  std::vector<Motor3> motors;
  double timestep = 0.002, tolerance = 1e-8, impratio = 1, gravity[3] = {0, 0, -9.81};
  int iterations = 100;
  std::string cone = "pyramidal", solver = "Newton";
};

struct Defaults { const XmlNode* joint = nullptr; const XmlNode* geom = nullptr; const XmlNode* motor = nullptr; };

std::string dattr(const XmlNode& e, const XmlNode* d, const char* name, const std::string& fallback) {
  if (e.has(name)) return e.get(name);
  if (d && d->has(name)) return d->get(name);
  return fallback;
}

void read_solimp(const std::string& s, double out[5]) {
  double v[5] = {0.9, 0.95, 0.001, 0.5, 2};  // 3-parameter (MuJoCo 1.50) input keeps midpoint .5, power 2
  std::istringstream is(s);
  for (int i = 0; i < 5; i++) { double x; if (is >> x) v[i] = x; else break; }
  for (int i = 0; i < 5; i++) out[i] = v[i];
}

bool read_geom(const XmlNode& g, const Defaults& df, Geom3* out, bool* skip, std::string* err) {
  const std::string type = dattr(g, df.geom, "type", "sphere");
  *skip = false;
  if (type == "mesh") { *skip = true; return true; }
  out->contype = atoi(dattr(g, df.geom, "contype", "1").c_str());
  out->conaffinity = atoi(dattr(g, df.geom, "conaffinity", "1").c_str());
  out->condim = atoi(dattr(g, df.geom, "condim", "3").c_str());
  parse_doubles(dattr(g, df.geom, "friction", "1 0.005 0.0001"), 3, out->friction);
  parse_doubles(dattr(g, df.geom, "solref", "0.02 1"), 2, out->solref);
  read_solimp(dattr(g, df.geom, "solimp", "0.9 0.95 0.001"), out->solimp);
  double sz[3] = {0, 0, 0};
  parse_doubles(dattr(g, df.geom, "size", "0"), 1, sz);
  double p[3] = {0, 0, 0};
  parse_doubles(dattr(g, df.geom, "pos", "0 0 0"), 3, p);
  out->pos = {p[0], p[1], p[2]};
  if (type == "plane") out->type = 0;
  else if (type == "sphere") { out->type = 2; out->radius = sz[0]; }
  else if (type == "capsule") {
    out->type = 3; out->radius = sz[0];
    double ft[6];
    if (!g.has("fromto") || !parse_doubles(g.get("fromto"), 6, ft)) { *err = "capsule without fromto"; return false; }
    out->from = {ft[0], ft[1], ft[2]};
    out->to = {ft[3], ft[4], ft[5]};
  } else { *err = "unsupported geom type '" + type + "'"; return false; }
  return true;
}

bool read_body(const XmlNode& e, int parent, const Defaults& df, double ang, Model3* M, std::string* err) {
  Body3 b;
  b.name = e.get("name");
  b.parent = parent;
  double p[3] = {0, 0, 0};
  if (e.has("pos") && !parse_doubles(e.get("pos"), 3, p)) { *err = "bad body pos"; return false; }
  b.pos = {p[0], p[1], p[2]};
  if (e.has("xyaxes")) {
    double a[6];
    if (!parse_doubles(e.get("xyaxes"), 6, a)) { *err = "bad xyaxes"; return false; }
    V3 x = normalized({a[0], a[1], a[2]});
    V3 y{a[3], a[4], a[5]};
    y = normalized(y - dot(x, y) * x);  // MuJoCo: Gram-Schmidt [EXT]
    b.mat = from_columns(x, y, cross(x, y));
  }
  if (const XmlNode* in = e.child("inertial")) {
    double ip[3], fi[6];
    if (!parse_doubles(in->get("pos"), 3, ip) || !in->has("mass") || !parse_doubles(in->get("fullinertia"), 6, fi)) {
      *err = "inertial needs pos, mass, fullinertia (body " + b.name + ")";
      return false;
    }
    b.ipos = {ip[0], ip[1], ip[2]};
    b.mass = atof(in->get("mass").c_str());
    for (int i = 0; i < 6; i++) b.I[i] = fi[i];
  }
  for (auto& k : e.kids) {
    if (k->tag == "joint") {
      Joint3 j;
      j.name = k->get("name");
      const std::string type = dattr(*k, df.joint, "type", "hinge");
      if (type != "hinge" && type != "slide" && type != "free") { *err = "unsupported joint type '" + type + "'"; return false; }
      j.hinge = type == "hinge";
      j.free = type == "free";
      double a[3] = {0, 0, 1}, jp[3] = {0, 0, 0}, rg[2] = {0, 0};
      parse_doubles(dattr(*k, df.joint, "axis", "0 0 1"), 3, a);
      parse_doubles(dattr(*k, df.joint, "pos", "0 0 0"), 3, jp);
      parse_doubles(dattr(*k, df.joint, "range", "0 0"), 2, rg);
      j.axis = normalized({a[0], a[1], a[2]});
      j.pos = {jp[0], jp[1], jp[2]};
      const double sc = j.hinge ? ang : 1.0;
      j.ref = atof(dattr(*k, df.joint, "ref", "0").c_str()) * sc;
      j.lo = rg[0] * sc; j.hi = rg[1] * sc;
      j.limited = dattr(*k, df.joint, "limited", "false") == "true";
      j.damping = atof(dattr(*k, df.joint, "damping", "0").c_str());
      j.armature = atof(dattr(*k, df.joint, "armature", "0").c_str());
      parse_doubles(dattr(*k, df.joint, "solreflimit", "0.02 1"), 2, j.solref);
      read_solimp(dattr(*k, df.joint, "solimplimit", "0.9 0.95 0.001"), j.solimp);
      b.joints.push_back(j);
    } else if (k->tag == "geom") {
      Geom3 g; bool skip;
      if (!read_geom(*k, df, &g, &skip, err)) return false;
      if (!skip) b.geoms.push_back(g);
    } else if (k->tag == "site") {
      Site3 s;
      s.name = k->get("name");
      double sp[3] = {0, 0, 0};
      parse_doubles(k->get("pos", "0 0 0"), 3, sp);
      s.pos = {sp[0], sp[1], sp[2]};
      b.sites.push_back(s);
    }
  }
  const int id = (int)M->bodies.size();
  M->bodies.push_back(b);
  for (auto& k : e.kids)
    if (k->tag == "body" && !read_body(*k, id, df, ang, M, err)) return false;
  return true;
}

bool read_model3(const std::string& xml, Model3* M, std::string* err) {
  XmlParser P(xml);
  auto root = P.element();
  if (!root) { *err = "XML: " + P.err; return false; }
  if (root->tag != "mujoco") { *err = "root element is not <mujoco>"; return false; }
  double ang = M_PI / 180.0;
  if (const XmlNode* c = root->child("compiler"))
    if (c->get("angle", "degree") == "radian") ang = 1.0;
  if (const XmlNode* o = root->child("option")) {
    if (o->has("timestep")) M->timestep = atof(o->get("timestep").c_str());
    if (o->has("iterations")) M->iterations = atoi(o->get("iterations").c_str());
    if (o->has("tolerance")) M->tolerance = atof(o->get("tolerance").c_str());
    if (o->has("impratio")) M->impratio = atof(o->get("impratio").c_str());
    if (o->has("gravity")) parse_doubles(o->get("gravity"), 3, M->gravity);
    M->cone = o->get("cone", M->cone);
    M->solver = o->get("solver", M->solver);
    if (o->has("integrator") && o->get("integrator") != "Euler") { *err = "only the Euler integrator is supported"; return false; }
  }
  Defaults df;
  if (const XmlNode* d = root->child("default")) { df.joint = d->child("joint"); df.geom = d->child("geom"); df.motor = d->child("motor"); }
  const XmlNode* wb = root->child("worldbody");
  if (!wb) { *err = "no <worldbody>"; return false; }
  Body3 world;
  world.name = "world";
  for (auto& k : wb->kids)
    if (k->tag == "geom") {
      Geom3 g; bool skip;
      if (!read_geom(*k, df, &g, &skip, err)) return false;
      if (!skip) world.geoms.push_back(g);
    }
  M->bodies.push_back(world);
  for (auto& k : wb->kids)
    if (k->tag == "body" && !read_body(*k, 0, df, ang, M, err)) return false;
  auto body_id = [&](const std::string& n) { for (size_t i = 0; i < M->bodies.size(); i++) if (M->bodies[i].name == n) return (int)i; return -1; };
  if (const XmlNode* eq = root->child("equality"))
    for (auto& k : eq->kids) {
      if (k->tag != "connect") { *err = "unsupported equality '" + k->tag + "'"; return false; }
      Connect3 c;
      c.b1 = body_id(k->get("body1")); c.b2 = body_id(k->get("body2"));
      double a[3];
      if (c.b1 < 0 || c.b2 < 0 || !parse_doubles(k->get("anchor"), 3, a)) { *err = "bad <connect>"; return false; }
      c.anchor = {a[0], a[1], a[2]};
      parse_doubles(k->get("solref", "0.02 1"), 2, c.solref);
      read_solimp(k->get("solimp", "0.9 0.95 0.001"), c.solimp);
      M->connects.push_back(c);
    }
  if (const XmlNode* ac = root->child("actuator"))
    for (auto& k : ac->kids) {
      if (k->tag != "motor") { *err = "unsupported actuator '" + k->tag + "'"; return false; }
      Motor3 mo;
      mo.joint = k->get("joint");
      mo.gear = atof(k->get("gear", "1").c_str());
      mo.limited = dattr(*k, df.motor, "ctrllimited", "false") == "true";
      double rg[2] = {0, 0};
      parse_doubles(k->get("ctrlrange", "0 0"), 2, rg);
      mo.lo = rg[0]; mo.hi = rg[1];
      M->motors.push_back(mo);
    }
  return true;
}

// ------------------------------------------------------------------ 3-D forward kinematics
struct Pose3 { std::vector<V3> xpos; std::vector<M3> xmat; };
struct JointRef { int body, idx; };

void fk3(const Model3& M, const std::vector<JointRef>& jr, const std::vector<double>& q, Pose3* P) {
  const size_t nb = M.bodies.size();
  P->xpos.assign(nb, V3{});
  P->xmat.assign(nb, M3{});
  for (size_t b = 1; b < nb; b++) {
    const Body3& B = M.bodies[b];
    V3 pos = P->xpos[B.parent] + mul(P->xmat[B.parent], B.pos);
    M3 mat = mul(P->xmat[B.parent], B.mat);
    for (size_t d = 0; d < jr.size(); d++) {
      if (jr[d].body != (int)b) continue;
      const Joint3& J = B.joints[jr[d].idx];
      const V3 ax = mul(mat, J.axis);
      if (J.hinge) {
        const V3 an = pos + mul(mat, J.pos);
        const M3 R = axis_angle(ax, q[d] - J.ref);
        pos = an + mul(R, pos - an);
        mat = mul(R, mat);
      } else
        pos = pos + (q[d] - J.ref) * ax;
    }
    P->xpos[b] = pos;
    P->xmat[b] = mat;
  }
}

struct V2 { double x, z; };
V2 xz(V3 v) { return {v.x, v.z}; }

// ------------------------------------------------------------------ flatten one 3-D model
// `anchor_q` = configuration at which the connect's second anchor is made to coincide with the
// first (qpos0 of the ORIGINAL file for both variants, DynamicModel.cpp:141-167).
bool flatten(const Model3& M, const std::vector<double>& anchor_q, PlanarModel<double>* out, std::string* err) {
  PlanarModel<double>& m = *out;
  std::memset(&m, 0, sizeof(m));
  const int nb = (int)M.bodies.size();
  // dof list in file order
  std::vector<JointRef> jr;
  for (int b = 1; b < nb; b++)
    for (size_t j = 0; j < M.bodies[b].joints.size(); j++) jr.push_back({b, (int)j});
  if ((int)jr.size() != kNV) { *err = "expected 13 joints, found " + std::to_string(jr.size()); return false; }
  for (auto& r : jr)
    if (M.bodies[r.body].joints[r.idx].free) { *err = "free joint: not a planar model (use the tree engine)"; return false; }
  auto J = [&](int d) -> const Joint3& { return M.bodies[jr[d].body].joints[jr[d].idx]; };
  // link of each body: bodies without joints are welded to the parent's link
  std::vector<int> link_root(nb, 0);  // body that owns the link
  for (int b = 1; b < nb; b++) link_root[b] = M.bodies[b].joints.empty() ? link_root[M.bodies[b].parent] : b;
  const int pelvis = jr[0].body;
  if (jr[1].body != pelvis || jr[2].body != pelvis || M.bodies[pelvis].joints.size() != 3 || M.bodies[pelvis].parent != 0) {
    *err = "expected a root body with exactly three joints (slide x, slide z, hinge y)"; return false;
  }
  // leg link bodies, dof d = 3 + 5L + a
  int lb[2][kLegLinks];
  for (int L = 0; L < 2; L++)
    for (int a = 0; a < kLegLinks; a++) {
      const int d = 3 + 5 * L + a;
      lb[L][a] = jr[d].body;
      if (M.bodies[lb[L][a]].joints.size() != 1 || !J(d).hinge) { *err = "leg joint " + J(d).name + ": expected one hinge per body"; return false; }
    }
  for (int L = 0; L < 2; L++)
    for (int a = 0; a < kLegLinks; a++) {
      const int want = a == kThigh ? pelvis : lb[L][link_parent(a)];
      if (link_root[M.bodies[lb[L][a]].parent] != want) { *err = "unexpected kinematic tree at joint " + J(3 + 5 * L + a).name; return false; }
    }
  // qpos0 pose
  std::vector<double> q0(kNV);
  for (int d = 0; d < kNV; d++) q0[d] = J(d).ref;
  Pose3 P0;
  fk3(M, jr, q0, &P0);
  auto world_axis = [&](int d) { return mul(P0.xmat[jr[d].body], J(d).axis); };
  const double tol = 1e-9;
  {
    const V3 a0 = world_axis(0), a1 = world_axis(1), a2 = world_axis(2);
    if (J(0).hinge || J(1).hinge || !J(2).hinge || std::fabs(a0.x - 1) > tol || std::fabs(a1.z - 1) > tol || std::fabs(a2.y - 1) > tol) {
      *err = "root joints must be slide +x, slide +z, hinge +y"; return false;
    }
  }
  auto pivot = [&](int d) { return P0.xpos[jr[d].body] + mul(P0.xmat[jr[d].body], J(d).pos); };
  const V3 piv0 = pivot(2);
  m.pel_org[0] = piv0.x; m.pel_org[1] = piv0.z;
  for (int i = 0; i < 3; i++) m.pel_ref[i] = J(i).ref;
  // composite inertia of a link = all bodies whose link_root is the link's body
  auto composite = [&](int root, V3 piv, double* com2, double* mass, double* inertia) {
    double mt = 0; V3 c{};
    for (int b = 1; b < nb; b++) if (link_root[b] == root) {
      const V3 cb = P0.xpos[b] + mul(P0.xmat[b], M.bodies[b].ipos);
      mt += M.bodies[b].mass; c = c + M.bodies[b].mass * cb;
    }
    c = (1.0 / mt) * c;
    double I = 0;
    for (int b = 1; b < nb; b++) if (link_root[b] == root) {
      const Body3& B = M.bodies[b];
      M3 Ib; Ib.m[0] = B.I[0]; Ib.m[4] = B.I[1]; Ib.m[8] = B.I[2];
      Ib.m[1] = Ib.m[3] = B.I[3]; Ib.m[2] = Ib.m[6] = B.I[4]; Ib.m[5] = Ib.m[7] = B.I[5];
      const M3 Iw = mul(mul(P0.xmat[b], Ib), transpose(P0.xmat[b]));
      const V3 cb = P0.xpos[b] + mul(P0.xmat[b], B.ipos);
      const double dx = cb.x - c.x, dz = cb.z - c.z;
      I += Iw.m[4] + B.mass * (dx * dx + dz * dz);
    }
    com2[0] = c.x - piv.x; com2[1] = c.z - piv.z; *mass = mt; *inertia = I;
  };
  composite(pelvis, piv0, m.pel_com, &m.pel_mass, &m.pel_inertia);
  m.total_mass = m.pel_mass;
  for (int L = 0; L < 2; L++)
    for (int a = 0; a < kLegLinks; a++) {
      const int d = 3 + 5 * L + a;
      const V3 ax = world_axis(d);
      if (std::fabs(std::fabs(ax.y) - 1) > tol) { *err = "hinge " + J(d).name + " is not about the world y axis"; return false; }
      m.sgn[L][a] = ax.y > 0 ? 1.0 : -1.0;
      m.ang0[L][a] = -m.sgn[L][a] * J(d).ref;
      const V3 pv = pivot(d);
      const V3 pp = a == kThigh ? piv0 : pivot(3 + 5 * L + link_parent(a));
      m.off[L][a][0] = pv.x - pp.x; m.off[L][a][1] = pv.z - pp.z;
      composite(lb[L][a], pv, m.com[L][a], &m.mass[L][a], &m.inertia[L][a]);
      m.total_mass += m.mass[L][a];
    }
  for (int d = 0; d < kNV; d++) {
    m.damping[d] = J(d).damping; m.armature[d] = J(d).armature;
    m.has_limit[d] = J(d).limited ? 1 : 0;
    m.lim_lo[d] = J(d).lo; m.lim_hi[d] = J(d).hi;
    if (J(d).limited && d < 3) { *err = "limited root joints are not supported"; return false; }
    if (J(d).limited) {
      for (int i = 0; i < 2; i++) m.lim_solref[i] = J(d).solref[i];
      for (int i = 0; i < 5; i++) m.lim_solimp[i] = J(d).solimp[i];
    }
  }
  if (m.lim_solref[0] == 0) { m.lim_solref[0] = 0.02; m.lim_solref[1] = 1; double si[5] = {0.9, 0.95, 0.001, 0.5, 2}; for (int i = 0; i < 5; i++) m.lim_solimp[i] = si[i]; }
  // actuators
  if ((int)M.motors.size() != kNU) { *err = "expected 6 motors"; return false; }
  for (int a = 0; a < kNU; a++) {
    int d = -1;
    for (int i = 0; i < kNV; i++) if (J(i).name == M.motors[a].joint) d = i;
    if (d < 3) { *err = "motor on unknown or root joint '" + M.motors[a].joint + "'"; return false; }
    m.act_dof[a] = d; m.act_gear[a] = M.motors[a].gear;
    m.act_lo[a] = M.motors[a].limited ? M.motors[a].lo : -1e30;
    m.act_hi[a] = M.motors[a].limited ? M.motors[a].hi : 1e30;
  }
  // sites in file order (xml_parser.h:151-163)
  {
    int ns = 0;
    for (int b = 1; b < nb; b++)
      for (auto& s : M.bodies[b].sites) {
        if (ns >= kNumSites) { *err = "more than 6 sites"; return false; }
        const int root = link_root[b];
        int link = -2; V3 pv = piv0;
        if (root == pelvis) link = -1;
        for (int L = 0; L < 2; L++) for (int a = 0; a < kLegLinks; a++) if (lb[L][a] == root) { link = 5 * L + a; pv = pivot(3 + link); }
        if (link == -2) { *err = "site on unknown link"; return false; }
        const V3 w = P0.xpos[b] + mul(P0.xmat[b], s.pos);
        m.site_link[ns] = link; m.site_off[ns][0] = w.x - pv.x; m.site_off[ns][1] = w.z - pv.z;
        ns++;
      }
    if (ns != kNumSites) { *err = "expected 6 sites, found " + std::to_string(ns); return false; }
  }
  // geoms: floor plane in the world body, pelvis sphere, four capsules per leg
  const Geom3* floor = nullptr;
  for (auto& g : M.bodies[0].geoms) if (g.type == 0) floor = &g;
  if (!floor) { *err = "no floor plane"; return false; }
  auto collides = [&](const Geom3& g) { return (floor->contype & g.conaffinity) || (g.contype & floor->conaffinity); };
  bool have_sphere = false;
  int ncap[2] = {0, 0};
  const Geom3* any = nullptr;
  std::vector<int> cap_body(kNumCaps, -1);
  int sph_body = -1;
  for (int b = 1; b < nb; b++)
    for (auto& g : M.bodies[b].geoms) {
      if (!collides(g)) continue;
      any = &g;
      const int root = link_root[b];
      if (g.type == 2) {
        if (root != pelvis || have_sphere) { *err = "only one colliding sphere on the pelvis is supported"; return false; }
        const V3 w = P0.xpos[b] + mul(P0.xmat[b], g.pos);
        m.sph_c[0] = w.x - piv0.x; m.sph_c[1] = w.z - piv0.z; m.sph_r = g.radius; have_sphere = true; sph_body = b;
      } else if (g.type == 3) {
        int L = -1, a = -1;
        for (int l = 0; l < 2; l++) for (int x = 0; x < kLegLinks; x++) if (lb[l][x] == root) { L = l; a = x; }
        if (L < 0 || a != ncap[L] || a > kToe) { *err = "colliding capsules must be, per leg, on thigh, knee(shin), tarsus, toe in this order"; return false; }
        const int c = 4 * L + a;
        const V3 pv = pivot(3 + 5 * L + a);
        const V3 wt = P0.xpos[b] + mul(P0.xmat[b], g.to), wf = P0.xpos[b] + mul(P0.xmat[b], g.from);
        m.cap_link[c] = a;
        m.cap_to[c][0] = wt.x - pv.x; m.cap_to[c][1] = wt.z - pv.z;
        m.cap_from[c][0] = wf.x - pv.x; m.cap_from[c][1] = wf.z - pv.z;
        m.cap_r[c] = g.radius; cap_body[c] = b;
        ncap[L]++;
      } else { *err = "unsupported colliding geom"; return false; }
    }
  if (!have_sphere || ncap[0] != 4 || ncap[1] != 4) { *err = "expected pelvis sphere + 4 capsules per leg"; return false; }
  // contact parameter mixing floor x geom [EXT mj_contactParam]: max condim / friction, equal solref/solimp
  {
    const int condim = floor->condim > any->condim ? floor->condim : any->condim;
    if (condim != 3) { *err = "floor contacts must be condim 3"; return false; }
    if (M.cone != "elliptic" || M.solver != "PGS") { *err = "only solver=PGS cone=elliptic is implemented"; return false; }
    m.con_mu = floor->friction[0] > any->friction[0] ? floor->friction[0] : any->friction[0];
    for (int i = 0; i < 2; i++) m.con_solref[i] = 0.5 * (floor->solref[i] + any->solref[i]);
    for (int i = 0; i < 5; i++) m.con_solimp[i] = 0.5 * (floor->solimp[i] + any->solimp[i]);
  }
  // connects: rod anchor <-> tarsus link, one per leg, in leg order
  if (M.connects.size() != 2) { *err = "expected two <connect> constraints"; return false; }
  Pose3 PA;
  fk3(M, jr, anchor_q, &PA);
  int eq_b1[2], eq_b2[2];
  for (int L = 0; L < 2; L++) {
    const Connect3& c = M.connects[L];
    if (link_root[c.b1] != lb[L][kRod] || link_root[c.b2] != lb[L][kTarsus]) { *err = "connect must join the rod to the tarsus link of the same leg"; return false; }
    eq_b1[L] = c.b1; eq_b2[L] = c.b2;
    // anchor 1 in the rod zero frame
    const V3 w1 = P0.xpos[c.b1] + mul(P0.xmat[c.b1], c.anchor);
    const V3 pr = pivot(3 + 5 * L + kRod), pt = pivot(3 + 5 * L + kTarsus);
    m.eq_a1[L][0] = w1.x - pr.x; m.eq_a1[L][1] = w1.z - pr.z;
    // anchor 2: body-2 local coordinates of anchor 1 at `anchor_q`, then into the zero frame
    const V3 wa = PA.xpos[c.b1] + mul(PA.xmat[c.b1], c.anchor);
    const V3 a2 = tmul(PA.xmat[c.b2], wa - PA.xpos[c.b2]);
    const V3 w2 = P0.xpos[c.b2] + mul(P0.xmat[c.b2], a2);
    m.eq_a2[L][0] = w2.x - pt.x; m.eq_a2[L][1] = w2.z - pt.z;
    for (int i = 0; i < 2; i++) m.eq_solref[i] = c.solref[i];
    for (int i = 0; i < 5; i++) m.eq_solimp[i] = c.solimp[i];
  }
  m.timestep = M.timestep; m.gravity_z = M.gravity[2]; m.tolerance = M.tolerance; m.impratio = M.impratio;
  m.iterations = M.iterations;
  if (M.gravity[0] != 0 || M.gravity[1] != 0) { *err = "gravity must be along z"; return false; }

  // ---- invweight0 / meaninertia at qpos0 (mj_setConst [EXT]); planar: tran = (Axx + Azz)/3
  {
    double qd0[kNV] = {0};
    Kin<double> k;
    forward_kinematics(m, q0.data(), qd0, k);
    double Mm[kNV][kNV], Dinv[kNV];
    std::memset(Mm, 0, sizeof(Mm));
    mass_matrix(m, k, Mm);
    double tr = 0;
    for (int i = 0; i < kNV; i++) tr += Mm[i][i];
    m.meaninertia = tr / kNV;
    factor(Mm, Dinv);
    for (int d = 0; d < kNV; d++) {
      double e[kNV] = {0};
      e[d] = 1;
      solve(Mm, Dinv, e);
      m.lim_diag[d] = e[d];
    }
    auto body_tran = [&](int b) {
      const int root = link_root[b];
      int L = 0, a = -1;
      for (int l = 0; l < 2; l++) for (int x = 0; x < kLegLinks; x++) if (lb[l][x] == root) { L = l; a = x; }
      const V3 cb = P0.xpos[b] + mul(P0.xmat[b], M.bodies[b].ipos);
      double Jx[8], Jz[8], x[kNV];
      const double lpx = a >= 0 ? k.px[L][a] : 0.0, lpz = a >= 0 ? k.pz[L][a] : 0.0;
      point_jac(m, k, L, a, cb.x - piv0.x - lpx, cb.z - piv0.z - lpz, Jx, Jz);
      double s = 0;
      expand_row(Jx, L, x); solve(Mm, Dinv, x); s += dot8_dense(Jx, L, x);
      expand_row(Jz, L, x); solve(Mm, Dinv, x); s += dot8_dense(Jz, L, x);
      s /= 3.0;
      return s > kMinVal ? s : kMinVal;
    };
    m.sph_diag = body_tran(sph_body);
    for (int c = 0; c < kNumCaps; c++) m.cap_diag[c] = body_tran(cap_body[c]);
    for (int L = 0; L < 2; L++) m.eq_diag[L] = body_tran(eq_b1[L]) + body_tran(eq_b2[L]);
  }
  return true;
}

}  // namespace

bool flatten_mjcf_text(const std::string& xml, FlatModels* out, std::string* err) {
  Model3 M;
  if (!read_model3(xml, &M, err)) return false;
  std::vector<double> q0;
  for (size_t b = 1; b < M.bodies.size(); b++)
    for (auto& j : M.bodies[b].joints) q0.push_back(j.ref);
  if (!flatten(M, q0, &out->phys, err)) return false;
  // RBDL-loader variant (DynamicModel.cpp:84-103): a body whose LAST joint has |ref| >= 1e-3
  // (degrees in the file) loses its xyaxes rotation and its joints lose their ref.
  // Not modelled: RBDL gets xyaxes normalised but not orthogonalised (DESIGN.md, known quirks).
  Model3 R = M;
  for (size_t b = 1; b < R.bodies.size(); b++) {
    Body3& B = R.bodies[b];
    if (B.joints.empty()) continue;
    const Joint3& last = B.joints.back();
    if (last.hinge && std::fabs(last.ref * 180.0 / M_PI) >= 1e-3) {
      B.mat = M3{};
      for (auto& j : B.joints) j.ref = 0.0;
    }
  }
  return flatten(R, q0, &out->ctrl, err);
}

bool flatten_mjcf_file(const std::string& path, FlatModels* out, std::string* err) {
  std::ifstream f(path);
  if (!f) { *err = "cannot open model file '" + path + "'"; return false; }
  std::stringstream ss;
  ss << f.rdbuf();
  return flatten_mjcf_text(ss.str(), out, err);
}

// ------------------------------------------------------------------ 3-D tree flattener (cassie3d_stiff.xml)
namespace {

struct Rigid { V3 p; M3 R; };
Rigid compose(const Rigid& a, const Rigid& b) { return {a.p + mul(a.R, b.p), mul(a.R, b.R)}; }

M3 full_inertia(const double I[6]) {
  M3 A;
  A.m[0] = I[0]; A.m[4] = I[1]; A.m[8] = I[2];
  A.m[1] = A.m[3] = I[3]; A.m[2] = A.m[6] = I[4]; A.m[5] = A.m[7] = I[5];
  return A;
}

void mat_to_quat(const M3& R, double q[4]) {
  const double* m = R.m;
  const double tr = m[0] + m[4] + m[8];
  if (tr > 0) {
    const double s = std::sqrt(tr + 1.0) * 2;
    q[0] = 0.25 * s; q[1] = (m[7] - m[5]) / s; q[2] = (m[2] - m[6]) / s; q[3] = (m[3] - m[1]) / s;
  } else if (m[0] > m[4] && m[0] > m[8]) {
    const double s = std::sqrt(1.0 + m[0] - m[4] - m[8]) * 2;
    q[0] = (m[7] - m[5]) / s; q[1] = 0.25 * s; q[2] = (m[1] + m[3]) / s; q[3] = (m[2] + m[6]) / s;
  } else if (m[4] > m[8]) {
    const double s = std::sqrt(1.0 + m[4] - m[0] - m[8]) * 2;
    q[0] = (m[2] - m[6]) / s; q[1] = (m[1] + m[3]) / s; q[2] = 0.25 * s; q[3] = (m[5] + m[7]) / s;
  } else {
    const double s = std::sqrt(1.0 + m[8] - m[0] - m[4]) * 2;
    q[0] = (m[3] - m[1]) / s; q[1] = (m[2] + m[6]) / s; q[2] = (m[5] + m[7]) / s; q[3] = 0.25 * s;
  }
}

// dense symmetric positive-definite inverse (Gauss-Jordan, n <= 24): init-time only
bool spd_inverse(int n, const std::vector<double>& A, std::vector<double>* Ainv) {
  std::vector<double> W(A);
  Ainv->assign((size_t)n * n, 0.0);
  for (int i = 0; i < n; i++) (*Ainv)[(size_t)i * n + i] = 1.0;
  for (int k = 0; k < n; k++) {
    const double piv = W[(size_t)k * n + k];
    if (!(piv > 1e-14)) return false;
    for (int j = 0; j < n; j++) { W[(size_t)k * n + j] /= piv; (*Ainv)[(size_t)k * n + j] /= piv; }
    for (int i = 0; i < n; i++) {
      if (i == k) continue;
      const double f = W[(size_t)i * n + k];
      if (f == 0) continue;
      for (int j = 0; j < n; j++) { W[(size_t)i * n + j] -= f * W[(size_t)k * n + j]; (*Ainv)[(size_t)i * n + j] -= f * (*Ainv)[(size_t)k * n + j]; }
    }
  }
  return true;
}

}  // namespace

bool flatten_tree(const Model3& M, tree::TreeModel<double>* out, std::string* err) {
  using namespace tree;
  TreeModel<double>& m = *out;
  std::memset(&m, 0, sizeof(m));
  const int nb = (int)M.bodies.size();
  // ---- links: one per jointed body; the free body first
  int base = -1;
  for (int b = 1; b < nb; b++)
    for (auto& j : M.bodies[b].joints)
      if (j.free) {
        if (base >= 0 || M.bodies[b].joints.size() != 1 || M.bodies[b].parent != 0) { *err = "expected exactly one free joint, alone on a child of the world"; return false; }
        base = b;
      }
  if (base < 0) { *err = "no free joint: not a floating-base model"; return false; }
  std::vector<int> owner(nb, -1), depth(nb, 0);   // body that owns the link a body belongs to; link depth
  std::vector<int> link_bodies;
  for (int b = 1; b < nb; b++) {
    const Body3& B = M.bodies[b];
    if (!B.joints.empty()) {
      if (b != base && (B.joints.size() != 1 || !B.joints[0].hinge)) { *err = "body " + B.name + ": expected one hinge per moving body"; return false; }
      owner[b] = b;
      depth[b] = B.parent == 0 ? 0 : depth[owner[B.parent]] + 1;
      if (b != base && B.parent == 0) { *err = "only the free body may hang on the world"; return false; }
      link_bodies.push_back(b);
    } else {
      if (B.parent == 0) { *err = "static bodies are not supported"; return false; }
      owner[b] = owner[B.parent];
    }
  }
  std::stable_sort(link_bodies.begin(), link_bodies.end(), [&](int a, int b) { return depth[a] < depth[b]; });
  const int nl = (int)link_bodies.size();
  if (nl > kMaxLinks || 5 + nl > kMaxDof) { *err = "too many links"; return false; }
  std::vector<int> link_of(nb, -1);
  for (int l = 0; l < nl; l++) link_of[link_bodies[l]] = l;
  for (int b = 1; b < nb; b++) link_of[b] = link_of[owner[b]];
  m.nl = nl; m.nv = 5 + nl; m.nq = 6 + nl;
  // ---- rigid placement of every body in its link frame
  std::vector<Rigid> in_link(nb);
  for (int b = 1; b < nb; b++) {
    const Body3& B = M.bodies[b];
    if (owner[b] == b) in_link[b] = Rigid{V3{}, M3{}};
    else in_link[b] = compose(in_link[B.parent], Rigid{B.pos, B.mat});
  }
  int nlev = 0;
  for (int l = 0; l < nl; l++) {
    const int b = link_bodies[l];
    const Body3& B = M.bodies[b];
    const int dl = depth[b];
    if (dl + 1 > kMaxLevels) { *err = "tree too deep"; return false; }
    if (dl + 1 > nlev) nlev = dl + 1;
    m.level_off[dl + 1] = l + 1;
    if (l == 0) {
      m.parent[0] = -1;
      m.anc[0] = 0x3fu;
      m.qpos0[0] = B.pos.x; m.qpos0[1] = B.pos.y; m.qpos0[2] = B.pos.z;
      mat_to_quat(B.mat, m.qpos0 + 3);
      m.lmat[0][0] = m.lmat[0][4] = m.lmat[0][8] = 1;
    } else {
      const int pl = link_of[B.parent];
      m.parent[l] = pl;
      m.anc[l] = m.anc[pl] | (1u << (5 + l));
      const Rigid X = compose(in_link[B.parent], Rigid{B.pos, B.mat});
      m.lpos[l][0] = X.p.x; m.lpos[l][1] = X.p.y; m.lpos[l][2] = X.p.z;
      for (int i = 0; i < 9; i++) m.lmat[l][i] = X.R.m[i];
      const Joint3& J = B.joints[0];
      m.axis[l][0] = J.axis.x; m.axis[l][1] = J.axis.y; m.axis[l][2] = J.axis.z;
      m.jpos[l][0] = J.pos.x; m.jpos[l][1] = J.pos.y; m.jpos[l][2] = J.pos.z;
      m.ref[l] = J.ref;
      m.qpos0[6 + l] = J.ref;
      const int d = 5 + l;
      m.damping[d] = J.damping; m.armature[d] = J.armature; m.limited[d] = J.limited ? 1 : 0;
      m.range[d][0] = J.lo; m.range[d][1] = J.hi;
      for (int k = 0; k < 2; k++) m.lim_solref[d][k] = J.solref[k];
      for (int k = 0; k < 5; k++) m.lim_solimp[d][k] = J.solimp[k];
    }
  }
  {  // MuJoCo numbers dofs in file (depth-first) order; links are stored by depth
    int next = 6;
    for (int d = 0; d < 6; d++) m.user_dof[d] = d;
    for (int b = 1; b < nb; b++)
      if (owner[b] == b && b != base) m.user_dof[5 + link_of[b]] = next++;
    for (int d = 0; d < m.nv; d++) m.dof_of_user[m.user_dof[d]] = d;
  }
  m.nlevels = nlev;
  for (int k = 1; k <= nlev; k++) if (m.level_off[k] < m.level_off[k - 1]) m.level_off[k] = m.level_off[k - 1];
  {
    const Joint3& J = M.bodies[base].joints[0];
    for (int d = 0; d < 6; d++) { m.damping[d] = J.damping; m.armature[d] = J.armature; }
  }
  {  // children lists
    int k = 0;
    for (int l = 0; l < nl; l++) {
      m.child_off[l] = k;
      for (int c = 0; c < nl; c++) if (m.parent[c] == l) m.child[k++] = c;
    }
    m.child_off[nl] = k;
  }
  // ---- welded bodies folded into their links
  for (int l = 0; l < nl; l++) {
    double mass = 0; V3 mc{};
    for (int b = 1; b < nb; b++)
      if (link_of[b] == l) { const V3 c = in_link[b].p + mul(in_link[b].R, M.bodies[b].ipos); mass += M.bodies[b].mass; mc = mc + M.bodies[b].mass * c; }
    if (!(mass > 0)) { *err = "massless link"; return false; }
    const V3 com = (1.0 / mass) * mc;
    double I[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int b = 1; b < nb; b++) {
      if (link_of[b] != l) continue;
      const M3 Ib = mul(mul(in_link[b].R, full_inertia(M.bodies[b].I)), transpose(in_link[b].R));
      const V3 c = in_link[b].p + mul(in_link[b].R, M.bodies[b].ipos);
      const V3 d = c - com;
      const double dv[3] = {d.x, d.y, d.z}, d2 = dot(d, d), mb = M.bodies[b].mass;
      for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) I[3 * i + j] += Ib.m[3 * i + j] + mb * ((i == j ? d2 : 0.0) - dv[i] * dv[j]);
    }
    m.mass[l] = mass;
    m.com[l][0] = com.x; m.com[l][1] = com.y; m.com[l][2] = com.z;
    m.inertia[l][0] = I[0]; m.inertia[l][1] = I[4]; m.inertia[l][2] = I[8];
    m.inertia[l][3] = I[1]; m.inertia[l][4] = I[2]; m.inertia[l][5] = I[5];
  }
  // ---- options
  m.timestep = M.timestep; m.tolerance = M.tolerance; m.impratio = M.impratio; m.iterations = M.iterations;
  for (int i = 0; i < 3; i++) m.gravity[i] = M.gravity[i];
  if (M.solver != "PGS" || M.cone != "elliptic") { *err = "only solver='PGS' with cone='elliptic' is implemented (cassie3d_stiff.xml:5)"; return false; }
  // ---- qpos0 pose of every body (all hinges at ref: static composition), mass matrix, invweight0 (mj_setConst [EXT])
  Pose3 P0;
  fk3(M, std::vector<JointRef>(), std::vector<double>(), &P0);
  const int nv = m.nv;
  struct DofAxis { V3 w, p; bool rot; };
  std::vector<DofAxis> dof(nv);
  for (int k = 0; k < 3; k++) {
    V3 e{k == 0 ? 1.0 : 0.0, k == 1 ? 1.0 : 0.0, k == 2 ? 1.0 : 0.0};
    dof[k] = {e, V3{}, false};
    dof[3 + k] = {mul(P0.xmat[base], e), P0.xpos[base], true};
  }
  for (int l = 1; l < nl; l++) {
    const int b = link_bodies[l];
    const Joint3& J = M.bodies[b].joints[0];
    dof[5 + l] = {mul(P0.xmat[b], J.axis), P0.xpos[b] + mul(P0.xmat[b], J.pos), true};
  }
  auto moves = [&](int d, int b) { return (m.anc[link_of[b]] >> d) & 1u; };
  auto jac = [&](int b, V3 P, std::vector<V3>* jp, std::vector<V3>* jr) {
    jp->assign(nv, V3{}); jr->assign(nv, V3{});
    for (int d = 0; d < nv; d++) {
      if (!moves(d, b)) continue;
      if (dof[d].rot) { (*jr)[d] = dof[d].w; (*jp)[d] = cross(dof[d].w, P - dof[d].p); }
      else (*jp)[d] = dof[d].w;
    }
  };
  std::vector<double> Mq((size_t)nv * nv, 0.0), Minv;
  std::vector<V3> jp, jr;
  for (int b = 1; b < nb; b++) {
    const Body3& B = M.bodies[b];
    if (B.mass <= 0) continue;
    const V3 c = P0.xpos[b] + mul(P0.xmat[b], B.ipos);
    const M3 Iw = mul(mul(P0.xmat[b], full_inertia(B.I)), transpose(P0.xmat[b]));
    jac(b, c, &jp, &jr);
    for (int i = 0; i < nv; i++) {
      if (!moves(i, b)) continue;
      const V3 Ir = mul(Iw, jr[i]);
      for (int j = 0; j < nv; j++)
        if (moves(j, b)) Mq[(size_t)i * nv + j] += B.mass * dot(jp[i], jp[j]) + dot(Ir, jr[j]);
    }
  }
  double tr = 0;
  for (int d = 0; d < nv; d++) { Mq[(size_t)d * nv + d] += m.armature[d]; tr += Mq[(size_t)d * nv + d]; }
  m.meaninertia = tr / nv;
  if (!spd_inverse(nv, Mq, &Minv)) { *err = "mass matrix at qpos0 is not positive definite"; return false; }
  for (int d = 0; d < nv; d++) m.dof_invweight[d] = Minv[(size_t)d * nv + d];
  std::vector<double> biw(nb, 0.0);
  for (int b = 1; b < nb; b++) {
    const V3 c = P0.xpos[b] + mul(P0.xmat[b], M.bodies[b].ipos);
    jac(b, c, &jp, &jr);
    double st = 0;
    for (int r = 0; r < 3; r++)
      for (int i = 0; i < nv; i++)
        for (int j = 0; j < nv; j++) {
          const double a = r == 0 ? jp[i].x : (r == 1 ? jp[i].y : jp[i].z), bb = r == 0 ? jp[j].x : (r == 1 ? jp[j].y : jp[j].z);
          st += a * Minv[(size_t)i * nv + j] * bb;
        }
    biw[b] = std::max(st / 3, 1e-15);
  }
  // ---- geoms and collision pairs (mj_collision order: world geoms first, then bodies in tree order)
  struct GRef { int body; const Geom3* g; int idx; };
  std::vector<GRef> all;
  for (int b = 0; b < nb; b++)
    for (auto& g : M.bodies[b].geoms) all.push_back({b, &g, -1});
  int ng = 0;
  for (auto& r : all) {
    if (r.body == 0) {
      if (r.g->type != kPlane || m.has_plane) { *err = "the world may carry one plane only"; return false; }
      m.has_plane = 1;
      m.plane_pos[0] = r.g->pos.x; m.plane_pos[1] = r.g->pos.y; m.plane_pos[2] = r.g->pos.z;
      m.plane_n[2] = 1.0;
      continue;
    }
    if (ng >= kMaxGeoms) { *err = "too many collision geoms"; return false; }
    const Rigid& X = in_link[r.body];
    auto put = [&](double* d, V3 v) { const V3 w = X.p + mul(X.R, v); d[0] = w.x; d[1] = w.y; d[2] = w.z; };
    m.g_link[ng] = link_of[r.body]; m.g_type[ng] = r.g->type; m.g_radius[ng] = r.g->radius;
    if (r.g->type == kSphere) put(m.g_p0[ng], r.g->pos);
    else if (r.g->type == kCapsule) { put(m.g_p0[ng], r.g->to); put(m.g_p1[ng], r.g->from); }
    else { *err = "unsupported geom on a moving body"; return false; }
    r.idx = ng++;
  }
  m.ng = ng;
  int np = 0;
  for (size_t i = 0; i < all.size(); i++)
    for (size_t j = i + 1; j < all.size(); j++) {
      const Geom3 &a = *all[i].g, &b = *all[j].g;
      if (!((a.contype & b.conaffinity) || (b.contype & a.conaffinity))) continue;
      if (all[i].body == all[j].body) continue;
      const bool plane = all[i].body == 0;
      if (!plane && !(a.type == kCapsule && b.type == kCapsule)) { *err = "only plane-sphere, plane-capsule and capsule-capsule pairs are implemented"; return false; }
      if (!plane && link_of[all[i].body] == link_of[all[j].body]) continue;   // welded into one link: no relative motion
      if (np >= kMaxPairs) { *err = "too many collision pairs"; return false; }
      m.pair_a[np] = plane ? -1 : all[i].idx; m.pair_b[np] = all[j].idx;
      m.pair_condim[np] = std::max(a.condim, b.condim);
      if (m.pair_condim[np] != 3 && m.pair_condim[np] != 1) { *err = "only condim 1 and condim 3 contacts are implemented"; return false; }
      for (int k = 0; k < 3; k++) m.pair_friction[np][k] = std::max(a.friction[k], b.friction[k]);
      for (int k = 0; k < 2; k++) m.pair_solref[np][k] = 0.5 * (a.solref[k] + b.solref[k]);
      for (int k = 0; k < 5; k++) m.pair_solimp[np][k] = 0.5 * (a.solimp[k] + b.solimp[k]);
      m.pair_invweight[np] = biw[all[i].body] + biw[all[j].body];
      np++;
    }
  m.npair = np;
  // ---- connects: anchor2 = anchor1 seen from body2 at qpos0 (mjCModel compile [EXT]); both re-expressed in the link frames
  if ((int)M.connects.size() > kMaxEq) { *err = "too many connects"; return false; }
  m.neq = (int)M.connects.size();
  for (int e = 0; e < m.neq; e++) {
    const Connect3& C = M.connects[e];
    const V3 Pw = P0.xpos[C.b1] + mul(P0.xmat[C.b1], C.anchor);
    const V3 a2 = tmul(P0.xmat[C.b2], Pw - P0.xpos[C.b2]);
    const V3 l1 = in_link[C.b1].p + mul(in_link[C.b1].R, C.anchor), l2 = in_link[C.b2].p + mul(in_link[C.b2].R, a2);
    m.eq_l1[e] = link_of[C.b1]; m.eq_l2[e] = link_of[C.b2];
    m.eq_a1[e][0] = l1.x; m.eq_a1[e][1] = l1.y; m.eq_a1[e][2] = l1.z;
    m.eq_a2[e][0] = l2.x; m.eq_a2[e][1] = l2.y; m.eq_a2[e][2] = l2.z;
    for (int k = 0; k < 2; k++) m.eq_solref[e][k] = C.solref[k];
    for (int k = 0; k < 5; k++) m.eq_solimp[e][k] = C.solimp[k];
    m.eq_invweight[e] = biw[C.b1] + biw[C.b2];
  }
  // ---- motors
  if ((int)M.motors.size() > kMaxAct) { *err = "too many motors"; return false; }
  m.nu = (int)M.motors.size();
  for (int a = 0; a < m.nu; a++) {
    const Motor3& mo = M.motors[a];
    int d = -1;
    for (int l = 1; l < nl; l++) if (M.bodies[link_bodies[l]].joints[0].name == mo.joint) d = 5 + l;
    if (d < 0) { *err = "motor on unknown joint '" + mo.joint + "'"; return false; }
    m.act_dof[a] = d; m.act_gear[a] = mo.gear; m.act_limited[a] = mo.limited ? 1 : 0; m.act_lo[a] = mo.lo; m.act_hi[a] = mo.hi;
  }
  // ---- foot sites of the env observation (a foot = the mean of its front and rear contact site), in the link frame
  static const char* const foot_sites[kNumFootSites] = {"left_contact_front", "left_contact_rear", "right_contact_front", "right_contact_rear"};
  for (int k = 0; k < kNumFootSites; k++) {
    int found = 0;
    for (int b = 1; b < nb; b++)
      for (auto& s : M.bodies[b].sites)
        if (s.name == foot_sites[k]) {
          const V3 p = in_link[b].p + mul(in_link[b].R, s.pos);
          m.site_link[k] = link_of[b];
          m.site_pos[k][0] = p.x; m.site_pos[k][1] = p.y; m.site_pos[k][2] = p.z;
          found++;
        }
    if (found != 1) {
      *err = std::string(found ? "more than one site named '" : "the model has no site named '") + foot_sites[k] +
             "' (the 3-D env observes the feet at the sites left/right_contact_front/rear)";
      return false;
    }
  }
  return true;
}

bool flatten_tree_file(const std::string& path, tree::TreeModel<double>* out, std::string* err) {
  std::ifstream f(path);
  if (!f) { *err = "cannot open model file '" + path + "'"; return false; }
  std::stringstream ss;
  ss << f.rdbuf();
  Model3 M;
  if (!read_model3(ss.str(), &M, err)) return false;
  return flatten_tree(M, out, err);
}

namespace {
template <class A, class B> void cp(A& d, const B& s) { d = (A)s; }
template <class A, class B, size_t N> void cp(A (&d)[N], const B (&s)[N]) { for (size_t i = 0; i < N; i++) cp(d[i], s[i]); }
}  // namespace

template <typename T>
PlanarModel<T> cast_model(const PlanarModel<double>& s) {
  PlanarModel<T> o;
#define CP(f) cp(o.f, s.f)
  CP(pel_org); CP(pel_ref); CP(pel_com); CP(pel_mass); CP(pel_inertia);
  CP(off); CP(sgn); CP(ang0); CP(com); CP(mass); CP(inertia);
  CP(damping); CP(armature); CP(lim_lo); CP(lim_hi); CP(lim_diag); CP(has_limit); CP(lim_solref); CP(lim_solimp);
  CP(act_dof); CP(act_gear); CP(act_lo); CP(act_hi);
  CP(eq_a1); CP(eq_a2); CP(eq_solref); CP(eq_solimp); CP(eq_diag);
  CP(sph_c); CP(sph_r); CP(sph_diag); CP(cap_link); CP(cap_to); CP(cap_from); CP(cap_r); CP(cap_diag);
  CP(con_solref); CP(con_solimp); CP(con_mu);
  CP(site_link); CP(site_off);
  CP(timestep); CP(gravity_z); CP(tolerance); CP(meaninertia); CP(impratio); CP(iterations); CP(total_mass);
#undef CP
  return o;
}
template PlanarModel<float> cast_model<float>(const PlanarModel<double>&);
template PlanarModel<double> cast_model<double>(const PlanarModel<double>&);

}  // namespace cassie
