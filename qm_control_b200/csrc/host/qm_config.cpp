#include "qm_config.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <functional>
#include <sstream>

namespace qmb {

namespace {
std::string slurp(const std::string& path, const char* what) {
  std::ifstream in(path);
  if (!in) throw std::invalid_argument(std::string("[QMInterface] ") + what + " not found: " + path);   // QMInterface.cpp:45,53,61
  std::stringstream ss; ss << in.rdbuf(); return ss.str();
}
}  // namespace

// ------------------------------------------------------------------ INFO
InfoFile::InfoFile(const std::string& path) {
  const std::string txt = slurp(path, "info file");
  std::vector<std::string> scope;           // current path components
  std::string pending_key; bool have_pending = false;
  auto full = [&](const std::string& leaf) { std::string p; for (auto& s : scope) { p += s; p += '.'; } return p + leaf; };
  auto scope_path = [&]() { std::string p; for (size_t i = 0; i < scope.size(); ++i) { if (i) p += '.'; p += scope[i]; } return p; };
  size_t i = 0; const size_t n = txt.size();
  while (i < n) {
    // one logical line
    size_t e = txt.find('\n', i); if (e == std::string::npos) e = n;
    std::string line = txt.substr(i, e - i); i = e + 1;
    size_t cpos = line.find(';'); if (cpos != std::string::npos) line.erase(cpos);
    cpos = line.find("//"); if (cpos != std::string::npos) line.erase(cpos);
    std::vector<std::string> tok; { size_t k = 0; while (k < line.size()) { while (k < line.size() && isspace((unsigned char)line[k])) ++k; if (k >= line.size()) break;
        if (line[k] == '"') { size_t q = line.find('"', k + 1); tok.push_back(line.substr(k + 1, q - k - 1)); k = q + 1; }
        else if (line[k] == '{' || line[k] == '}') { tok.push_back(std::string(1, line[k])); ++k; }
        else { size_t s = k; while (k < line.size() && !isspace((unsigned char)line[k]) && line[k] != '{' && line[k] != '}') ++k; tok.push_back(line.substr(s, k - s)); } } }
    for (size_t t = 0; t < tok.size(); ++t) {
      if (tok[t] == "{") { if (!have_pending) throw std::runtime_error("INFO: unexpected '{' in " + path); scope.push_back(pending_key); have_pending = false; }
      else if (tok[t] == "}") { if (scope.empty()) throw std::runtime_error("INFO: unexpected '}' in " + path); scope.pop_back(); have_pending = false; }
      else {
        const std::string key = tok[t]; nodes_[scope_path()].push_back(key);
        if (t + 1 < tok.size() && tok[t + 1] != "{" && tok[t + 1] != "}") { values_[full(key)] = tok[t + 1]; ++t; have_pending = false; }
        else { pending_key = key; have_pending = true; }
      }
    }
  }
}
double InfoFile::number(const std::string& key) const { auto it = values_.find(key); if (it == values_.end()) throw std::runtime_error("INFO key missing: " + key); return std::stod(it->second); }
std::string InfoFile::text(const std::string& key) const { auto it = values_.find(key); if (it == values_.end()) throw std::runtime_error("INFO key missing: " + key); return it->second; }
bool InfoFile::boolean(const std::string& key, bool fallback) const {
  auto it = values_.find(key); if (it == values_.end()) return fallback;
  if (it->second == "true" || it->second == "1") return true; if (it->second == "false" || it->second == "0") return false;
  throw std::runtime_error("INFO key " + key + ": not a boolean: " + it->second);
}
std::vector<double> InfoFile::matrix(const std::string& key, int rows, int cols) const {
  std::vector<double> m((size_t)rows * cols, 0.0); auto it = nodes_.find(key); if (it == nodes_.end()) throw std::runtime_error("INFO matrix missing: " + key);
  const double scaling = number(key + ".scaling", 1.0);
  for (const std::string& k : it->second) { int r, c; if (sscanf(k.c_str(), "(%d,%d)", &r, &c) == 2 && r < rows && c < cols) m[(size_t)r * cols + c] = scaling * number(key + "." + k); }
  return m;
}
std::vector<std::string> InfoFile::list(const std::string& key) const {
  std::vector<std::string> out; auto it = nodes_.find(key); if (it == nodes_.end()) return out;
  for (const std::string& k : it->second) { int idx; if (sscanf(k.c_str(), "[%d]", &idx) == 1) { if ((int)out.size() <= idx) out.resize(idx + 1); out[idx] = text(key + "." + k); } }
  return out;
}

int mode_from_name(const std::string& name) {   // ocs2_legged_robot string2ModeNumber [upstream]
  if (name == "STANCE") return 15; if (name == "FLY") return 0;
  int m = 0; std::stringstream ss(name); std::string part;
  while (std::getline(ss, part, '_')) { if (part == "LF") m |= 8; else if (part == "RF") m |= 4; else if (part == "LH") m |= 2; else if (part == "RH") m |= 1; else throw std::runtime_error("unknown mode name: " + name); }
  return m;
}
ModeTemplate read_mode_template(const InfoFile& f, const std::string& key) {
  ModeTemplate t; for (auto& s : f.list(key + ".modeSequence")) t.modes.push_back(mode_from_name(s));
  for (auto& s : f.list(key + ".switchingTimes")) t.switching_times.push_back(std::stod(s));
  if (t.modes.empty() || t.switching_times.size() != t.modes.size() + 1) throw std::runtime_error("bad mode sequence template: " + key);
  return t;
}

// ------------------------------------------------------------------ URDF
namespace {
// attribute value of `name="..."` inside the tag text [b, e)
bool attr(const std::string& s, size_t b, size_t e, const char* name, std::string& out) {
  const std::string pat = std::string(name) + "=";
  size_t p = b;
  while ((p = s.find(pat, p)) != std::string::npos && p < e) {
    if (p > b && (isalnum((unsigned char)s[p - 1]) || s[p - 1] == '_')) { p += pat.size(); continue; }
    const char q = s[p + pat.size()]; const size_t vs = p + pat.size() + 1; const size_t ve = s.find(q, vs); out = s.substr(vs, ve - vs); return true;
  }
  return false;
}
void triple(const std::string& v, double* o) { std::istringstream is(v); is >> o[0] >> o[1] >> o[2]; }
// find the first child element <tag ...> within [b, e); returns tag extent
bool child_tag(const std::string& s, size_t b, size_t e, const char* tag, size_t& tb, size_t& te) {
  const std::string pat = std::string("<") + tag; size_t p = b;
  while ((p = s.find(pat, p)) != std::string::npos && p < e) { const char nx = s[p + pat.size()]; if (isspace((unsigned char)nx) || nx == '>' || nx == '/') { tb = p; te = s.find('>', p); return true; } p += pat.size(); }
  return false;
}
}  // namespace

UrdfRobot read_urdf(const std::string& path) {
  std::string s = slurp(path, "URDF file");
  // strip comments
  for (size_t p; (p = s.find("<!--")) != std::string::npos;) { size_t q = s.find("-->", p); s.erase(p, q == std::string::npos ? std::string::npos : q + 3 - p); }
  UrdfRobot robot; size_t pos = s.find("<robot"); if (pos == std::string::npos) throw std::runtime_error("URDF: no <robot> element");
  pos = s.find('>', pos) + 1; int depth = 0;
  while (pos < s.size()) {
    size_t lt = s.find('<', pos); if (lt == std::string::npos) break; size_t gt = s.find('>', lt); if (gt == std::string::npos) break;
    const bool closing = s[lt + 1] == '/'; const bool selfclose = s[gt - 1] == '/';
    if (closing) { --depth; pos = gt + 1; if (depth < 0) break; continue; }
    size_t ne = lt + 1; while (ne < gt && !isspace((unsigned char)s[ne]) && s[ne] != '/' ) ++ne; const std::string tag = s.substr(lt + 1, ne - lt - 1);
    if (depth == 0 && (tag == "link" || tag == "joint")) {
      size_t end = gt + 1; if (!selfclose) { const std::string close = "</" + tag + ">"; end = s.find(close, gt); if (end == std::string::npos) throw std::runtime_error("URDF: unterminated <" + tag + ">"); }
      std::string name; attr(s, lt, gt, "name", name);
      if (tag == "link") {
        UrdfLink l; l.name = name; size_t ib, ie;
        if (!selfclose && child_tag(s, gt, end, "inertial", ib, ie)) {
          const size_t iend = s.find("</inertial>", ie); size_t tb, te; std::string v; l.has_inertial = true;
          if (child_tag(s, ie, iend, "origin", tb, te)) { if (attr(s, tb, te, "xyz", v)) triple(v, l.com); if (attr(s, tb, te, "rpy", v)) triple(v, l.rpy); }
          if (child_tag(s, ie, iend, "mass", tb, te) && attr(s, tb, te, "value", v)) l.mass = std::stod(v);
          if (child_tag(s, ie, iend, "inertia", tb, te)) { const char* k[6] = {"ixx", "ixy", "ixz", "iyy", "iyz", "izz"}; for (int a = 0; a < 6; ++a) if (attr(s, tb, te, k[a], v)) l.inertia[a] = std::stod(v); }
        }
        robot.links[name] = l;
      } else {
        std::string type; if (attr(s, lt, gt, "type", type)) {
          UrdfJoint j; j.name = name; j.type = type; size_t tb, te; std::string v;
          if (child_tag(s, gt, end, "parent", tb, te)) attr(s, tb, te, "link", j.parent);
          if (child_tag(s, gt, end, "child", tb, te)) attr(s, tb, te, "link", j.child);
          if (child_tag(s, gt, end, "origin", tb, te)) { if (attr(s, tb, te, "xyz", v)) triple(v, j.xyz); if (attr(s, tb, te, "rpy", v)) triple(v, j.rpy); }
          if (child_tag(s, gt, end, "axis", tb, te) && attr(s, tb, te, "xyz", v)) triple(v, j.axis);
          if (child_tag(s, gt, end, "limit", tb, te)) { if (attr(s, tb, te, "lower", v)) j.lower = std::stod(v); if (attr(s, tb, te, "upper", v)) j.upper = std::stod(v); if (attr(s, tb, te, "effort", v)) j.effort = std::stod(v); if (attr(s, tb, te, "velocity", v)) j.velocity = std::stod(v); }
          robot.joints[name] = j;
        }
      }
      pos = selfclose ? gt + 1 : end + tag.size() + 3; continue;
    }
    if (!selfclose && tag[0] != '?' && tag[0] != '!') ++depth;
    pos = gt + 1;
  }
  return robot;
}

// ------------------------------------------------------------------ model
namespace {
struct Rot { double m[9]; };
Rot mul(const Rot& a, const Rot& b) { Rot c; for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) c.m[3 * i + j] = a.m[3 * i] * b.m[j] + a.m[3 * i + 1] * b.m[3 + j] + a.m[3 * i + 2] * b.m[6 + j]; return c; }
Rot transpose(const Rot& a) { Rot c; for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) c.m[3 * i + j] = a.m[3 * j + i]; return c; }
void apply(const Rot& a, const double* v, double* o) { for (int i = 0; i < 3; ++i) o[i] = a.m[3 * i] * v[0] + a.m[3 * i + 1] * v[1] + a.m[3 * i + 2] * v[2]; }
Rot from_rpy(const double* rpy) {   // URDF fixed-axis roll-pitch-yaw = Rz(y) Ry(p) Rx(r)
  const double sr = sin(rpy[0]), cr = cos(rpy[0]), sp = sin(rpy[1]), cp = cos(rpy[1]), sy = sin(rpy[2]), cy = cos(rpy[2]);
  return Rot{{cy * cp, cy * sp * sr - sy * cr, cy * sp * cr + sy * sr, sy * cp, sy * sp * sr + cy * cr, sy * sp * cr - cy * sr, -sp, cp * sr, cp * cr}};
}
Rot identity() { return Rot{{1, 0, 0, 0, 1, 0, 0, 0, 1}}; }
Rot about_axis(int ax, double q) { const double s = sin(q), c = cos(q); if (ax == 0) return Rot{{1, 0, 0, 0, c, -s, 0, s, c}}; if (ax == 1) return Rot{{c, 0, s, 0, 1, 0, -s, 0, c}}; return Rot{{c, -s, 0, s, c, 0, 0, 0, 1}}; }

struct Lump { double m = 0, c[3] = {0, 0, 0}, I[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}; };
// add rigid body (mass, com, inertia about com) expressed in the same frame
void lump_add(Lump& a, double m, const double* c, const double* I) {
  if (m == 0.0) { for (int i = 0; i < 9; ++i) a.I[i] += I[i]; return; }
  const double mt = a.m + m; double cn[3]; for (int i = 0; i < 3; ++i) cn[i] = (a.m * a.c[i] + m * c[i]) / mt;
  auto shifted = [&](double mm, const double* cc, const double* II, double* out) { double d[3] = {cc[0] - cn[0], cc[1] - cn[1], cc[2] - cn[2]}; const double dd = d[0] * d[0] + d[1] * d[1] + d[2] * d[2];
    for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) out[3 * i + j] = II[3 * i + j] + mm * ((i == j ? dd : 0.0) - d[i] * d[j]); };
  double I1[9], I2[9]; shifted(a.m, a.c, a.I, I1); shifted(m, c, I, I2);
  for (int i = 0; i < 9; ++i) a.I[i] = I1[i] + I2[i]; a.m = mt; for (int i = 0; i < 3; ++i) a.c[i] = cn[i];
}
int axis_index(const double* a, const std::string& name) {
  if (a[0] == 1 && a[1] == 0 && a[2] == 0) return 0; if (a[0] == 0 && a[1] == 1 && a[2] == 0) return 1; if (a[0] == 0 && a[1] == 0 && a[2] == 1) return 2;
  throw std::runtime_error("URDF: joint " + name + " has an axis other than +x/+y/+z (unsupported)");
}
}  // namespace

HostModel build_host_model(const std::string& task_file, const std::string& urdf_file, const std::string& reference_file, const std::string& gains_file) {
  InfoFile task(task_file); UrdfRobot urdf = read_urdf(urdf_file); InfoFile reference(reference_file);
  HostModel hm; DevModel& d = hm.dev; std::memset(&d, 0, sizeof(d));
  // --- kinematic tree (setupModel, QMInterface.cpp:408-439) ---
  std::map<std::string, bool> is_child; for (auto& kv : urdf.joints) is_child[kv.second.child] = true;
  std::string root; for (auto& kv : urdf.links) if (!is_child.count(kv.first)) root = kv.first;
  if (root.empty()) throw std::runtime_error("URDF: no root link");
  Lump lumps[NB]; int nj = 0;
  auto add_link_inertia = [&](int body, const UrdfLink& l, const Rot& R, const double* p) {
    if (!l.has_inertial) return; Rot Rin = from_rpy(l.rpy); Rot Rt = mul(R, Rin);
    const double Il[9] = {l.inertia[0], l.inertia[1], l.inertia[2], l.inertia[1], l.inertia[3], l.inertia[4], l.inertia[2], l.inertia[4], l.inertia[5]};
    Rot I0; std::memcpy(I0.m, Il, sizeof(Il)); Rot Iw = mul(mul(Rt, I0), transpose(Rt));
    double c[3]; apply(R, l.com, c); for (int i = 0; i < 3; ++i) c[i] += p[i];
    lump_add(lumps[body], l.mass, c, Iw.m);
  };
  const double zero3[3] = {0, 0, 0};
  add_link_inertia(0, urdf.links[root], identity(), zero3);
  { HostFrame f; f.name = root; f.body = 0; std::memcpy(f.R, identity().m, sizeof(f.R)); std::memcpy(f.p, zero3, sizeof(f.p)); hm.frames.push_back(f); }
  d.depth[0] = 0;
  std::function<void(const std::string&, int, const Rot&, const double*, int)> visit = [&](const std::string& link, int body, const Rot& R, const double* p, int chain_first) {
    for (auto& kv : urdf.joints) {   // std::map → children in joint-name order (urdfdom)
      const UrdfJoint& j = kv.second; if (j.parent != link) continue;
      Rot Rj = mul(R, from_rpy(j.rpy)); double pj[3]; apply(R, j.xyz, pj); for (int i = 0; i < 3; ++i) pj[i] += p[i];
      if (j.type == "fixed") {
        add_link_inertia(body, urdf.links[j.child], Rj, pj);
        HostFrame f; f.name = j.child; f.body = body; std::memcpy(f.R, Rj.m, sizeof(f.R)); std::memcpy(f.p, pj, sizeof(f.p)); hm.frames.push_back(f);
        visit(j.child, body, Rj, pj, chain_first);
      } else if (j.type == "revolute" || j.type == "continuous") {
        if (nj >= NJ) throw std::runtime_error("URDF: more than 18 actuated joints");
        const int id = nj++; d.parent[id] = body; d.axis[id] = axis_index(j.axis, j.name); std::memcpy(d.Rj[id], Rj.m, sizeof(Rj.m)); std::memcpy(d.pj[id], pj, sizeof(pj));
        d.effort[id] = j.effort; d.depth[id + 1] = d.depth[body] + 1; d.chain_start[id] = (body == 0) ? id : chain_first;
        hm.joint_names.push_back(j.name);
        if (id >= 12) { d.arm_pos_lower[id - 12] = j.lower; d.arm_pos_upper[id - 12] = j.upper; }
        add_link_inertia(id + 1, urdf.links[j.child], identity(), zero3);
        HostFrame f; f.name = j.child; f.body = id + 1; std::memcpy(f.R, identity().m, sizeof(f.R)); std::memcpy(f.p, zero3, sizeof(f.p)); hm.frames.push_back(f);
        visit(j.child, id + 1, identity(), zero3, (body == 0) ? id : chain_first);
      } else throw std::runtime_error("URDF: unsupported joint type " + j.type);
    }
  };
  visit(root, 0, identity(), zero3, 0);
  if (nj != NJ) throw std::runtime_error("URDF: expected 18 actuated joints, found " + std::to_string(nj));
  // the kernels assume 4 three-joint legs followed by one six-joint arm, joints contiguous per chain
  for (int l = 0; l < 4; ++l) for (int k = 0; k < 3; ++k) if (d.chain_start[3 * l + k] != 3 * l || d.depth[3 * l + k + 1] != k + 1) throw std::runtime_error("URDF: unexpected leg topology");
  for (int k = 0; k < 6; ++k) if (d.chain_start[12 + k] != 12 || d.depth[13 + k] != k + 1) throw std::runtime_error("URDF: unexpected arm topology");
  d.total_mass = 0;
  for (int b = 0; b < NB; ++b) { d.mass[b] = lumps[b].m; std::memcpy(d.com[b], lumps[b].c, sizeof(lumps[b].c)); std::memcpy(d.Ib[b], lumps[b].I, sizeof(lumps[b].I)); d.total_mass += lumps[b].m; }
  auto frame = [&](const std::string& n) -> const HostFrame& { for (auto& f : hm.frames) if (f.name == n) return f; throw std::runtime_error("URDF: frame not found: " + n); };
  const char* feet[4] = {"LF_FOOT", "RF_FOOT", "LH_FOOT", "RH_FOOT"};   // ModelSettings.h:38
  for (int i = 0; i < 4; ++i) { const HostFrame& f = frame(feet[i]); d.foot_body[i] = f.body; std::memcpy(d.foot_p[i], f.p, sizeof(f.p)); d.foot_leg[i] = d.chain_start[f.body - 1]; d.leg_foot[d.foot_leg[i] / 3] = i; }
  { const HostFrame& f = frame(task.text("model_settings.eeFrame")); d.ee_body = f.body; std::memcpy(d.ee_R, f.R, sizeof(f.R)); std::memcpy(d.ee_p, f.p, sizeof(f.p)); }

  // --- CentroidalModelInfo, SRBD (createCentroidalModelInfo [upstream]) ---
  { auto djs = reference.matrix("defaultJointState", NJ, 1); for (int i = 0; i < NJ; ++i) hm.default_joint_state[i] = djs[i]; }
  Rot Rw[NB]; double pw[NB][3];
  auto host_fk = [&](const double* q /*24*/) {
    const double rz[3] = {q[5], q[4], q[3]}; Rw[0] = from_rpy(rz); for (int i = 0; i < 3; ++i) pw[0][i] = q[i];   // Rz(q3) Ry(q4) Rx(q5)
    for (int j = 0; j < NJ; ++j) { const int pb = d.parent[j]; Rot Rl; std::memcpy(Rl.m, d.Rj[j], sizeof(Rl.m)); Rw[j + 1] = mul(mul(Rw[pb], Rl), about_axis(d.axis[j], q[6 + j])); apply(Rw[pb], d.pj[j], pw[j + 1]); for (int i = 0; i < 3; ++i) pw[j + 1][i] += pw[pb][i]; }
  };
  { double qn[NQ] = {0}; for (int j = 0; j < NJ; ++j) qn[6 + j] = hm.default_joint_state[j]; host_fk(qn);
    Lump whole; for (int b = 0; b < NB; ++b) { double c[3]; apply(Rw[b], d.com[b], c); for (int i = 0; i < 3; ++i) c[i] += pw[b][i]; Rot I0; std::memcpy(I0.m, d.Ib[b], sizeof(I0.m)); Rot Iw = mul(mul(Rw[b], I0), transpose(Rw[b])); lump_add(whole, d.mass[b], c, Iw.m); }
    std::memcpy(d.I_nom, whole.I, sizeof(whole.I)); for (int i = 0; i < 3; ++i) d.c_nom[i] = -whole.c[i];
    const double* m = d.I_nom; const double c00 = m[4] * m[8] - m[5] * m[7], c01 = m[5] * m[6] - m[3] * m[8], c02 = m[3] * m[7] - m[4] * m[6]; const double id = 1.0 / (m[0] * c00 + m[1] * c01 + m[2] * c02);
    double* o = d.I_nom_inv; o[0] = c00 * id; o[1] = (m[2] * m[7] - m[1] * m[8]) * id; o[2] = (m[1] * m[5] - m[2] * m[4]) * id; o[3] = c01 * id; o[4] = (m[0] * m[8] - m[2] * m[6]) * id; o[5] = (m[2] * m[3] - m[0] * m[5]) * id;
    o[6] = c02 * id; o[7] = (m[1] * m[6] - m[0] * m[7]) * id; o[8] = (m[0] * m[4] - m[1] * m[3]) * id; }

  // --- WBC gains (wbcWigeht.cfg defaults; optional override file) and friction (WbcBase.cpp:584-594) ---
  d.kp_swing = 350; d.kd_swing = 37; d.base_height_kp = 400; d.base_height_kd = 140; d.base_linear_kp = 400; d.base_linear_kd = 100; d.base_angular_kp = 400; d.base_angular_kd = 140;
  { const double kp[6] = {4000, 4200, 4000, 4000, 4200, 6000}; for (int i = 0; i < 6; ++i) { d.arm_joint_kp[i] = kp[i]; d.arm_joint_kd[i] = 75; } }
  for (int i = 0; i < 3; ++i) { d.ee_linear_kp[i] = 3000; d.ee_linear_kd[i] = 75; d.ee_angular_kp[i] = 2000; d.ee_angular_kd[i] = 75; }
  if (!gains_file.empty()) {
    InfoFile g(gains_file); auto get = [&](const std::string& k, double& v) { v = g.number("wbcGains." + k, v); };
    get("kp_swing", d.kp_swing); get("kd_swing", d.kd_swing); get("baseHeightKp", d.base_height_kp); get("baseHeightKd", d.base_height_kd); get("kp_base_linear", d.base_linear_kp); get("kd_base_linear", d.base_linear_kd);
    get("kp_base_angular", d.base_angular_kp); get("kd_base_angular", d.base_angular_kd);
    for (int i = 0; i < 6; ++i) { get("kp_arm_joint_" + std::to_string(i + 1), d.arm_joint_kp[i]); get("kd_arm_joint_" + std::to_string(i + 1), d.arm_joint_kd[i]); }
    const char* ax[3] = {"x", "y", "z"}; for (int i = 0; i < 3; ++i) { get(std::string("kp_ee_linear_") + ax[i], d.ee_linear_kp[i]); get(std::string("kd_ee_linear_") + ax[i], d.ee_linear_kd[i]); get(std::string("kp_ee_angular_") + ax[i], d.ee_angular_kp[i]); get(std::string("kd_ee_angular_") + ax[i], d.ee_angular_kd[i]); }
  }
  d.wbc_friction = task.number("frictionConeTask.frictionCoefficient", 0.3);

  // --- MPC settings and weights ---
  { auto init = task.matrix("initialState", NX, 1); for (int i = 0; i < NX; ++i) hm.initial_state[i] = init[i]; }
  { auto Q = task.matrix("Q", NX, NX); std::memcpy(d.Q, Q.data(), sizeof(d.Q)); auto Rt = task.matrix("R", NU, NU); std::memcpy(d.R, Rt.data(), sizeof(d.R));
    // initializeInputCostWeight (QMInterface.cpp:274-299): R[12:24,12:24] = J^T Rtask[12:24,12:24] J, J = d(foot pos)/d(leg joints) at initialState
    host_fk(hm.initial_state + 6); double J[12][12] = {{0}};
    for (int f = 0; f < 4; ++f) { const int body = d.foot_body[f]; double pf[3]; apply(Rw[body], d.foot_p[f], pf); for (int i = 0; i < 3; ++i) pf[i] += pw[body][i];
      for (int k = 0; k < 3; ++k) { const int j = d.foot_leg[f] + k; const int ax = d.axis[j]; const double a[3] = {Rw[j + 1].m[ax], Rw[j + 1].m[3 + ax], Rw[j + 1].m[6 + ax]}; const double r[3] = {pf[0] - pw[j + 1][0], pf[1] - pw[j + 1][1], pf[2] - pw[j + 1][2]};
        J[3 * f + 0][j] = a[1] * r[2] - a[2] * r[1]; J[3 * f + 1][j] = a[2] * r[0] - a[0] * r[2]; J[3 * f + 2][j] = a[0] * r[1] - a[1] * r[0]; } }
    for (int a = 0; a < 12; ++a) for (int b = 0; b < 12; ++b) { double s = 0; for (int i = 0; i < 12; ++i) for (int k = 0; k < 12; ++k) s += J[i][a] * Rt[(size_t)(12 + i) * NU + 12 + k] * J[k][b]; d.R[(12 + a) * NU + 12 + b] = s; }
    // compact block form used by the kernels; anything outside the blocks is refused (the structured projection relies on it)
    double rmax = 0.0; for (int i = 0; i < NU * NU; ++i) rmax = std::max(rmax, std::fabs(d.R[i]));
    for (int i = 0; i < NU; ++i) for (int j = 0; j < NU; ++j) { const bool in_block = (i < 24 && j < 24) ? (i / 3 == j / 3) : (i == j);
      if (!in_block && std::fabs(d.R[i * NU + j]) > 1e-12 * rmax) throw std::runtime_error("task.info R: entry (" + std::to_string(i) + "," + std::to_string(j) + ") couples different feet/legs; only the block structure of QMInterface::initializeInputCostWeight is supported"); }
    for (int bq = 0; bq < 8; ++bq) for (int a = 0; a < 3; ++a) for (int b = 0; b < 3; ++b) d.Rblk[bq][3 * a + b] = d.R[(3 * bq + a) * NU + 3 * bq + b];
    for (int i = 0; i < 6; ++i) d.Rarm[i] = d.R[(24 + i) * NU + 24 + i];
    d.q_is_diag = 1; for (int i = 0; i < NX; ++i) { d.Qdiag[i] = d.Q[i * NX + i]; for (int j = 0; j < NX; ++j) if (i != j && d.Q[i * NX + j] != 0.0) d.q_is_diag = 0; } }
  d.mu_ee_pos = task.number("endEffector.muPosition", 1.0); d.mu_ee_ori = task.number("endEffector.muOrientation", 1.0);
  d.mu_final_ee_pos = task.number("finalEndEffector.muPosition", 1.0); d.mu_final_ee_ori = task.number("finalEndEffector.muOrientation", 1.0);
  d.friction_mu = task.number("frictionConeSoftConstraint.frictionCoefficient", 1.0); d.friction_barrier_mu = task.number("frictionConeSoftConstraint.mu", 0.1); d.friction_barrier_delta = task.number("frictionConeSoftConstraint.delta", 5.0);
  d.friction_reg = 25.0; d.friction_hess_shift = 1e-6;   // FrictionConeConstraint::Config defaults [upstream]
  d.pos_limit_mu = task.number("jointPositionLimits.mu", 1e-2); d.pos_limit_delta = task.number("jointPositionLimits.delta", 1e-3);
  d.vel_limit_mu = task.number("jointVelocityLimits.mu", 1e-2); d.vel_limit_delta = task.number("jointVelocityLimits.delta", 1e-3);
  { auto lo = task.matrix("jointVelocityLimits.lowerBound.arm", 6, 1), hi = task.matrix("jointVelocityLimits.upperBound.arm", 6, 1); for (int i = 0; i < 6; ++i) { d.arm_vel_lower[i] = lo[i]; d.arm_vel_upper[i] = hi[i]; } }
  d.lift_off_velocity = task.number("swing_trajectory_config.liftOffVelocity", 0.05); d.touch_down_velocity = task.number("swing_trajectory_config.touchDownVelocity", -0.1);
  d.swing_height = task.number("swing_trajectory_config.swingHeight", 0.15); d.swing_time_scale = task.number("swing_trajectory_config.swingTimeScale", 0.15);
  d.position_error_gain = task.number("model_settings.positionErrorGain", 0.0);
  d.sqp_iterations = (int)task.number("sqp.sqpIteration", 1.0); if (d.sqp_iterations < 1) d.sqp_iterations = 1; d.cost_tol = task.number("sqp.costTol", 1e-4);
  d.dt = task.number("sqp.dt", 0.015); d.time_horizon = task.number("mpc.timeHorizon", 1.0); d.delta_tol = task.number("sqp.deltaTol", 1e-4); d.g_max = task.number("sqp.g_max", 1e-2); d.g_min = task.number("sqp.g_min", 1e-6);
  d.alpha_decay = 0.5; d.alpha_min = 1e-4; d.gamma_c = 1e-6; d.armijo_factor = 1e-4;   // ocs2 sqp::Settings defaults [upstream]
  d.wbc_iter_cap0 = 30; d.wbc_iter_cap = 80;
  d.rk_c = 1.0; d.rk_w1 = 0.5; d.rk_w2 = 0.5;                                          // Heun (ocs2 SensitivityIntegrator rk2 [upstream])
  return hm;
}

}  // namespace qmb
