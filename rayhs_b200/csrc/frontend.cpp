// frontend.cpp — host-side front end above the C ABI, in C++ because GHC is not in
// this image.  It stands in for the Haskell layers that stay on the host:
//   JSON.hs:22-141 (scene schema), Descriptors.hs:39-55 (buildScene),
//   MaterialDescriptors.hs:27-45, Mesh.hs:118-221 (OBJ), Bitmap.hs:20-37 (P3 texture),
//   Transform.hs:16-24 + Mat.hs:55-81 (mesh transforms), Mesh.hs:89-101,
//   Image.hs:60-75 (P3 writer), RandomSamples.hs (sample-offset stream shape).
// Output is an rh_raw_scene (include/rayhs_b200.h): the scene before any tree build.
// Nothing here touches the GPU.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <memory>
#include <sstream>
#include <string>
#include <tuple>
#include <unordered_map>
#include <thread>
#include <vector>

#include "common.h"

namespace {

// ------------------------------------------------------------------ JSON (RFC 8259 subset)
struct JValue {
  enum Kind { Null, Bool, Num, Str, Arr, Obj } kind = Null;
  double num = 0;
  bool b = false;
  std::string str;
  std::vector<JValue> arr;
  std::vector<std::pair<std::string, JValue>> obj;
  const JValue* get(const char* key) const {
    if (kind != Obj) return nullptr;
    for (auto& kv : obj)
      if (kv.first == key) return &kv.second;
    return nullptr;
  }
};

struct JParser {
  const char* p;
  const char* end;
  std::string err;
  void ws() { while (p < end && (*p == ' ' || *p == '\t' || *p == '\n' || *p == '\r')) p++; }
  bool fail(const std::string& m) { if (err.empty()) err = m; return false; }
  bool value(JValue& v) {
    ws();
    if (p >= end) return fail("unexpected end of JSON");
    char c = *p;
    if (c == '{') return object(v);
    if (c == '[') return array(v);
    if (c == '"') { v.kind = JValue::Str; return string(v.str); }
    if (!strncmp(p, "true", 4)) { v.kind = JValue::Bool; v.b = true; p += 4; return true; }
    if (!strncmp(p, "false", 5)) { v.kind = JValue::Bool; v.b = false; p += 5; return true; }
    if (!strncmp(p, "null", 4)) { v.kind = JValue::Null; p += 4; return true; }
    char* e = nullptr;
    double d = strtod(p, &e);
    if (e == p) return fail("bad JSON token");
    v.kind = JValue::Num;
    v.num = d;
    p = e;
    return true;
  }
  bool string(std::string& s) {
    p++;  // opening quote
    while (p < end && *p != '"') {
      if (*p == '\\' && p + 1 < end) {
        p++;
        switch (*p) {
          case 'n': s += '\n'; break;
          case 't': s += '\t'; break;
          case 'r': s += '\r'; break;
          case 'b': s += '\b'; break;
          case 'f': s += '\f'; break;
          case 'u': s += '?'; p += 4; break;  // not needed for scene files
          default: s += *p;
        }
        p++;
      } else s += *p++;
    }
    if (p >= end) return fail("unterminated string");
    p++;
    return true;
  }
  bool array(JValue& v) {
    v.kind = JValue::Arr;
    p++;
    ws();
    if (p < end && *p == ']') { p++; return true; }
    for (;;) {
      v.arr.emplace_back();
      if (!value(v.arr.back())) return false;
      ws();
      if (p < end && *p == ',') { p++; continue; }
      if (p < end && *p == ']') { p++; return true; }
      return fail("expected , or ] in array");
    }
  }
  bool object(JValue& v) {
    v.kind = JValue::Obj;
    p++;
    ws();
    if (p < end && *p == '}') { p++; return true; }
    for (;;) {
      ws();
      if (p >= end || *p != '"') return fail("expected key string");
      std::string key;
      if (!string(key)) return false;
      ws();
      if (p >= end || *p != ':') return fail("expected :");
      p++;
      v.obj.emplace_back(key, JValue());
      if (!value(v.obj.back().second)) return false;
      ws();
      if (p < end && *p == ',') { p++; continue; }
      if (p < end && *p == '}') { p++; return true; }
      return fail("expected , or } in object");
    }
  }
};

struct ParseError { std::string msg; };
[[noreturn]] void bad(const std::string& m) { throw ParseError{m}; }

const JValue& field(const JValue& o, const char* key) {  // aeson `.:` — missing key fails the parse
  const JValue* v = o.get(key);
  if (!v) bad(std::string("missing key \"") + key + "\"");
  return *v;
}
double num(const JValue& o, const char* key) {
  const JValue& v = field(o, key);
  if (v.kind != JValue::Num) bad(std::string("key \"") + key + "\" is not a number");
  return v.num;
}
std::string str(const JValue& o, const char* key) {
  const JValue& v = field(o, key);
  if (v.kind != JValue::Str) bad(std::string("key \"") + key + "\" is not a string");
  return v.str;
}
void vec3(const JValue& o, const char* key, double* out) {  // JSON.hs:22-27
  const JValue& v = field(o, key);
  out[0] = num(v, "x"); out[1] = num(v, "y"); out[2] = num(v, "z");
}
void color3(const JValue& o, const char* key, double* out) {  // JSON.hs:29-34
  const JValue& v = field(o, key);
  out[0] = num(v, "r"); out[1] = num(v, "g"); out[2] = num(v, "b");
}

// ------------------------------------------------------------------ Mat.hs / Transform.hs
struct V3 { double x, y, z; };
struct M3 { double a, b, c, d, e, f, g, h, i; };
inline V3 apply(const M3& m, V3 v) {  // Mat.hs:40-44
  return {m.a * v.x + m.b * v.y + m.c * v.z, m.d * v.x + m.e * v.y + m.f * v.z, m.g * v.x + m.h * v.y + m.i * v.z};
}
inline M3 mmul(const M3& p, const M3& q) {  // Mat.hs:24-30
  return {p.a * q.a + p.b * q.d + p.c * q.g, p.a * q.b + p.b * q.e + p.c * q.h, p.a * q.c + p.b * q.f + p.c * q.i,
          p.d * q.a + p.e * q.d + p.f * q.g, p.d * q.b + p.e * q.e + p.f * q.h, p.d * q.c + p.e * q.f + p.f * q.i,
          p.g * q.a + p.h * q.d + p.i * q.g, p.g * q.b + p.h * q.e + p.i * q.h, p.g * q.c + p.h * q.f + p.i * q.i};
}
inline M3 transpose(const M3& m) { return {m.a, m.d, m.g, m.b, m.e, m.h, m.c, m.f, m.i}; }  // Mat.hs:47-49
inline M3 rotateX(double t) { return {1, 0, 0, 0, cos(t), -(sin(t)), 0, sin(t), cos(t)}; }    // Mat.hs:70-74
inline M3 rotateY(double t) { return {cos(t), 0, sin(t), 0, 1, 0, -(sin(t)), 0, cos(t)}; }    // Mat.hs:64-68
inline M3 rotateZ(double t) { return {cos(t), -(sin(t)), 0, sin(t), cos(t), 0, 0, 0, 1}; }    // Mat.hs:58-62
inline V3 vnormalize(V3 v) { double s = 1 / sqrt(v.x * v.x + v.y * v.y + v.z * v.z); return {s * v.x, s * v.y, s * v.z}; }
inline V3 vcross(V3 a, V3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
inline M3 rotateAxis(V3 r, double angle) {  // Mat.hs:76-81 with Vec.hs:151-158 orthonormal
  V3 s;
  if (fabs(r.x) < fabs(r.y) && fabs(r.x) < fabs(r.z)) s = vnormalize({0, -(r.z), r.y});
  else if (fabs(r.y) < fabs(r.x) && fabs(r.y) < fabs(r.z)) s = vnormalize({-(r.z), 0, r.x});
  else s = vnormalize({-(r.y), r.x, 0});
  V3 t = vcross(r, s);
  M3 m{r.x, s.x, t.x, r.y, s.y, t.y, r.z, s.z, t.z};  // fromColumns r s t
  return mmul(mmul(transpose(m), rotateX(angle)), m);
}

struct Transform {  // Transform.hs:7-13
  enum Kind { Translate, Scale, Rotate, RotX, RotY, RotZ, Sequence } kind;
  V3 v{0, 0, 0};
  double angle = 0;
  std::vector<Transform> seq;
};
V3 xform(const Transform& t, V3 p) {  // Transform.hs:16-24
  switch (t.kind) {
    case Transform::Translate: return {p.x + t.v.x, p.y + t.v.y, p.z + t.v.z};
    case Transform::Scale: return {t.v.x * p.x, t.v.y * p.y, t.v.z * p.z};
    case Transform::Rotate: return apply(rotateAxis(t.v, t.angle), p);
    case Transform::RotX: return apply(rotateX(t.angle), p);
    case Transform::RotY: return apply(rotateY(t.angle), p);
    case Transform::RotZ: return apply(rotateZ(t.angle), p);
    case Transform::Sequence: for (auto& s : t.seq) p = xform(s, p); return p;  // foldl (flip transform)
  }
  return p;
}
Transform parseTransform(const JValue& o) {  // JSON.hs:86-97
  Transform t;
  std::string kind = str(o, "type");
  if (kind == "scale") { t.kind = Transform::Scale; vec3(o, "vector", &t.v.x); }
  else if (kind == "translate") { t.kind = Transform::Translate; vec3(o, "vector", &t.v.x); }
  else if (kind == "rotateX") { t.kind = Transform::RotX; t.angle = num(o, "angle"); }
  else if (kind == "rotateY") { t.kind = Transform::RotY; t.angle = num(o, "angle"); }
  else if (kind == "rotateZ") { t.kind = Transform::RotZ; t.angle = num(o, "angle"); }
  else if (kind == "rotate") { t.kind = Transform::Rotate; vec3(o, "axis", &t.v.x); t.angle = num(o, "angle"); }
  else if (kind == "sequence") {
    t.kind = Transform::Sequence;
    const JValue& a = field(o, "transforms");
    if (a.kind != JValue::Arr) bad("transforms is not an array");
    for (auto& e : a.arr) t.seq.push_back(parseTransform(e));
  } else bad("Unknown type for transform " + kind);
  return t;
}

// ------------------------------------------------------------------ file helpers
bool read_file(const std::string& path, std::string& out) {
  std::ifstream f(path, std::ios::binary);
  if (!f) return false;
  std::ostringstream ss;
  ss << f.rdbuf();
  out = ss.str();
  return true;
}
std::vector<std::string> split_lines(const std::string& s) {  // Prelude.lines
  std::vector<std::string> out;
  size_t i = 0;
  while (i < s.size()) {
    size_t j = s.find('\n', i);
    if (j == std::string::npos) { out.push_back(s.substr(i)); break; }
    out.push_back(s.substr(i, j - i));
    i = j + 1;
  }
  return out;
}
std::vector<std::string> words(const std::string& s) {  // Prelude.words
  std::vector<std::string> out;
  size_t i = 0;
  while (i < s.size()) {
    while (i < s.size() && isspace((unsigned char)s[i])) i++;
    size_t j = i;
    while (j < s.size() && !isspace((unsigned char)s[j])) j++;
    if (j > i) out.push_back(s.substr(i, j - i));
    i = j;
  }
  return out;
}
double read_double(const std::string& w) {
  char* e = nullptr;
  double d = strtod(w.c_str(), &e);
  if (e == w.c_str() || *e) bad("cannot read number \"" + w + "\"");
  return d;
}
bool read_maybe_int(const std::string& w, long* out) {  // Text.Read.readMaybe :: Maybe Int
  if (w.empty()) return false;
  char* e = nullptr;
  long v = strtol(w.c_str(), &e, 10);
  if (e == w.c_str() || *e) return false;
  *out = v;
  return true;
}

}  // namespace

// ==================================================================== rh_loaded
struct rh_loaded {
  struct Mesh { std::vector<double> pos, nrm, uv; std::vector<uint32_t> idx; };
  std::vector<rh_raw_object> objects;
  std::vector<std::unique_ptr<Mesh>> meshes;  // index-aligned with objects (null for shapes)
  std::vector<rh_material> materials;
  std::vector<rh_light> lights;
  std::vector<rh_texture> textures;
  std::vector<double> texels;
  rh_camera camera{};
  int32_t width = 0, height = 0, max_depth = 0;
  rh_raw_scene raw{};
  void finalize() {
    for (size_t i = 0; i < objects.size(); i++) {
      Mesh* m = meshes[i].get();
      if (m) {
        objects[i].n_verts = (uint32_t)(m->pos.size() / 3);
        objects[i].n_indices = (uint32_t)m->idx.size();
        objects[i].positions = m->pos.data();
        objects[i].normals = m->nrm.data();
        objects[i].uvs = m->uv.data();
        objects[i].indices = m->idx.data();
      }
    }
    raw.n_objects = (uint32_t)objects.size();
    raw.n_materials = (uint32_t)materials.size();
    raw.n_lights = (uint32_t)lights.size();
    raw.n_textures = (uint32_t)textures.size();
    raw.objects = objects.data();
    raw.materials = materials.data();
    raw.lights = lights.data();
    raw.textures = textures.data();
    raw.texels = texels.data();
    raw.n_texels = texels.size() / 3;
  }
};

namespace {

// Mesh.hs:118-221: readOBJ = buildMesh . catMaybes . map readLine . lines
void load_obj(const std::string& path, rh_loaded::Mesh& out) {
  std::string content;
  if (!read_file(path, content)) bad("cannot open mesh " + path);
  std::vector<V3> pos, norms;
  std::vector<std::pair<double, double>> uvs;
  typedef std::tuple<long, long, long> OBJIndex;  // 0 = Nothing (OBJ indices are 1-based)
  std::vector<OBJIndex> inds;
  for (const std::string& line : split_lines(content)) {
    if (line.size() >= 2 && line[0] == 'v' && line[1] == ' ') {  // Mesh.hs:171, 132-136
      auto w = words(line.substr(2));
      if (w.size() == 3) pos.push_back({read_double(w[0]), read_double(w[1]), read_double(w[2])});
    } else if (line.size() >= 3 && line[0] == 'v' && line[1] == 'n' && line[2] == ' ') {  // Mesh.hs:172, 138-142
      auto w = words(line.substr(3));
      if (w.size() == 3) norms.push_back({read_double(w[0]), read_double(w[1]), read_double(w[2])});
    } else if (line.size() >= 3 && line[0] == 'v' && line[1] == 't' && line[2] == ' ') {  // Mesh.hs:173, 144-148
      auto w = words(line.substr(3));
      if (w.size() == 2) uvs.push_back({read_double(w[0]), read_double(w[1])});
    } else if (line.size() >= 2 && line[0] == 'f' && line[1] == ' ') {  // Mesh.hs:174, 150-169
      std::vector<OBJIndex> face;
      for (const std::string& tok : words(line.substr(2))) {
        std::vector<std::string> parts;  // splitOn "/"
        size_t i = 0;
        for (;;) {
          size_t j = tok.find('/', i);
          if (j == std::string::npos) { parts.push_back(tok.substr(i)); break; }
          parts.push_back(tok.substr(i, j - i));
          i = j + 1;
        }
        long pi = 0, ti = 0, ni = 0;
        if (!read_maybe_int(parts[0], &pi)) continue;  // parseIndex _ = Nothing
        if (parts.size() >= 2 && !read_maybe_int(parts[1], &ti)) ti = 0;
        if (parts.size() >= 3 && !read_maybe_int(parts[2], &ni)) ni = 0;
        if (parts.size() < 3) ni = 0;
        face.emplace_back(pi, ti, ni);
      }
      if (face.size() > 2) inds.insert(inds.end(), face.begin(), face.end());
    }
  }
  // flattenVertices, Mesh.hs:195-212: de-duplicate (p,t,n) triples in first-seen order
  std::map<OBJIndex, uint32_t> imap;
  for (const OBJIndex& id : inds) {
    auto it = imap.find(id);
    if (it != imap.end()) { out.idx.push_back(it->second); continue; }
    long pi = std::get<0>(id), ti = std::get<1>(id), ni = std::get<2>(id);
    if (pi < 1 || (size_t)pi > pos.size()) bad("OBJ position index out of range in " + path);
    if (ti && (ti < 1 || (size_t)ti > uvs.size())) bad("OBJ uv index out of range in " + path);
    if (ni && (ni < 1 || (size_t)ni > norms.size())) bad("OBJ normal index out of range in " + path);
    uint32_t next = (uint32_t)(out.pos.size() / 3);
    V3 p = pos[pi - 1];
    V3 n = ni ? norms[ni - 1] : V3{0, 0, 0};
    std::pair<double, double> t = ti ? uvs[ti - 1] : std::pair<double, double>(0, 0);
    out.pos.insert(out.pos.end(), {p.x, p.y, p.z});
    out.nrm.insert(out.nrm.end(), {n.x, n.y, n.z});
    out.uv.insert(out.uv.end(), {t.first, t.second});
    out.idx.push_back(next);
    imap.emplace(id, next);
  }
  // Mesh.hs:105-109 `faces` is partial: a trailing 1-2 indices would crash the reference.
  if (out.idx.size() % 3) bad("OBJ index count is not a multiple of 3 in " + path);
}

// Mesh.hs:89-101
void transform_mesh(rh_loaded::Mesh& m, const Transform& t) {
  size_t n = m.pos.size() / 3;
  for (size_t i = 0; i < n; i++) {
    V3 p = xform(t, {m.pos[3 * i], m.pos[3 * i + 1], m.pos[3 * i + 2]});
    m.pos[3 * i] = p.x; m.pos[3 * i + 1] = p.y; m.pos[3 * i + 2] = p.z;
    if (t.kind != Transform::Translate) {  // every other transform is applied to normals too (App. A-P4)
      V3 q = xform(t, {m.nrm[3 * i], m.nrm[3 * i + 1], m.nrm[3 * i + 2]});
      m.nrm[3 * i] = q.x; m.nrm[3 * i + 1] = q.y; m.nrm[3 * i + 2] = q.z;
    }
  }
}

// Bitmap.hs:20-37
int load_ppm_texture(const std::string& path, rh_loaded& L) {
  std::string content;
  if (!read_file(path, content)) bad("cannot open texture " + path);
  auto lines = split_lines(content);
  if (lines.size() < 3) bad("texture " + path + " has no header");
  auto wh = words(lines[1]);
  if (wh.size() < 2) bad("texture " + path + ": bad size line");
  long w = strtol(wh[0].c_str(), nullptr, 10), h = strtol(wh[1].c_str(), nullptr, 10);
  std::vector<double> vals;
  for (size_t i = 3; i < lines.size(); i++)
    for (auto& wd : words(lines[i])) vals.push_back(read_double(wd) / 255);
  size_t ntex = vals.size() / 3;  // `colors` drops a trailing partial triple
  if (w <= 0 || h <= 0 || ntex < (size_t)(w * h)) bad("texture " + path + ": too few texels");
  rh_texture t{};
  t.w = (int32_t)w;
  t.h = (int32_t)h;
  t.offset = L.texels.size() / 3;
  L.texels.insert(L.texels.end(), vals.begin(), vals.begin() + 3 * ntex);
  L.textures.push_back(t);
  return (int)L.textures.size() - 1;
}

std::string join_path(const std::string& base, const std::string& rel) {
  if (!rel.empty() && rel[0] == '/') return rel;
  if (base.empty()) return rel;
  return base + "/" + rel;
}

void parse_colormap(const JValue& o, const std::string& base, rh_loaded& L, rh_material& m) {  // JSON.hs:40-50
  std::string kind = str(o, "type");
  if (kind == "flat") { m.cmap_kind = RH_CMAP_FLAT; color3(o, "color", m.color1); }
  else if (kind == "checker") {
    m.cmap_kind = RH_CMAP_CHECKER;
    color3(o, "color1", m.color1);
    color3(o, "color2", m.color2);
    m.size = num(o, "size");
  } else if (kind == "texture") {
    m.cmap_kind = RH_CMAP_TEXTURE;
    m.texture = load_ppm_texture(join_path(base, str(o, "fileName")), L);
  } else bad("Unknown type for color map " + kind);
}

rh_material parse_material(const JValue& o, const std::string& base, rh_loaded& L) {  // JSON.hs:52-61
  rh_material m{};
  m.texture = -1;
  std::string kind = str(o, "type");
  if (kind == "mirror") { m.kind = RH_MAT_MIRROR; m.ior = num(o, "ior"); }
  else if (kind == "diffuse") { m.kind = RH_MAT_DIFFUSE; parse_colormap(field(o, "cd"), base, L, m); }
  else if (kind == "plastic") { m.kind = RH_MAT_PLASTIC; parse_colormap(field(o, "cd"), base, L, m); m.ior = num(o, "ior"); }
  else if (kind == "emmit") { m.kind = RH_MAT_EMMIT; color3(o, "ce", m.color1); }
  else if (kind == "transparent") { m.kind = RH_MAT_TRANSPARENT; m.ior = num(o, "ior"); }
  else if (kind == "showNormal") m.kind = RH_MAT_SHOWNORMAL;  // no JSON tag in the reference (App. A-M1); harness extension
  else if (kind == "showUV") m.kind = RH_MAT_SHOWUV;
  else bad("Unknown type for material " + kind);
  return m;
}

rh_light parse_light(const JValue& o) {  // JSON.hs:63-72
  rh_light l{};
  std::string kind = str(o, "type");
  if (kind == "directional") { l.kind = RH_LIGHT_DIRECTIONAL; vec3(o, "direction", l.vec); color3(o, "color", l.color); }
  else if (kind == "point") { l.kind = RH_LIGHT_POINT; vec3(o, "position", l.vec); color3(o, "color", l.color); l.radius = num(o, "radius"); }
  else if (kind == "sphere") {  // no JSON tag in the reference: a point light that emits from its ball (rh_light, RH_LIGHT_SPHERE)
    l.kind = RH_LIGHT_SPHERE; vec3(o, "position", l.vec); color3(o, "color", l.color); l.radius = num(o, "radius");
  }
  else bad("Unknown type for light " + kind);
  return l;
}

void parse_camera(const JValue& o, rh_camera& c) {  // JSON.hs:99-105, 74-84
  vec3(o, "position", c.position);
  vec3(o, "target", c.target);
  vec3(o, "up", c.up);
  const JValue& p = field(o, "projection");
  std::string kind = str(p, "type");
  if (kind == "orthographic") {
    c.projection = RH_PROJ_ORTHOGRAPHIC;
    c.proj_width = num(p, "width");
    c.proj_height = num(p, "height");
  } else if (kind == "perspective") {
    c.projection = RH_PROJ_PERSPECTIVE;
    c.fovy = num(p, "fovy");
    c.proj_width = num(p, "width");
    c.proj_height = num(p, "height");
    c.near_ = num(p, "near");
  } else if (kind == "thinLens") {  // no JSON tag in the reference: depth of field (rh_camera, RH_PROJ_THIN_LENS)
    c.projection = RH_PROJ_THIN_LENS;
    c.fovy = num(p, "fovy");
    c.proj_width = num(p, "aperture");
    c.proj_height = num(p, "focusDistance");
  } else bad("Unknown type for projection " + kind);
}

void build_from_json(const JValue& root, const std::string& base, rh_loaded& L) {
  const JValue& scene = field(root, "scene");  // JSON.hs:135-141
  parse_camera(field(root, "camera"), L.camera);
  L.width = (int32_t)num(root, "width");
  L.height = (int32_t)num(root, "height");
  L.max_depth = (int32_t)num(root, "maxDepth");
  const JValue& objs = field(scene, "objects");  // JSON.hs:129-133
  const JValue& lights = field(scene, "lights");
  if (objs.kind != JValue::Arr || lights.kind != JValue::Arr) bad("objects / lights must be arrays");
  for (const JValue& o : objs.arr) {  // Descriptors.hs:44-55
    const JValue& g = field(o, "geometry");
    rh_raw_object ro{};
    std::unique_ptr<rh_loaded::Mesh> mesh;
    std::string kind = str(g, "type");
    if (kind == "sphere") {
      ro.kind = RH_OBJ_SPHERE;
      vec3(g, "center", ro.a);
      ro.b[0] = num(g, "radius");
    } else if (kind == "plane") {
      ro.kind = RH_OBJ_PLANE;
      vec3(g, "point", ro.a);
      vec3(g, "normal", ro.b);
      vec3(g, "tangent", ro.c);
    } else if (kind == "mesh") {
      ro.kind = RH_OBJ_MESH;
      std::string fn = str(g, "fileName");
      Transform t = parseTransform(field(g, "transform"));  // mandatory, JSON.hs:119-121
      mesh = std::make_unique<rh_loaded::Mesh>();
      load_obj(join_path(base, fn), *mesh);
      transform_mesh(*mesh, t);
    } else bad("Unknown type for geometry " + kind);
    ro.material = (int32_t)L.materials.size();
    L.materials.push_back(parse_material(field(o, "material"), base, L));
    L.objects.push_back(ro);
    L.meshes.push_back(std::move(mesh));
  }
  for (const JValue& l : lights.arr) L.lights.push_back(parse_light(l));
  L.finalize();
}

// ------------------------------------------------------------------ SplitMix64
struct SplitMix64 {
  uint64_t s;
  explicit SplitMix64(uint64_t seed) : s(seed) {}
  uint64_t next() {
    uint64_t z = (s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
  }
  double uniform01() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }
  double uniform(double a, double b) { return a + (b - a) * uniform01(); }
};

// SplitMix64 is counter-based (state after k steps = seed + k * gamma), so any stretch of the stream can be produced on
// its own: the generators below fill [first_pixel, first_pixel + n_pixels) of the full-frame stream, on several threads.
template <class T>
void sample_offsets_at(uint64_t seed, uint64_t first_pixel, uint64_t n_pixels, int spp, T* out) {
  const uint64_t n = n_pixels * (uint64_t)spp * 2, first = first_pixel * (uint64_t)spp * 2;
  const unsigned threads = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>(std::min(32u, std::max(1u, std::thread::hardware_concurrency())), n >> 20));
  auto work = [=](uint64_t b, uint64_t e) {
    SplitMix64 rng(seed + (first + b) * 0x9E3779B97F4A7C15ull);
    for (uint64_t i = b; i < e; i++) out[i] = (T)(rng.uniform01() - 0.5);
  };
  if (threads == 1) {
    work(0, n);
    return;
  }
  std::vector<std::thread> pool;
  for (unsigned t = 0; t < threads; t++) pool.emplace_back(work, n * t / threads, n * (t + 1) / threads);
  for (std::thread& t : pool) t.join();
}
// ------------------------------------------------------------------ pack I/O
const char kPackMagic[8] = {'R', 'H', 'P', 'K', '0', '0', '0', '1'};
template <class T> void wr(FILE* f, const T* p, size_t n) { if (n && fwrite(p, sizeof(T), n, f) != n) bad("pack write failed"); }
template <class T> void rd(FILE* f, T* p, size_t n) { if (n && fread(p, sizeof(T), n, f) != n) bad("pack truncated"); }

}  // namespace

extern "C" {

int rh_load_json(const char* json_path, const char* base_dir, rh_loaded** out) {
  if (!json_path || !out) return rh::set_error(RH_ERR_ARG, "rh_load_json: null argument");
  std::string text;
  if (!read_file(json_path, text)) return rh::set_error(RH_ERR_IO, std::string("cannot open ") + json_path);
  JParser jp{text.data(), text.data() + text.size(), {}};
  JValue root;
  if (!jp.value(root)) return rh::set_error(RH_ERR_IO, "Failed to read scene: " + jp.err);  // RayHs.hs:226
  auto L = std::make_unique<rh_loaded>();
  try {
    build_from_json(root, base_dir ? base_dir : "", *L);
  } catch (const ParseError& e) {
    return rh::set_error(RH_ERR_IO, "Failed to read scene: " + e.msg);
  } catch (const std::bad_alloc&) {
    return rh::set_error(RH_ERR_OOM, "out of host memory loading scene");
  }
  *out = L.release();
  return RH_OK;
}

int rh_save_pack(const rh_loaded* L, const char* path) {
  if (!L || !path) return rh::set_error(RH_ERR_ARG, "rh_save_pack: null argument");
  FILE* f = fopen(path, "wb");
  if (!f) return rh::set_error(RH_ERR_IO, std::string("cannot create ") + path);
  try {
    wr(f, kPackMagic, 8);
    int32_t hdr[3] = {L->width, L->height, L->max_depth};
    wr(f, hdr, 3);
    wr(f, &L->camera, 1);
    uint32_t counts[4] = {(uint32_t)L->objects.size(), (uint32_t)L->materials.size(), (uint32_t)L->lights.size(),
                          (uint32_t)L->textures.size()};
    wr(f, counts, 4);
    wr(f, L->materials.data(), L->materials.size());
    wr(f, L->lights.data(), L->lights.size());
    wr(f, L->textures.data(), L->textures.size());
    // texels: one byte each when every value is k/255 exactly (Bitmap.hs:28-29), else doubles
    uint64_t nt = L->texels.size();
    uint8_t as_bytes = 1;
    for (double v : L->texels) {
      double k = std::nearbyint(v * 255);
      if (k < 0 || k > 255 || k / 255 != v) { as_bytes = 0; break; }
    }
    wr(f, &nt, 1);
    wr(f, &as_bytes, 1);
    if (as_bytes) {
      std::vector<uint8_t> b(nt);
      for (uint64_t i = 0; i < nt; i++) b[i] = (uint8_t)std::nearbyint(L->texels[i] * 255);
      wr(f, b.data(), nt);
    } else wr(f, L->texels.data(), nt);
    for (size_t i = 0; i < L->objects.size(); i++) {
      rh_raw_object o = L->objects[i];
      o.positions = o.normals = o.uvs = nullptr;
      o.indices = nullptr;
      wr(f, &o, 1);
      const rh_loaded::Mesh* m = L->meshes[i].get();
      if (m) {
        wr(f, m->pos.data(), m->pos.size());
        wr(f, m->nrm.data(), m->nrm.size());
        wr(f, m->uv.data(), m->uv.size());
        wr(f, m->idx.data(), m->idx.size());
      }
    }
  } catch (const ParseError& e) {
    fclose(f);
    return rh::set_error(RH_ERR_IO, e.msg);
  }
  fclose(f);
  return RH_OK;
}

int rh_load_pack(const char* path, rh_loaded** out) {
  if (!path || !out) return rh::set_error(RH_ERR_ARG, "rh_load_pack: null argument");
  FILE* f = fopen(path, "rb");
  if (!f) return rh::set_error(RH_ERR_IO, std::string("cannot open ") + path);
  auto L = std::make_unique<rh_loaded>();
  try {
    char magic[8];
    rd(f, magic, 8);
    if (memcmp(magic, kPackMagic, 8)) bad("not a scene pack");
    int32_t hdr[3];
    rd(f, hdr, 3);
    L->width = hdr[0]; L->height = hdr[1]; L->max_depth = hdr[2];
    rd(f, &L->camera, 1);
    uint32_t counts[4];
    rd(f, counts, 4);
    if (counts[0] > (1u << 24) || counts[1] > (1u << 24) || counts[2] > (1u << 20) || counts[3] > (1u << 20)) bad("pack header corrupt");
    L->materials.resize(counts[1]);
    L->lights.resize(counts[2]);
    L->textures.resize(counts[3]);
    rd(f, L->materials.data(), counts[1]);
    rd(f, L->lights.data(), counts[2]);
    rd(f, L->textures.data(), counts[3]);
    uint64_t nt;
    uint8_t as_bytes;
    rd(f, &nt, 1);
    rd(f, &as_bytes, 1);
    L->texels.resize(nt);
    if (as_bytes) {
      std::vector<uint8_t> b(nt);
      rd(f, b.data(), nt);
      for (uint64_t i = 0; i < nt; i++) L->texels[i] = (double)b[i] / 255;
    } else rd(f, L->texels.data(), nt);
    for (uint32_t i = 0; i < counts[0]; i++) {
      rh_raw_object o;
      rd(f, &o, 1);
      std::unique_ptr<rh_loaded::Mesh> m;
      if (o.kind == RH_OBJ_MESH) {
        m = std::make_unique<rh_loaded::Mesh>();
        m->pos.resize((size_t)o.n_verts * 3);
        m->nrm.resize((size_t)o.n_verts * 3);
        m->uv.resize((size_t)o.n_verts * 2);
        m->idx.resize(o.n_indices);
        rd(f, m->pos.data(), m->pos.size());
        rd(f, m->nrm.data(), m->nrm.size());
        rd(f, m->uv.data(), m->uv.size());
        rd(f, m->idx.data(), m->idx.size());
      }
      L->objects.push_back(o);
      L->meshes.push_back(std::move(m));
    }
  } catch (const ParseError& e) {
    fclose(f);
    return rh::set_error(RH_ERR_IO, std::string(path) + ": " + e.msg);
  } catch (const std::bad_alloc&) {
    fclose(f);
    return rh::set_error(RH_ERR_OOM, "out of host memory loading pack");
  }
  fclose(f);
  L->finalize();
  *out = L.release();
  return RH_OK;
}

// SURVEY 8d config C5.  Draw order: per triangle centroid(3), e1(3), e2(3); then per sphere
// centre(3), radius(1), colour(3).  Object order: mesh, spheres, floor plane.
int rh_make_synthetic(uint64_t n_tris, uint32_t n_spheres, uint64_t seed, rh_loaded** out) {
  if (!out) return rh::set_error(RH_ERR_ARG, "rh_make_synthetic: null out");
  if (n_tris > 0x3FFFFFFFull / 3) return rh::set_error(RH_ERR_ARG, "rh_make_synthetic: too many triangles");
  try {
    auto L = std::make_unique<rh_loaded>();
    SplitMix64 rng(seed);
    auto mesh = std::make_unique<rh_loaded::Mesh>();
    mesh->pos.resize(n_tris * 9);
    mesh->nrm.resize(n_tris * 9);
    mesh->uv.assign(n_tris * 6, 0.0);
    mesh->idx.resize(n_tris * 3);
    for (uint64_t i = 0; i < n_tris; i++) {
      double c[3], e1[3], e2[3];
      for (double& v : c) v = rng.uniform(-1, 1);
      for (double& v : e1) v = rng.uniform(-0.01, 0.01);
      for (double& v : e2) v = rng.uniform(-0.01, 0.01);
      double p0[3], p1[3], p2[3];
      for (int k = 0; k < 3; k++) {
        p0[k] = c[k] - (e1[k] + e2[k]) / 3;
        p1[k] = p0[k] + e1[k];
        p2[k] = p0[k] + e2[k];
      }
      V3 n = vcross({e1[0], e1[1], e1[2]}, {e2[0], e2[1], e2[2]});
      double len = sqrt(n.x * n.x + n.y * n.y + n.z * n.z);
      if (len > 0) n = {n.x / len, n.y / len, n.z / len};
      else n = {0, 1, 0};
      double* P = &mesh->pos[i * 9];
      double* N = &mesh->nrm[i * 9];
      for (int k = 0; k < 3; k++) { P[k] = p0[k]; P[3 + k] = p1[k]; P[6 + k] = p2[k]; }
      for (int v = 0; v < 3; v++) { N[3 * v] = n.x; N[3 * v + 1] = n.y; N[3 * v + 2] = n.z; }
      for (int v = 0; v < 3; v++) mesh->idx[i * 3 + v] = (uint32_t)(i * 3 + v);
    }
    auto add_mat = [&](rh_material m) { L->materials.push_back(m); return (int32_t)L->materials.size() - 1; };
    {
      rh_material m{};
      m.kind = RH_MAT_PLASTIC; m.cmap_kind = RH_CMAP_FLAT; m.ior = 1.5; m.texture = -1;
      m.color1[0] = m.color1[1] = m.color1[2] = 0.8;
      rh_raw_object o{};
      o.kind = RH_OBJ_MESH;
      o.material = add_mat(m);
      L->objects.push_back(o);
      L->meshes.push_back(std::move(mesh));
    }
    for (uint32_t i = 0; i < n_spheres; i++) {
      rh_raw_object o{};
      o.kind = RH_OBJ_SPHERE;
      for (int k = 0; k < 3; k++) o.a[k] = rng.uniform(-1, 1);
      o.b[0] = rng.uniform(0.005, 0.02);
      rh_material m{};
      m.texture = -1;
      m.cmap_kind = RH_CMAP_FLAT;
      for (int k = 0; k < 3; k++) m.color1[k] = rng.uniform(0.2, 1.0);
      if (i % 3 == 0) m.kind = RH_MAT_DIFFUSE;
      else if (i % 3 == 1) { m.kind = RH_MAT_PLASTIC; m.ior = 1.9; }
      else { m.kind = RH_MAT_MIRROR; m.ior = 0.1; }
      o.material = add_mat(m);
      L->objects.push_back(o);
      L->meshes.push_back(nullptr);
    }
    {  // floor: data/dragon.json's checker plastic plane y = -1
      rh_raw_object o{};
      o.kind = RH_OBJ_PLANE;
      o.a[1] = -1; o.b[1] = 1; o.c[2] = 1;
      rh_material m{};
      m.kind = RH_MAT_PLASTIC; m.cmap_kind = RH_CMAP_CHECKER; m.ior = 2; m.size = 0.5; m.texture = -1;
      m.color2[0] = m.color2[1] = m.color2[2] = 2;
      o.material = add_mat(m);
      L->objects.push_back(o);
      L->meshes.push_back(nullptr);
    }
    auto add_light = [&](double x, double y, double z, double c) {
      rh_light l{};
      l.kind = RH_LIGHT_POINT;
      l.vec[0] = x; l.vec[1] = y; l.vec[2] = z;
      l.color[0] = l.color[1] = l.color[2] = c;
      l.radius = 0.1;
      L->lights.push_back(l);
    };
    add_light(0.0, 0.9, 0.75, 150);  // data/dragon.json lights
    add_light(-0.5, -0.2, 0.12, 50);
    add_light(0.4, -0.1, -0.1, 50);
    rh_camera& c = L->camera;  // data/dragon.json camera
    c.position[2] = -2;
    c.up[1] = 1;
    c.projection = RH_PROJ_PERSPECTIVE;
    c.fovy = 0.9272952180016123;
    c.proj_width = c.proj_height = 2;
    c.near_ = 2;
    L->width = 7680; L->height = 4320; L->max_depth = 3;
    L->finalize();
    *out = L.release();
  } catch (const std::bad_alloc&) {
    return rh::set_error(RH_ERR_OOM, "out of host memory generating synthetic scene");
  }
  return RH_OK;
}

const rh_raw_scene* rh_loaded_raw(const rh_loaded* l) { return l ? &l->raw : nullptr; }
const rh_camera* rh_loaded_camera(const rh_loaded* l) { return l ? &l->camera : nullptr; }
void rh_loaded_size(const rh_loaded* l, int32_t* w, int32_t* h, int32_t* d) {
  if (!l) return;
  if (w) *w = l->width;
  if (h) *h = l->height;
  if (d) *d = l->max_depth;
}
void rh_loaded_destroy(rh_loaded* l) { delete l; }

// RayHs.hs:173-188: per pixel 2*spp uniform [0,1) draws, x before y, pair = (x-0.5, y-0.5).
// The reference's StdGen algorithm is un-pinned (rayhs.cabal: random -any; SURVEY 8c);
// offsets are INPUTS to the render call, so any host stream of this shape is valid.
void rh_sample_offsets_f64(uint64_t seed, uint64_t n_pixels, int spp, double* out) { sample_offsets_at(seed, 0, n_pixels, spp, out); }
void rh_sample_offsets_f32(uint64_t seed, uint64_t n_pixels, int spp, float* out) { sample_offsets_at(seed, 0, n_pixels, spp, out); }
void rh_sample_offsets_f64_at(uint64_t seed, uint64_t first_pixel, uint64_t n_pixels, int spp, double* out) {
  sample_offsets_at(seed, first_pixel, n_pixels, spp, out);
}

// Image.hs:60-75: "P3\nW H\n255\n", rows joined by "\n", each pixel "R G B" + two spaces, no trailing newline.
int rh_write_ppm(const char* path, const uint8_t* rgb, int width, int height) {
  if (!path || !rgb || width <= 0 || height <= 0) return rh::set_error(RH_ERR_ARG, "rh_write_ppm: bad argument");
  FILE* f = fopen(path, "wb");
  if (!f) return rh::set_error(RH_ERR_IO, std::string("cannot create ") + path);
  static const char digits[] = "0123456789";
  std::vector<char> line;
  line.reserve((size_t)width * 14 + 32);
  fprintf(f, "P3\n%d %d\n255\n", width, height);
  for (int y = 0; y < height; y++) {
    line.clear();
    if (y) line.push_back('\n');
    const uint8_t* row = rgb + (size_t)y * width * 3;
    for (int x = 0; x < width; x++) {
      for (int k = 0; k < 3; k++) {
        unsigned v = row[3 * x + k];
        if (v >= 100) line.push_back(digits[v / 100]);
        if (v >= 10) line.push_back(digits[(v / 10) % 10]);
        line.push_back(digits[v % 10]);
        line.push_back(' ');
      }
      line.push_back(' ');  // "R G B" ++ "  "
    }
    if (fwrite(line.data(), 1, line.size(), f) != line.size()) {
      fclose(f);
      return rh::set_error(RH_ERR_IO, "short write");
    }
  }
  fclose(f);
  return RH_OK;
}

}  // extern "C"
