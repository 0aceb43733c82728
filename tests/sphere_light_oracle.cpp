// sphere_light_oracle.cpp — the tests' restatement of sphere lights (RH_LIGHT_SPHERE, beside rh_light in
// include/rayhs_b200.h) on top of the oracle.  TEST INFRASTRUCTURE ONLY.
//
// oracle/oracle.cpp is the reference's restatement and knows only the reference's two light kinds (it treats any other
// kind as a point light at vec); a sphere light is this project's extension.  This file includes oracle.cpp unchanged
// (as oracle/batch.cpp does) and restates accumDiffuse, specular, irradiance and traceRay (RayHs.hs:89-154) on the
// oracle's own lightAt, shadowIntersection, closestIntersection, colorAt and SplitMix64, with each sphere light replaced,
// per shading point, by the point light at its sample.  It shares no code with the product.  tests/sphere_light_oracle.py
// compiles it with the oracle's flags (rayhs_b200/build.py ORACLE_FLAGS: -ffp-contract=off) and folds the samples of a
// pixel (RayHs.hs:156-195).
#include "../oracle/oracle.cpp"

namespace {

uint64_t mix64(uint64_t z) {  // SplitMix64's output function
  z ^= z >> 30;
  z *= 0xBF58476D1CE4E5B9ull;
  z ^= z >> 27;
  z *= 0x94D049BB133111EBull;
  z ^= z >> 31;
  return z;
}

uint64_t bitsOf(double x) {
  uint64_t b;
  std::memcpy(&b, &x, sizeof b);
  return b;
}

// The point of light l's ball that shading point p samples: the first of 16 triples drawn from [-1, 1)^3 by a hash of
// (p, l) that falls inside the unit ball, else the centre, scaled by the radius and moved to the centre.
Vec spherePoint(const rh_light& L, uint32_t l, Vec p) {
  const uint64_t key = bitsOf(p.x) ^ mix64(bitsOf(p.y) ^ mix64(bitsOf(p.z) ^ mix64((uint64_t)l)));
  double a = 0, b = 0, c = 0;
  for (uint64_t j = 0; j < 16; j++) {
    const double x = 2 * splitmix01_at(key, 3 * j) - 1;
    const double y = 2 * splitmix01_at(key, 3 * j + 1) - 1;
    const double z = 2 * splitmix01_at(key, 3 * j + 2) - 1;
    if ((x * x + y * y) + z * z < 1) {
      a = x;
      b = y;
      c = z;
      break;
    }
  }
  const double r = L.radius;
  return {L.vec[0] + r * a, L.vec[1] + r * b, L.vec[2] + r * c};
}

// The light the pair (p, l) sees: a sphere light becomes the point light at its sample, every other light stays.
rh_light pairLight(const rh_light& L, uint32_t l, Vec p) {
  if (L.kind != RH_LIGHT_SPHERE) return L;
  rh_light q = L;
  const Vec s = spherePoint(L, l, p);
  q.kind = RH_LIGHT_POINT;
  q.vec[0] = s.x;
  q.vec[1] = s.y;
  q.vec[2] = s.z;
  return q;
}

Color sTraceRay(const Scene& sc, int depth, int maxDepth, const Ray& ray, Counters& c, int cls, int* hit_obj, int* hit_tri);

// RayHs.hs:89-97
Color sAccumDiffuse(const Scene& sc, Vec p, Vec n, Color color, Counters& c) {
  Color acc = black;
  for (uint32_t l = 0; l < sc.lights.size(); l++) {
    const rh_light q = pairLight(sc.lights[l], l, p);
    Vec ld;
    Color lc;
    lightAt(q, p, &ld, &lc);
    bool shadowed = shadowIntersection(sc, q, rayEps(p, ld), c);
    acc = acc + (shadowed ? black : diffuse(color, lc, ld, n));
  }
  return acc;
}

// RayHs.hs:99-104
Color sSpecular(const Scene& sc, int depth, int maxDepth, Vec v, Vec p, Vec n, Counters& c) {
  if (depth < maxDepth) {
    Vec rdir = reflect(v, n);
    return mul(dot(rdir, n), sTraceRay(sc, depth + 1, maxDepth, rayEps(p, rdir), c, 1, nullptr, nullptr));
  }
  return black;
}

// RayHs.hs:107-147
Color sIrradiance(int d, int maxDepth, const Scene& sc, const rh_material& m, Vec v, Vec p, Vec n, UV uv, Counters& c) {
  switch (m.kind) {
    case RH_MAT_DIFFUSE: {
      Color cd = colorAt(sc, m, uv);
      return mul(0.2, cd) + sAccumDiffuse(sc, p, n, cd, c);
    }
    case RH_MAT_PLASTIC: {
      Color cd = colorAt(sc, m, uv);
      Color diff = sAccumDiffuse(sc, p, n, cd, c);
      return diff + mul(fresnel(m.ior, dot(n, neg(v))), sSpecular(sc, d, maxDepth, v, p, n, c));
    }
    case RH_MAT_MIRROR:
      return mul(fresnel(m.ior, dot(n, neg(v))), sSpecular(sc, d, maxDepth, v, p, n, c));
    case RH_MAT_EMMIT:
      return {m.color1[0], m.color1[1], m.color1[2]};
    case RH_MAT_TRANSPARENT: {
      bool have = false;
      Color radiance = black;
      if (d != maxDepth) {
        Vec refDir;
        if (refract(v, n, 1.0, m.ior, &refDir)) {
          Ray refr = rayEps(p, refDir);
          MatHit out;
          if (closestIntersection(sc, refr, &out, c, 2)) {
            Vec outDir;
            if (refract(refDir, neg(out.n), m.ior, 1.0, &outDir)) {
              radiance = sTraceRay(sc, d + 1, maxDepth, rayEps(out.p, outDir), c, 3, nullptr, nullptr);
              have = true;
            }
          }
        }
      }
      Color spec = mul(fresnel(m.ior, dot(n, neg(v))), sSpecular(sc, d, maxDepth, v, p, n, c));
      if (!have) return spec;
      return mul(1 - r0(m.ior, 1.0), radiance) + spec;
    }
    case RH_MAT_SHOWNORMAL:
      return {n.x, n.y, n.z};
    case RH_MAT_SHOWUV:
      return {uv.u, uv.v, 0};
  }
  return black;
}

// RayHs.hs:149-154
Color sTraceRay(const Scene& sc, int depth, int maxDepth, const Ray& ray, Counters& c, int cls, int* hit_obj, int* hit_tri) {
  MatHit h;
  if (closestIntersection(sc, ray, &h, c, cls)) {
    if (hit_obj) { *hit_obj = h.object; *hit_tri = h.tri; }
    return sIrradiance(depth, maxDepth, sc, sc.materials[h.material], ray.d, h.p, h.n, h.uv, c);
  }
  if (hit_obj) { *hit_obj = -1; *hit_tri = -1; }
  return black;
}

}  // namespace

extern "C" {

// L' of light `light` of the scene for n shading points p[n][3]: out[n][3].  -1: no such light
int sl_sphere_points(void* s, uint32_t light, const double* p, uint64_t n, double* out) {
  const Scene& sc = ((OracleScene*)s)->sc;
  if (light >= sc.lights.size()) return -1;
  for (uint64_t i = 0; i < n; i++) {
    const Vec q = spherePoint(sc.lights[light], light, Vec{p[3 * i], p[3 * i + 1], p[3 * i + 2]});
    out[3 * i] = q.x;
    out[3 * i + 1] = q.y;
    out[3 * i + 2] = q.z;
  }
  return 0;
}

// traceRay sc 0 max_depth r per ray with sphere lights (orc_trace_batch's outputs): colors_out double[n][3], ids_out
// int32[n][2] and counts_out[5] (primary, reflect, probe, exit, shadow).  One thread: the counts are sums either way.
int sl_trace_batch(void* s, const double* rays, uint64_t n, int max_depth, double* colors_out, int32_t* ids_out, uint64_t* counts_out) {
  const Scene& sc = ((OracleScene*)s)->sc;
  Counters c;
  for (uint64_t i = 0; i < n; i++) {
    const double* q = rays + 6 * i;
    int obj, tri;
    const Color col = sTraceRay(sc, 0, max_depth, Ray{{q[0], q[1], q[2]}, {q[3], q[4], q[5]}}, c, 0, &obj, &tri);
    colors_out[3 * i] = col.r;
    colors_out[3 * i + 1] = col.g;
    colors_out[3 * i + 2] = col.b;
    ids_out[2 * i] = obj;
    ids_out[2 * i + 1] = tri;
  }
  for (int k = 0; k < 5; k++) counts_out[k] = c.rays[k];
  return 0;
}

}  // extern "C"
