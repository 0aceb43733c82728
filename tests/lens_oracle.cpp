// lens_oracle.cpp — the tests' restatement of the thin-lens camera (RH_PROJ_THIN_LENS, beside rh_camera in
// include/rayhs_b200.h) on top of the oracle.  TEST INFRASTRUCTURE ONLY.
//
// oracle/oracle.cpp is the reference's restatement and knows only the reference's two projections; a thin lens is this
// project's extension.  This file includes oracle.cpp unchanged (as oracle/batch.cpp does) and adds the lens ray from
// the oracle's own lookAt, normalize, apply and SplitMix64; it shares no code with the product.  tests/lens_oracle.py
// compiles it with the oracle's flags (rayhs_b200/build.py ORACLE_FLAGS: -ffp-contract=off).
#include "../oracle/oracle.cpp"

namespace {

// The lens point (a, b) of image position (px, py), in the unit disk: the first of 16 pairs drawn from [-1, 1)^2 by a
// hash of the position that falls inside it, else the centre.
void lensPoint(double px, double py, double* a, double* b) {
  uint64_t xbits, ybits;
  std::memcpy(&xbits, &px, sizeof xbits);
  std::memcpy(&ybits, &py, sizeof ybits);
  uint64_t m = ybits;  // SplitMix64's output function
  m ^= m >> 30;
  m *= 0xBF58476D1CE4E5B9ull;
  m ^= m >> 27;
  m *= 0x94D049BB133111EBull;
  m ^= m >> 31;
  const uint64_t key = xbits ^ m;
  for (uint64_t j = 0; j < 16; j++) {
    const double x = 2 * splitmix01_at(key, 2 * j) - 1;
    const double y = 2 * splitmix01_at(key, 2 * j + 1) - 1;
    if (x * x + y * y < 1) {
      *a = x;
      *b = y;
      return;
    }
  }
  *a = *b = 0;
}

// rayFromPixel (Projection.hs:22-39) and, for a thin lens of radius R != 0, the lens ray
Ray cameraRay(double w, double h, const rh_camera& cam, double px, double py) {
  if (cam.projection != RH_PROJ_THIN_LENS || cam.proj_width == 0) return rayFromPixel(w, h, cam, px, py);
  const Vec p{cam.position[0], cam.position[1], cam.position[2]};
  const Vec t{cam.target[0], cam.target[1], cam.target[2]};
  const Vec up{cam.up[0], cam.up[1], cam.up[2]};
  double apw, aph;
  aspectSize(w, h, &apw, &aph);
  const double f = 0.5 * h / (std::tan(0.5) * cam.fovy);
  const Vec d = normalize(Vec{apw * (px - (w / 2)) / w, aph * ((-py) + (h / 2)) / h, f});
  const double R = cam.proj_width, F = cam.proj_height;
  double a, b;
  lensPoint(px, py, &a, &b);
  const Vec lens{R * a, R * b, 0};
  const double s = F / d.z;
  const Vec focal{s * d.x, s * d.y, s * d.z};
  const Mat3 mat = lookAt(p, t, up);
  return {apply(mat, lens) + p, apply(mat, normalize(focal - lens))};
}

}  // namespace

extern "C" {

// The camera rays of any rh_camera at n pixel coordinates xy[n][2]: rays_out[n][6] = origin, direction
void lens_camera_rays(const rh_camera* cam, double w, double h, const double* xy, uint64_t n, double* rays_out) {
  for (uint64_t i = 0; i < n; i++) {
    const Ray r = cameraRay(w, h, *cam, xy[2 * i], xy[2 * i + 1]);
    double* o = rays_out + 6 * i;
    o[0] = r.o.x; o[1] = r.o.y; o[2] = r.o.z;
    o[3] = r.d.x; o[4] = r.d.y; o[5] = r.d.z;
  }
}

}  // extern "C"
