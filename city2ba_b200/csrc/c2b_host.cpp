// c2b_host.cpp — host-only entry points of libcity2ba_cuda.so: the deterministic input
// generators of `city2ba synthetic` / `synthetic-line` (camera and point lattices,
// src/synthetic.rs:178-258, 323-344), the city-block box mesh that stands in for the OBJ scene
// on synthetic cities, and SnavelyCamera helpers for the host mirror.  No GPU work here.
// Compiled with -ffp-contract=off (c2b_math.cuh's host path relies on it).
#include <algorithm>
#include <cmath>
#include <cstring>

#include "../../include/city2ba_cuda.h"
#include "c2b_math.cuh"

using namespace c2b;

namespace {
// cgmath: Rad::from(Deg(d)) = d * (pi/180)
inline double deg_to_rad(double deg) { return deg * (3.14159265358979323846 / 180.0); }
}  // namespace

extern "C" {

uint64_t c2b_grid_num_cameras(uint64_t cpb, uint64_t n) { return 4 * cpb * n * (n + 1); }
uint64_t c2b_grid_num_points(uint64_t ppb, uint64_t n) { return 12 * ppb * n * (n + 1); }

// src/synthetic.rs:178-210: for every lattice corner (bx,by) and i < cpb, two cameras on the
// x-street (yaw -90 then +90 degrees) if bx != n, two on the z-street (yaw 180, identity) if by != n
int c2b_grid_cameras(uint64_t cpb, uint64_t n, double L, double h, double *out) {
  if (!out) return C2B_ERR_INVALID;
  double Rm90[9], Rp90[9], R180[9];
  const double R1[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  from_angle_y(deg_to_rad(-90.), Rm90);
  from_angle_y(deg_to_rad(90.), Rp90);
  from_angle_y(deg_to_rad(180.), R180);
  double *w = out;
  for (uint64_t bx = 0; bx <= n; ++bx) {
    const double ox = L * (double)bx;
    for (uint64_t by = 0; by <= n; ++by) {
      const double oz = L * (double)by;
      for (uint64_t i = 0; i < cpb; ++i) {
        const double frac = (double)i / (double)cpb * L;
        if (bx != n) {
          V3 pos{ox + frac, h, oz};
          camera_from_position_direction(pos, Rm90, w);
          w += C2B_CAM_STRIDE;
          camera_from_position_direction(pos, Rp90, w);
          w += C2B_CAM_STRIDE;
        }
        if (by != n) {
          V3 pos{ox, h, oz + frac};
          camera_from_position_direction(pos, R180, w);
          w += C2B_CAM_STRIDE;
          camera_from_position_direction(pos, R1, w);
          w += C2B_CAM_STRIDE;
        }
      }
    }
  }
  return C2B_OK;
}

// src/synthetic.rs:213-258: per (bx,by,i) six points per street: two wall points at
// point_height, two ground points at +-inset and two at +-inset/2 (shifted by step/2)
int c2b_grid_points(uint64_t ppb, uint64_t n, double L, double inset, double ph, double *out) {
  if (!out) return C2B_ERR_INVALID;
  double *w = out;
  auto push = [&](double x, double y, double z) {
    w[0] = x;
    w[1] = y;
    w[2] = z;
    w += 3;
  };
  const double step = (L - inset * 2.) / (double)ppb;
  for (uint64_t bx = 0; bx <= n; ++bx) {
    const double ox = L * (double)bx;
    for (uint64_t by = 0; by <= n; ++by) {
      const double oz = L * (double)by;
      for (uint64_t i = 0; i < ppb; ++i) {
        if (bx != n) {
          const double lx = ox + inset + (double)i * step;
          const double mx = lx + step / 2.;
          push(lx, ph, oz - inset);
          push(lx, ph, oz + inset);
          push(mx, 0., oz - inset);
          push(mx, 0., oz + inset);
          push(mx, 0., oz - inset / 2.);
          push(mx, 0., oz + inset / 2.);
        }
        if (by != n) {
          const double lz = oz + inset + (double)i * step;
          const double mz = lz + step / 2.;
          push(ox - inset, ph, lz);
          push(ox + inset, ph, lz);
          push(ox - inset, 0., mz);
          push(ox + inset, 0., mz);
          push(ox - inset / 2., 0., mz);
          push(ox + inset / 2., 0., mz);
        }
      }
    }
  }
  return C2B_OK;
}

// src/synthetic.rs:323-333
int c2b_line_cameras(uint64_t nc, double length, double h, double *out) {
  if (!out) return C2B_ERR_INVALID;
  double R180[9];
  from_angle_y(deg_to_rad(180.), R180);
  for (uint64_t i = 0; i < nc; ++i) {
    V3 pos{0., h, (double)i * length / (double)(nc - 1)};
    camera_from_position_direction(pos, R180, out + C2B_CAM_STRIDE * i);
  }
  return C2B_OK;
}

// src/synthetic.rs:334-344
int c2b_line_points(uint64_t np, double length, double off, double ph, double *out) {
  if (!out) return C2B_ERR_INVALID;
  for (uint64_t i = 0; i < np; ++i) {
    out[3 * i] = (i % 2 == 0) ? -off : off;
    out[3 * i + 1] = ph;
    out[3 * i + 2] = (double)(i / 2) * length / (double)(np / 2 - 1);
  }
  return C2B_OK;
}

// one axis-aligned box per city block: footprint [b*L+inset, (b+1)*L-inset]^2, y in [0,H];
// vertex k: bit0 -> x hi, bit1 -> y hi, bit2 -> z hi; 4 walls + floor + roof = 12 triangles
int c2b_city_mesh(uint64_t n, double L, double inset, double H, float *xyz, uint32_t *tri) {
  if (!xyz || !tri) return C2B_ERR_INVALID;
  static const uint32_t F[12][3] = {{0, 2, 1}, {1, 2, 3}, {4, 5, 6}, {5, 7, 6}, {0, 4, 2}, {2, 4, 6},
                                    {1, 3, 5}, {3, 7, 5}, {0, 1, 4}, {1, 5, 4}, {2, 6, 3}, {3, 6, 7}};
  uint64_t b = 0;
  for (uint64_t bx = 0; bx < n; ++bx)
    for (uint64_t bz = 0; bz < n; ++bz, ++b) {
      const double x[2] = {(double)bx * L + inset, (double)(bx + 1) * L - inset};
      const double y[2] = {0.0, H};
      const double z[2] = {(double)bz * L + inset, (double)(bz + 1) * L - inset};
      for (uint32_t k = 0; k < 8; ++k) {
        float *v = xyz + 3 * (8 * b + k);
        v[0] = (float)x[k & 1];
        v[1] = (float)y[(k >> 1) & 1];
        v[2] = (float)z[(k >> 2) & 1];
      }
      for (uint32_t f = 0; f < 12; ++f)
        for (int j = 0; j < 3; ++j) tri[3 * (12 * b + f) + j] = (uint32_t)(8 * b) + F[f][j];
    }
  return C2B_OK;
}

void c2b_camera_center(const double *cam, double out[3]) {
  V3 c = camera_center(cam);
  out[0] = c.x;
  out[1] = c.y;
  out[2] = c.z;
}
void c2b_camera_project_world(const double *cam, const double p[3], double out[3]) {
  V3 r = project_world(cam, V3{p[0], p[1], p[2]});
  out[0] = r.x;
  out[1] = r.y;
  out[2] = r.z;
}
void c2b_camera_project(const double *cam, const double pc[3], double out[2]) {
  project(cam[12], cam[13], cam[14], V3{pc[0], pc[1], pc[2]}, out[0], out[1]);
}
void c2b_camera_from_position_direction(const double pos[3], const double R[9], double *cam_out) {
  double Rc[9];
  memcpy(Rc, R, sizeof Rc);
  camera_from_position_direction(V3{pos[0], pos[1], pos[2]}, Rc, cam_out);
}
void c2b_camera_transform(const double *cam, const double dR[9], const double dloc[3],
                          double *cam_out) {
  double c[15], out[15];
  memcpy(c, cam, sizeof c);
  camera_transform(c, dR, V3{dloc[0], dloc[1], dloc[2]}, out);
  memcpy(cam_out, out, sizeof out);
}

// cgmath Quaternion::from(Matrix3) (Shepperd branches) as include/city2ba.hpp's detail::quat_from_mat: m column-major,
// q = (s, x, y, z)
static void quat_from_mat(const double *m, double q[4]) {
  auto M = [&](int c, int r) { return m[c * 3 + r]; };
  const double trace = (M(0, 0) + M(1, 1)) + M(2, 2);
  if (trace >= 0.0) {
    double s = std::sqrt(1.0 + trace);
    const double w = 0.5 * s;
    s = 0.5 / s;
    q[0] = w, q[1] = (M(1, 2) - M(2, 1)) * s, q[2] = (M(2, 0) - M(0, 2)) * s, q[3] = (M(0, 1) - M(1, 0)) * s;
  } else if (M(0, 0) > M(1, 1) && M(0, 0) > M(2, 2)) {
    double s = std::sqrt(((M(0, 0) - M(1, 1)) - M(2, 2)) + 1.0);
    const double x = 0.5 * s;
    s = 0.5 / s;
    q[0] = (M(1, 2) - M(2, 1)) * s, q[1] = x, q[2] = (M(1, 0) + M(0, 1)) * s, q[3] = (M(0, 2) + M(2, 0)) * s;
  } else if (M(1, 1) > M(2, 2)) {
    double s = std::sqrt(((M(1, 1) - M(0, 0)) - M(2, 2)) + 1.0);
    const double y = 0.5 * s;
    s = 0.5 / s;
    q[0] = (M(2, 0) - M(0, 2)) * s, q[1] = (M(1, 0) + M(0, 1)) * s, q[2] = y, q[3] = (M(2, 1) + M(1, 2)) * s;
  } else {
    double s = std::sqrt(((M(2, 2) - M(0, 0)) - M(1, 1)) + 1.0);
    const double z = 0.5 * s;
    s = 0.5 / s;
    q[0] = (M(0, 1) - M(1, 0)) * s, q[1] = (M(0, 2) + M(2, 0)) * s, q[2] = (M(2, 1) + M(1, 2)) * s, q[3] = z;
  }
}

// SnavelyCamera::to_vec (src/baproblem.rs:192-202, to_rodrigues :93-102): the same operations in the same order as
// include/city2ba.hpp's to_vec / to_rodrigues / detail::quat_from_mat, so that the BAL writer's camera lines equal
// the C++ mirror's bit for bit (acos is the host libm's; the device's differs)
void c2b_camera_to_vec(const double *cam, double out[9]) {
  double q[4];
  quat_from_mat(cam, q);
  const double angle = 2.0 * std::acos(std::max(-1.0, std::min(1.0, q[0])));
  const double d = 1.0 - q[0] * q[0];
  if (d < 2.220446049250313e-16) {
    out[0] = out[1] = out[2] = 0.0;
  } else {
    const double sd = std::sqrt(d);
    const double a[3] = {q[1] / sd, q[2] / sd, q[3] / sd};
    const double inv = 1.0 / std::sqrt((a[0] * a[0] + a[1] * a[1]) + a[2] * a[2]);
    for (int k = 0; k < 3; ++k) out[k] = a[k] * inv * angle;
  }
  for (int k = 0; k < 6; ++k) out[3 + k] = cam[9 + k];
}

// SnavelyCamera::from_vec (src/baproblem.rs:180-190, from_rodrigues :78-90): the operations of include/city2ba.hpp's
// from_vec / from_rodrigues / from_axis_angle / detail::mat_from_quat in the same order, so that the BAL reader's
// camera records equal the C++ mirror's bit for bit (sin / cos / sqrt are the host libm's; the device's differ)
void c2b_camera_from_vec(const double v[9], double *cam_out) {
  const double x[3] = {v[0], v[1], v[2]};
  double R[9];
  const double theta2 = (x[0] * x[0] + x[1] * x[1]) + x[2] * x[2];
  if (theta2 > 2.220446049250313e-16) {
    const double angle = std::sqrt(theta2), inv = 1.0 / angle;
    const double a[3] = {x[0] * inv, x[1] * inv, x[2] * inv};
    const double s = std::sin(angle), c = std::cos(angle), k = 1.0 - c;
    const double m[9] = {k * a[0] * a[0] + c,        k * a[0] * a[1] + s * a[2], k * a[0] * a[2] - s * a[1],
                         k * a[0] * a[1] - s * a[2], k * a[1] * a[1] + c,        k * a[1] * a[2] + s * a[0],
                         k * a[0] * a[2] + s * a[1], k * a[1] * a[2] - s * a[0], k * a[2] * a[2] + c};
    memcpy(R, m, sizeof R);
  } else {
    const double m[9] = {1.0, x[2], -x[1], -x[2], 1.0, x[0], x[1], -x[0], 1.0};
    double q[4];
    quat_from_mat(m, q);
    const double s = q[0], qx = q[1], y = q[2], z = q[3];
    const double x2 = qx + qx, y2 = y + y, z2 = z + z;
    const double xx2 = x2 * qx, xy2 = x2 * y, xz2 = x2 * z, yy2 = y2 * y, yz2 = y2 * z, zz2 = z2 * z;
    const double sy2 = y2 * s, sz2 = z2 * s, sx2 = x2 * s;
    const double r[9] = {1.0 - yy2 - zz2, xy2 + sz2, xz2 - sy2, xy2 - sz2, 1.0 - xx2 - zz2, yz2 + sx2,
                         xz2 + sy2, yz2 - sx2, 1.0 - xx2 - yy2};
    memcpy(R, r, sizeof R);
  }
  memcpy(cam_out, R, sizeof R);
  for (int k = 0; k < 6; ++k) cam_out[9 + k] = v[3 + k];
}

}  // extern "C"
