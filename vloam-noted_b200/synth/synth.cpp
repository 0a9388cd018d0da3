// synth.cpp -- seeded synthetic lidar sweeps and planted cube maps (SURVEY.md 8d).
//
// Host-only helper shared by tests/ and bench.py so the oracle and the CUDA path
// read identical bytes.  Not part of the product library.
//
// World: ground plane, axis-aligned boxes (buildings) and vertical cylinders
// (poles) on a block grid; a sweep ray-casts every beam through a 2-D uniform
// grid.  Emission order is azimuth-major (all beams of azimuth k, then k+1),
// the Velodyne driver order the reference's startOri/endOri/halfPassed logic
// assumes (scan_registration.cpp:183-298); KITTI-style ring-major order is
// available as a robustness variant.
#include <math.h>
#include <stdint.h>
#include <string.h>
#include <algorithm>
#include <vector>

namespace {

struct Rng {  // splitmix64 / xorshift; deterministic across platforms
  uint64_t s;
  explicit Rng(uint64_t seed) : s(seed * 0x9E3779B97F4A7C15ull + 0x1234567ull) { next(); next(); }
  uint64_t next() { uint64_t z = (s += 0x9E3779B97F4A7C15ull); z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull; z = (z ^ (z >> 27)) * 0x94D049BB133111EBull; return z ^ (z >> 31); }
  double uni() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }
  double uni(double a, double b) { return a + (b - a) * uni(); }
  double gauss() { double u = uni(), v = uni(); if (u < 1e-300) u = 1e-300; return sqrt(-2.0 * log(u)) * cos(6.283185307179586 * v); }
};

struct Box { double x0, y0, x1, y1, h; };
struct Pole { double cx, cy, r, h; };

struct World {
  double zg;  // ground height in the world frame (sensor starts at z = 0)
  std::vector<Box> boxes;
  std::vector<Pole> poles;
  // acceleration grid
  double gx0, gy0, cell; int gw, gh;
  std::vector<std::vector<int>> cells;  // prim id: >=0 box, <0 => pole ~id
  void build_grid() {
    double x0 = 1e30, y0 = 1e30, x1 = -1e30, y1 = -1e30;
    for (auto& b : boxes) { x0 = std::min(x0, b.x0); y0 = std::min(y0, b.y0); x1 = std::max(x1, b.x1); y1 = std::max(y1, b.y1); }
    for (auto& p : poles) { x0 = std::min(x0, p.cx - p.r); y0 = std::min(y0, p.cy - p.r); x1 = std::max(x1, p.cx + p.r); y1 = std::max(y1, p.cy + p.r); }
    if (x0 > x1) { x0 = y0 = 0; x1 = y1 = 1; }
    cell = 10.0; gx0 = x0 - 1; gy0 = y0 - 1;
    gw = (int)((x1 + 1 - gx0) / cell) + 1; gh = (int)((y1 + 1 - gy0) / cell) + 1;
    cells.assign((size_t)gw * gh, {});
    auto add = [&](double ax0, double ay0, double ax1, double ay1, int id) {
      int i0 = (int)((ax0 - gx0) / cell), i1 = (int)((ax1 - gx0) / cell), j0 = (int)((ay0 - gy0) / cell), j1 = (int)((ay1 - gy0) / cell);
      for (int j = j0; j <= j1; ++j) for (int i = i0; i <= i1; ++i) cells[(size_t)j * gw + i].push_back(id);
    };
    for (int k = 0; k < (int)boxes.size(); ++k) add(boxes[k].x0, boxes[k].y0, boxes[k].x1, boxes[k].y1, k);
    for (int k = 0; k < (int)poles.size(); ++k) add(poles[k].cx - poles[k].r, poles[k].cy - poles[k].r, poles[k].cx + poles[k].r, poles[k].cy + poles[k].r, ~k);
  }
  double hit_prim(int id, const double o[3], const double d[3]) const {
    if (id >= 0) {
      const Box& b = boxes[id];
      double t0 = 0, t1 = 1e30;
      const double lo[3] = {b.x0, b.y0, zg}, hi[3] = {b.x1, b.y1, zg + b.h};
      for (int a = 0; a < 3; ++a) {
        if (fabs(d[a]) < 1e-12) { if (o[a] < lo[a] || o[a] > hi[a]) return 1e30; continue; }
        double ta = (lo[a] - o[a]) / d[a], tb = (hi[a] - o[a]) / d[a];
        if (ta > tb) std::swap(ta, tb);
        t0 = std::max(t0, ta); t1 = std::min(t1, tb);
        if (t0 > t1) return 1e30;
      }
      return t0 > 1e-6 ? t0 : 1e30;
    }
    const Pole& p = poles[~id];
    const double ox = o[0] - p.cx, oy = o[1] - p.cy;
    const double A = d[0] * d[0] + d[1] * d[1];
    if (A < 1e-12) return 1e30;
    const double B = ox * d[0] + oy * d[1], C = ox * ox + oy * oy - p.r * p.r;
    const double disc = B * B - A * C;
    if (disc < 0) return 1e30;
    const double t = (-B - sqrt(disc)) / A;
    if (t < 1e-6) return 1e30;
    const double z = o[2] + t * d[2];
    return (z >= zg && z <= zg + p.h) ? t : 1e30;
  }
  double cast(const double o[3], const double d[3], double maxr) const {
    double best = 1e30;
    if (d[2] < -1e-9) { const double t = (zg - o[2]) / d[2]; if (t > 0) best = t; }
    // 2-D DDA
    const double dl = sqrt(d[0] * d[0] + d[1] * d[1]);
    if (dl > 1e-9 && !cells.empty()) {
      double t = 0;
      double px = o[0], py = o[1];
      int i = (int)floor((px - gx0) / cell), j = (int)floor((py - gy0) / cell);
      const int si = d[0] > 0 ? 1 : -1, sj = d[1] > 0 ? 1 : -1;
      double tmx = fabs(d[0]) > 1e-12 ? ((gx0 + (i + (si > 0)) * cell) - px) / d[0] : 1e30;
      double tmy = fabs(d[1]) > 1e-12 ? ((gy0 + (j + (sj > 0)) * cell) - py) / d[1] : 1e30;
      const double tdx = fabs(d[0]) > 1e-12 ? cell / fabs(d[0]) : 1e30, tdy = fabs(d[1]) > 1e-12 ? cell / fabs(d[1]) : 1e30;
      const double tend = std::min(maxr, best);
      while (t <= tend) {
        if (i >= 0 && i < gw && j >= 0 && j < gh)
          for (int id : cells[(size_t)j * gw + i]) { const double h = hit_prim(id, o, d); if (h < best) best = h; }
        const double tnext = std::min(tmx, tmy);
        if (best <= tnext) break;
        if (tmx < tmy) { i += si; t = tmx; tmx += tdx; } else { j += sj; t = tmy; tmy += tdy; }
        if ((si > 0 && i >= gw) || (si < 0 && i < 0) || (sj > 0 && j >= gh) || (sj < 0 && j < 0)) break;
      }
    }
    return best <= maxr ? best : 1e30;
  }
};

void euler_to_R(double yaw, double pitch, double roll, double R[9]) {
  const double cy = cos(yaw), sy = sin(yaw), cp = cos(pitch), sp = sin(pitch), cr = cos(roll), sr = sin(roll);
  R[0] = cy * cp; R[1] = cy * sp * sr - sy * cr; R[2] = cy * sp * cr + sy * sr;
  R[3] = sy * cp; R[4] = sy * sp * sr + cy * cr; R[5] = sy * sp * cr - cy * sr;
  R[6] = -sp;     R[7] = cp * sr;                R[8] = cp * cr;
}

// ZYX Euler angles -> quaternion {x, y, z, w} of R = Rz(yaw) Ry(pitch) Rx(roll) (the rotation euler_to_R builds)
void euler_to_q(double yaw, double pitch, double roll, double q[4]) {
  const double cy = cos(yaw * 0.5), sy = sin(yaw * 0.5), cp = cos(pitch * 0.5), sp = sin(pitch * 0.5), cr = cos(roll * 0.5), sr = sin(roll * 0.5);
  q[0] = sr * cp * cy - cr * sp * sy; q[1] = cr * sp * cy + sr * cp * sy; q[2] = cr * cp * sy - sr * sp * cy; q[3] = cr * cp * cy + sr * sp * sy;
}
void q_to_R(const double q[4], double R[9]) {
  const double x = q[0], y = q[1], z = q[2], w = q[3];
  R[0] = 1 - 2 * (y * y + z * z); R[1] = 2 * (x * y - z * w);     R[2] = 2 * (x * z + y * w);
  R[3] = 2 * (x * y + z * w);     R[4] = 1 - 2 * (x * x + z * z); R[5] = 2 * (y * z - x * w);
  R[6] = 2 * (x * z - y * w);     R[7] = 2 * (y * z + x * w);     R[8] = 1 - 2 * (x * x + y * y);
}
// sensor pose at sweep fraction f in [0, 1] between pose0 and pose1: translation linear, rotation slerp (shortest arc)
void interp_pose(const double* p0, const double* p1, double f, double o[3], double R[9]) {
  for (int a = 0; a < 3; ++a) o[a] = p0[a] + f * (p1[a] - p0[a]);
  double q0[4], q1[4];
  euler_to_q(p0[3], p0[4], p0[5], q0); euler_to_q(p1[3], p1[4], p1[5], q1);
  double d = q0[0] * q1[0] + q0[1] * q1[1] + q0[2] * q1[2] + q0[3] * q1[3];
  if (d < 0) { d = -d; for (int k = 0; k < 4; ++k) q1[k] = -q1[k]; }
  double s0 = 1 - f, s1 = f;
  if (d < 1 - 1e-12) { const double th = acos(d), st = sin(th); s0 = sin((1 - f) * th) / st; s1 = sin(f * th) / st; }
  double q[4], n = 0;
  for (int k = 0; k < 4; ++k) { q[k] = s0 * q0[k] + s1 * q1[k]; n += q[k] * q[k]; }
  n = sqrt(n);
  for (int k = 0; k < 4; ++k) q[k] /= n;
  q_to_R(q, R);
}

int beam_table(int sensor, std::vector<double>& elev, int* n_az) {
  elev.clear();
  if (sensor == 0) { for (int i = 0; i < 16; ++i) elev.push_back(-15.0 + 2.0 * i); *n_az = 1800; }
  else if (sensor == 1) {  // HDL-64E: scan_registration.cpp:243-249
    for (int i = 0; i < 32; ++i) elev.push_back(2.0 - i / 3.0);
    for (int i = 0; i < 32; ++i) elev.push_back(-8.83 - i / 2.0);
    *n_az = 1875;
  } else if (sensor == 2) { for (int i = 0; i < 128; ++i) elev.push_back(-22.5 + 45.0 * i / 127.0); *n_az = 2048; }
  else if (sensor == 3) { for (int i = 0; i < 32; ++i) elev.push_back(-92.0 / 3.0 + (i + 0.5) * 4.0 / 3.0); *n_az = 1800; }
  else return -1;
  return (int)elev.size();
}

}  // namespace

extern "C" {

// kind 0: open street (few buildings, poles); kind 1: dense city of towers sized so a
// 250 x 250 m window holds ~1M map points at 0.4 / 0.8 m leaves (config C3), kind 2: ~2M (C4).
void* vloam_synth_world_create(uint64_t seed, int kind, double extent) {
  World* w = new World();
  Rng r(seed);
  w->zg = -1.8;
  const double pitch = kind == 0 ? 40.0 : 12.5;
  const double foot = kind == 0 ? 20.0 : 8.5;
  const double hmin = kind == 0 ? 6.0 : (kind == 1 ? 24.0 : 64.0), hmax = kind == 0 ? 20.0 : (kind == 1 ? 72.0 : 120.0);
  const double street_half = kind == 0 ? 8.0 : 3.0;
  for (double bx = -extent; bx < extent; bx += pitch)
    for (double by = -extent; by < extent; by += pitch) {
      const double x0 = bx + (pitch - foot) * 0.5 + r.uni(-0.8, 0.8), y0 = by + (pitch - foot) * 0.5 + r.uni(-0.8, 0.8);
      const double fx = foot * r.uni(0.85, 1.0), fy = foot * r.uni(0.85, 1.0);
      // keep the driving corridor (along +x through the origin) free
      if (y0 < street_half && y0 + fy > -street_half) continue;
      w->boxes.push_back(Box{x0, y0, x0 + fx, y0 + fy, r.uni(hmin, hmax)});
    }
  const int npoles = (int)(extent * (kind == 0 ? 0.6 : 0.8));
  for (int k = 0; k < npoles; ++k) {
    const double cx = r.uni(-extent, extent), side = r.uni() < 0.5 ? -1.0 : 1.0;
    w->poles.push_back(Pole{cx, side * r.uni(street_half * 0.6, street_half * 0.95), r.uni(0.1, 0.3), r.uni(4.0, 9.0)});
  }
  w->build_grid();
  return w;
}
void vloam_synth_world_destroy(void* w) { delete (World*)w; }

// One sweep; pose1 == nullptr: from the fixed pose {x,y,z,yaw,pitch,roll} (world frame), otherwise azimuth column ia is cast
// from the pose interpolated between pose0 and pose1 at its emission fraction ia / n_az.
static int scan_impl(void* wv, int sensor, const double* pose, const double* pose1, uint64_t seed, double range_sigma, double nan_frac,
                     double max_range, int order, double az0, float* out, int cap) {
  const World* w = (const World*)wv;
  std::vector<double> elev; int n_az;
  const int nb = beam_table(sensor, elev, &n_az);
  if (nb < 0) return -1;
  double R[9]; euler_to_R(pose[3], pose[4], pose[5], R);
  double o[3] = {pose[0], pose[1], pose[2]};
  // per-column poses of a moving sensor (the columns follow the rotation sense ori = -atan2(y, x) of the emission loop below,
  // the sense ScanRegistration's relTime assumes, SR.cpp:183-298)
  std::vector<double> colO, colR;
  if (pose1) {
    colO.resize((size_t)n_az * 3); colR.resize((size_t)n_az * 9);
    for (int ia = 0; ia < n_az; ++ia) interp_pose(pose, pose1, (double)ia / n_az, &colO[(size_t)ia * 3], &colR[(size_t)ia * 9]);
  }
  Rng rng(seed);
  int n = 0;
  const int outer = order == 0 ? n_az : nb, inner = order == 0 ? nb : n_az;
  for (int a = 0; a < outer; ++a)
    for (int b = 0; b < inner; ++b) {
      const int ia = order == 0 ? a : b, ib = order == 0 ? b : a;
      // clockwise rotation: ori = -atan2(y, x) increases through the sweep
      const double az = -(az0 + 6.283185307179586 * ia / n_az);
      const double el = (elev[ib] + 0.03 * rng.gauss()) * 0.017453292519943295;
      const double ds[3] = {cos(el) * cos(az), cos(el) * sin(az), sin(el)};
      if (pose1) { memcpy(o, &colO[(size_t)ia * 3], sizeof o); memcpy(R, &colR[(size_t)ia * 9], sizeof R); }
      const double d[3] = {R[0] * ds[0] + R[1] * ds[1] + R[2] * ds[2], R[3] * ds[0] + R[4] * ds[1] + R[5] * ds[2],
                           R[6] * ds[0] + R[7] * ds[1] + R[8] * ds[2]};
      const double u_nan = rng.uni(), noise = rng.gauss();
      const double t = w->cast(o, d, max_range);
      if (t > max_range) continue;
      if (n >= cap) return n;
      float* p = out + (size_t)n * 4;
      if (u_nan < nan_frac) { p[0] = p[1] = p[2] = NAN; p[3] = 0; ++n; continue; }
      const double rr = t + range_sigma * noise;
      p[0] = (float)(rr * ds[0]); p[1] = (float)(rr * ds[1]); p[2] = (float)(rr * ds[2]); p[3] = 0.f;
      ++n;
    }
  return n;
}

// One sweep from pose {x,y,z,yaw,pitch,roll} (world frame).  Writes float32[n][4]
// (x,y,z,0) in the SENSOR frame; returns n.  order: 0 azimuth-major, 1 ring-major.
// nan_frac of returns become NaN; returns past max_range are dropped.
int vloam_synth_scan(void* wv, int sensor, const double* pose, uint64_t seed, double range_sigma, double nan_frac,
                     double max_range, int order, double az0, float* out, int cap) {
  return scan_impl(wv, sensor, pose, nullptr, seed, range_sigma, nan_frac, max_range, order, az0, out, cap);
}
// The same sweep from a MOVING sensor: azimuth column ia is cast from the pose at fraction ia / n_az between pose_start and
// pose_end (translation linear, rotation slerp) and its points are written in the sensor frame of that instant -- a sweep that
// is not motion-compensated.  With the only difference to vloam_synth_scan being those per-column poses, pose_start == pose_end
// gives exactly vloam_synth_scan(pose_start) (the fixed-pose path is taken then).
int vloam_synth_scan_moving(void* wv, int sensor, const double* pose_start, const double* pose_end, uint64_t seed, double range_sigma,
                            double nan_frac, double max_range, int order, double az0, float* out, int cap) {
  const bool still = memcmp(pose_start, pose_end, 6 * sizeof(double)) == 0;
  return scan_impl(wv, sensor, pose_start, still ? nullptr : pose_end, seed, range_sigma, nan_frac, max_range, order, az0, out, cap);
}

// Plant map points on the world's surfaces inside [cx-hw,cx+hw] x [cy-hw,cy+hw] x [zlo,zhi]:
// surf points one per `leaf_s` voxel on ground / walls / roofs, corner points one per
// `leaf_c` voxel on vertical box edges, roof edges and poles.  kind_out: 0 corner, 1 surf.
// Returns the number of points written (float32[n][4], intensity 0); duplicates per
// voxel are removed by the caller (python) with the filter's own float arithmetic.
int vloam_synth_plant(void* wv, uint64_t seed, int kind_out, double leaf, double cx, double cy, double hw, double zlo,
                      double zhi, float* out, int cap) {
  const World* w = (const World*)wv;
  Rng r(seed);
  int n = 0;
  auto emit = [&](double x, double y, double z) {
    if (x < cx - hw || x > cx + hw || y < cy - hw || y > cy + hw || z < zlo || z > zhi) return;
    if (n >= cap) return;
    float* p = out + (size_t)n * 4;
    p[0] = (float)(x + 0.01 * r.gauss()); p[1] = (float)(y + 0.01 * r.gauss()); p[2] = (float)(z + 0.01 * r.gauss()); p[3] = 0.f;
    ++n;
  };
  auto inside_box = [&](double x, double y) { for (auto& b : w->boxes) if (x > b.x0 && x < b.x1 && y > b.y0 && y < b.y1) return true; return false; };
  if (kind_out == 1) {
    for (double x = cx - hw; x < cx + hw; x += leaf)
      for (double y = cy - hw; y < cy + hw; y += leaf) {
        const double px = x + leaf * r.uni(0.15, 0.85), py = y + leaf * r.uni(0.15, 0.85);
        if (!inside_box(px, py)) emit(px, py, w->zg);
      }
    for (auto& b : w->boxes) {
      for (double z = w->zg + 0.1; z < w->zg + b.h; z += leaf) {
        for (double x = b.x0; x < b.x1; x += leaf) { emit(x + leaf * r.uni(0.15, 0.85), b.y0, z + leaf * r.uni(0.1, 0.8)); emit(x + leaf * r.uni(0.15, 0.85), b.y1, z + leaf * r.uni(0.1, 0.8)); }
        for (double y = b.y0; y < b.y1; y += leaf) { emit(b.x0, y + leaf * r.uni(0.15, 0.85), z + leaf * r.uni(0.1, 0.8)); emit(b.x1, y + leaf * r.uni(0.15, 0.85), z + leaf * r.uni(0.1, 0.8)); }
      }
    }
  } else {
    for (auto& b : w->boxes) {
      const double ex[4] = {b.x0, b.x1, b.x0, b.x1}, ey[4] = {b.y0, b.y0, b.y1, b.y1};
      for (int e = 0; e < 4; ++e)
        for (double z = w->zg + 0.2; z < w->zg + b.h; z += leaf) emit(ex[e], ey[e], z + leaf * r.uni(0.1, 0.8));
    }
    for (auto& p : w->poles)
      for (double z = w->zg + 0.2; z < w->zg + p.h; z += leaf) emit(p.cx, p.cy, z + leaf * r.uni(0.1, 0.8));
  }
  return n;
}

int vloam_synth_counts(void* wv, int* nboxes, int* npoles) {
  const World* w = (const World*)wv; *nboxes = (int)w->boxes.size(); *npoles = (int)w->poles.size(); return 0;
}

}  // extern "C"
