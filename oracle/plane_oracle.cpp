// plane_oracle.cpp — CPU restatement of the plane ground model (cp_set_ground_plane, contract in include/conesgpu.h).
// TEST INFRASTRUCTURE ONLY.  PARITY UNPINNED: the reference's ground node is the sector model and has nothing to
// compare a plane with; this file states the contract operation by operation, and the GPU kernels
// (cones_perception_b200/csrc/plane_kernels.cuh) are held to it bit for bit.  Built with -ffp-contract=off: every
// double operation of the plane is rounded on its own, and the fp32 distance is three explicit fmaf.
// Points are PCL PointXYZI records (8 floats: x y z 1 intensity 0 0 0), as orc_from_msg produces them.
#include <math.h>
#include <stdint.h>
#include <string.h>

namespace {

struct Pt {
  float x, y, z, pad, intensity, c1, c2, c3;
};

uint64_t splitmix64(uint64_t x) {
  uint64_t z = x + 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

bool finite3(const Pt& p) { return isfinite(p.x) && isfinite(p.y) && isfinite(p.z); }

// false: invalid hypothesis
bool plane_from(const Pt& a, const Pt& b, const Pt& c, double cos_tilt, float out[4]) {
  if (!finite3(a) || !finite3(b) || !finite3(c)) return false;
  const double x0 = a.x, y0 = a.y, z0 = a.z;
  const double ux = (double)b.x - x0, uy = (double)b.y - y0, uz = (double)b.z - z0;
  const double vx = (double)c.x - x0, vy = (double)c.y - y0, vz = (double)c.z - z0;
  double nx = uy * vz - uz * vy;
  double ny = uz * vx - ux * vz;
  double nz = ux * vy - uy * vx;
  const double L = sqrt(nx * nx + ny * ny + nz * nz);
  if (!(L > 0.0) || !isfinite(L)) return false;
  if (nz < 0.0) {
    nx = -nx;
    ny = -ny;
    nz = -nz;
  }
  if (nz / L < cos_tilt) return false;
  nx /= L;
  ny /= L;
  nz /= L;
  const double d = -(nx * x0 + ny * y0 + nz * z0);
  out[0] = (float)nx;
  out[1] = (float)ny;
  out[2] = (float)nz;
  out[3] = (float)d;
  return true;
}

float distance(const float* pl, const Pt& p) { return fmaf(pl[2], p.z, fmaf(pl[1], p.y, fmaf(pl[0], p.x, pl[3]))); }

}  // namespace

extern "C" {

uint32_t orc_plane_index(uint64_t seed, uint32_t h, uint32_t j, uint32_t n) {
  return (uint32_t)(((splitmix64(seed + 3ull * h + j) >> 32) * (uint64_t)n) >> 32);
}

double orc_plane_cos_tilt(float max_tilt_deg) { return cos((double)max_tilt_deg * (M_PI / 180.0)); }

// planes[H][4]: a, b, c, d of every hypothesis, NaN when invalid (every hypothesis of a frame with n < 3)
void orc_plane_hypotheses(const void* pts, uint32_t n, uint64_t seed, uint32_t H, float max_tilt_deg, float* planes) {
  const Pt* P = static_cast<const Pt*>(pts);
  const double ct = orc_plane_cos_tilt(max_tilt_deg);
  for (uint32_t h = 0; h < H; ++h) {
    float* o = planes + 4 * h;
    if (n < 3 || !plane_from(P[orc_plane_index(seed, h, 0, n)], P[orc_plane_index(seed, h, 1, n)],
                             P[orc_plane_index(seed, h, 2, n)], ct, o))
      o[0] = o[1] = o[2] = o[3] = NAN;
  }
}

// counts[H]: finite points with |s| <= inlier_distance
void orc_plane_counts(const void* pts, uint32_t n, const float* planes, uint32_t H, float inlier_distance,
                      uint32_t* counts) {
  const Pt* P = static_cast<const Pt*>(pts);
  for (uint32_t h = 0; h < H; ++h) {
    uint32_t c = 0;
    for (uint32_t i = 0; i < n; ++i)
      if (finite3(P[i]) && fabsf(distance(planes + 4 * h, P[i])) <= inlier_distance) ++c;
    counts[h] = c;
  }
}

// The ground node under the plane model: out[n] the message (survivors in input order, then n - kept PCL padding
// points), the chosen plane (NaN: none), its inliers and hypothesis (-1: none), keep[n] the verdict.
void orc_plane_ground_node(const void* pts, uint32_t n, uint64_t seed, uint32_t H, float inlier_distance,
                           float ground_height, float max_tilt_deg, void* out, uint32_t* kept, float* plane,
                           uint32_t* inliers, int32_t* hypothesis, uint8_t* keep) {
  const Pt* P = static_cast<const Pt*>(pts);
  float* planes = new float[4 * (size_t)H];
  uint32_t* counts = new uint32_t[H];
  orc_plane_hypotheses(pts, n, seed, H, max_tilt_deg, planes);
  orc_plane_counts(pts, n, planes, H, inlier_distance, counts);
  int32_t best = -1;
  for (uint32_t h = 0; h < H; ++h)
    if (!isnan(planes[4 * h]) && (best < 0 || counts[h] > counts[best])) best = (int32_t)h;
  const float nan4[4] = {NAN, NAN, NAN, NAN};
  const float* pl = best >= 0 ? planes + 4 * best : nan4;
  memcpy(plane, pl, sizeof(float) * 4);
  *inliers = best >= 0 ? counts[best] : 0u;
  *hypothesis = best;
  Pt* O = static_cast<Pt*>(out);
  uint32_t g = 0;
  for (uint32_t i = 0; i < n; ++i) {
    const bool k = finite3(P[i]) && (best < 0 || distance(pl, P[i]) >= ground_height);
    keep[i] = k ? 1 : 0;
    if (k) {
      Pt q;
      memset(&q, 0, sizeof(q));
      q.x = P[i].x;
      q.y = P[i].y;
      q.z = P[i].z;
      q.pad = 1.0f;
      q.intensity = P[i].intensity;
      O[g++] = q;
    }
  }
  for (uint32_t i = g; i < n; ++i) {
    Pt q;
    memset(&q, 0, sizeof(q));
    q.pad = 1.0f;
    O[i] = q;
  }
  *kept = g;
  delete[] planes;
  delete[] counts;
}

}  // extern "C"
