// core_math.cuh — the arithmetic of the path, written __host__ __device__ so that the exact
// same code can be exercised on the CPU by tests/host_check (logic check only; the product
// runs these functions inside CUDA kernels and nowhere else).
//
// Everything here that must agree with PCL bit-for-bit keeps PCL's operation order in plain
// float expressions; the library is built with -fmad=false, so nothing is contracted.
#pragma once

#include <cfloat>
#include <cmath>

#include "common.cuh"

namespace peb {

// ---- 4x4 column-major float matrices (Eigen::Matrix4f storage) -----------------------------
struct Mat4 {
  float m[16];
};

PEB_HD Mat4 mat4_identity() {
  Mat4 a;
#pragma unroll
  for (int i = 0; i < 16; ++i) a.m[i] = (i % 5 == 0) ? 1.0f : 0.0f;
  return a;
}

// [EIGEN] Matrix4f product: result(i,j) = ((a(i,0)b(0,j) + a(i,1)b(1,j)) + a(i,2)b(2,j)) + a(i,3)b(3,j)
// (final_transformation_ = transformation_ * final_transformation_, [PCL] registration/impl/icp.hpp)
PEB_HD Mat4 mat4_mul(const Mat4& a, const Mat4& b) {
  Mat4 r;
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float acc = a.m[0 * 4 + i] * b.m[j * 4 + 0];
      acc = acc + a.m[1 * 4 + i] * b.m[j * 4 + 1];
      acc = acc + a.m[2 * 4 + i] * b.m[j * 4 + 2];
      acc = acc + a.m[3 * 4 + i] * b.m[j * 4 + 3];
      r.m[j * 4 + i] = acc;
    }
  return r;
}

// [PCL] registration/impl/icp.hpp : transformCloud — pt_t = tr * (x,y,z,1), Eigen order
PEB_HD void transform_icp(const float* __restrict__ t, float x, float y, float z, float& ox, float& oy, float& oz) {
  ox = ((t[0] * x + t[4] * y) + t[8] * z) + t[12] * 1.0f;
  oy = ((t[1] * x + t[5] * y) + t[9] * z) + t[13] * 1.0f;
  oz = ((t[2] * x + t[6] * y) + t[10] * z) + t[14] * 1.0f;
}

// [PCL] common/impl/transforms.hpp : detail::Transformer<float>::se3 — c0*x + (c1*y + (c2*z + c3))
PEB_HD void transform_tpc(const float* __restrict__ t, float x, float y, float z, float& ox, float& oy, float& oz) {
  ox = x * t[0] + (y * t[4] + (z * t[8] + t[12]));
  oy = x * t[1] + (y * t[5] + (z * t[9] + t[13]));
  oz = x * t[2] + (y * t[6] + (z * t[10] + t[14]));
}

// [FLANN] algorithms/dist.h : L2_Simple<float> — ((0 + dx*dx) + dy*dy) + dz*dz
PEB_HD float l2_simple(float qx, float qy, float qz, float px, float py, float pz) {
  float dx = qx - px, dy = qy - py, dz = qz - pz;
  float r = dx * dx;
  r = r + dy * dy;
  r = r + dz * dz;
  return r;
}

PEB_HD bool finite3(float x, float y, float z) {
  // (v - v) is 0 for finite v and NaN for inf / NaN
  return (x - x) == 0.0f && (y - y) == 0.0f && (z - z) == 0.0f;
}

// ---- uniform-grid exact nearest neighbour ---------------------------------------------------
struct NnBest {
  float d2;
  int idx;  // original target index
  int j;    // position in the sorted array (for the normal / point gather)
};

PEB_HD void nn_consider(NnBest& b, float d2, int idx, int j) {
  if (d2 < b.d2 || (d2 == b.d2 && idx < b.idx)) {
    b.d2 = d2;
    b.idx = idx;
    b.j = j;
  }
}

PEB_HD int grid_coord(float q, float origin, float inv_h, int dim) {
  float v = floorf((q - origin) * inv_h);
  v = fminf(fmaxf(v, 0.0f), static_cast<float>(dim - 1));
  return static_cast<int>(v);
}

PEB_HD void grid_scan_range(const GridView& g, uint32_t s, uint32_t e, float qx, float qy, float qz, NnBest& best) {
  for (uint32_t j = s; j < e; ++j) {
    float4 p = g.pts[j];
    float d2 = l2_simple(qx, qy, qz, p.x, p.y, p.z);
#ifdef __CUDA_ARCH__
    nn_consider(best, d2, __float_as_int(p.w), static_cast<int>(j));
#else
    int id;
    memcpy(&id, &p.w, 4);
    nn_consider(best, d2, id, static_cast<int>(j));
#endif
  }
}

// Scans the rows of ring r around cell (cx,cy,cz) that belong to `lane` of a group of G lanes.
// full = true: every row of the (2r+1)^2 block is scanned over its whole x extent (first pass);
// full = false: only the shell — outer rows over the whole x extent, inner rows at their two
// end cells x = cx-r and x = cx+r.
PEB_HD void grid_scan_ring(const GridView& g, float qx, float qy, float qz, int cx, int cy, int cz, int r, bool full,
                           int lane, int G, NnBest& best) {
  const int w = 2 * r + 1;
  const int x0 = max(cx - r, 0), x1 = min(cx + r, g.dx - 1);
  for (int row = lane; row < w * w; row += G) {
    const int oy = row % w - r, oz = row / w - r;
    const int y = cy + oy, z = cz + oz;
    if (y < 0 || y >= g.dy || z < 0 || z >= g.dz) continue;
    const long long base = (static_cast<long long>(z) * g.dy + y) * g.dx;
    const bool outer = full || oy == -r || oy == r || oz == -r || oz == r;
    if (outer) {
      grid_scan_range(g, g.cell_start[base + x0], g.cell_start[base + x1 + 1], qx, qy, qz, best);
    } else {
      if (cx - r >= 0) grid_scan_range(g, g.cell_start[base + cx - r], g.cell_start[base + cx - r + 1], qx, qy, qz, best);
      if (cx + r < g.dx) grid_scan_range(g, g.cell_start[base + cx + r], g.cell_start[base + cx + r + 1], qx, qy, qz, best);
    }
  }
}

// Lower bound (squared) on the distance from q to any grid point OUTSIDE the searched block
// [c-r, c+r]^3 (clamped to the grid).  A point outside the block lies beyond at least one block
// face that still has grid on its far side; for such a face on axis a the distance is at least
// sqrt(gap_a^2 + sum_{b != a} out_b^2), out_b being q's distance to the grid box along b
// (non-zero only for queries outside the box).  The gap is shrunk by 1 % of a cell so that float
// rounding in cell assignment and in the distance sums can never make the test optimistic.
// covers_all: no face has grid beyond it, i.e. every point has been examined.
PEB_HD float grid_ring_bound2(const GridView& g, float qx, float qy, float qz, int cx, int cy, int cz, int r,
                              bool& covers_all) {
  const float q[3] = {qx, qy, qz};
  const float o[3] = {g.ox, g.oy, g.oz};
  const int c[3] = {cx, cy, cz};
  const int d[3] = {g.dx, g.dy, g.dz};
  float out2[3];
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    float lo = o[a], hi = o[a] + static_cast<float>(d[a]) * g.h;
    float od = fmaxf(fmaxf(lo - q[a], q[a] - hi), 0.0f);
    od = fmaxf(od - 0.01f * g.h, 0.0f);
    out2[a] = od * od;
  }
  const float margin = 0.01f * g.h;
  float best = FLT_MAX;
  covers_all = true;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    const float others = out2[(a + 1) % 3] + out2[(a + 2) % 3];
    const int lo = c[a] - r, hi = c[a] + r;
    if (lo > 0) {
      covers_all = false;
      float gap = fmaxf(q[a] - (o[a] + static_cast<float>(lo) * g.h) - margin, 0.0f);
      best = fminf(best, gap * gap + others);
    }
    if (hi < d[a] - 1) {
      covers_all = false;
      float gap = fmaxf((o[a] + static_cast<float>(hi + 1) * g.h) - q[a] - margin, 0.0f);
      best = fminf(best, gap * gap + others);
    }
  }
  return best;
}

// Distance (>= 0) from coordinate q to the slab of cell index c along one axis, shrunk by the
// same 1 % safety margin as grid_ring_bound2 (cell membership is decided in float arithmetic).
PEB_HD float grid_slab_dist(float q, float origin, float h, int c) {
  const float lo = origin + static_cast<float>(c) * h;
  const float hi = origin + static_cast<float>(c + 1) * h;
  return fmaxf(fmaxf(lo - q, q - hi) - 0.01f * h, 0.0f);
}

PEB_HD int point_index(const float4& p) {
#ifdef __CUDA_ARCH__
  return __float_as_int(p.w);
#else
  int id;
  memcpy(&id, &p.w, 4);
  return id;
#endif
}

// ---- ball search: everything closer than the current best ---------------------------------------
// `best` holds a candidate; any point that beats it lies inside the ball of radius sqrt(best.d2)
// (capped by limit_d2: matches farther than that are rejected by the caller anyway), so only the
// cells intersecting that ball are examined.  Rows (fixed y, z) whose slab is farther than the
// current best are skipped and every row is cut to the chord of the ball; both shrink as better
// points are found.  All slab / chord tests carry the same conservative margins as the ring
// search, so the result is exact for any starting candidate.

// (A 4 x 4 x 4 occupancy bitmap that lets a large ball skip its empty bulk was built and measured:
//  no gain on C2 / C4 — the slab test already rejects empty rows at ~10 instructions each — so the
//  rows of the ball's bounding box are walked directly.)
//
// The walk runs in CELL units: f = (q - origin) / h once per search, then a row costs a subtraction
// where the world-unit form cost two multiply-adds per slab and per chord end (-11 of ~46 instructions
// per row).  f is computed with the expression that assigned the target points to their cells
// (grid_coord), so both sides carry the same rounding, at most a few ulps of the largest cell
// coordinate: `pad` covers it at the chord ends and the 1 % shrink of the slab distances in the row test.

// distance (>= 0, in cells) from cell coordinate f to the slab of cell index c, shrunk by 1 % of a cell
PEB_HD float grid_slab_dist_cells(float f, int c) {
  const float t = f - static_cast<float>(c);
  return fmaxf(fmaxf(-t, t - 1.0f) - 0.01f, 0.0f);
}

PEB_HD int grid_clamp_cell(float v, int dim) {
  v = fminf(fmaxf(floorf(v), 0.0f), static_cast<float>(dim - 1));
  return static_cast<int>(v);
}

PEB_HD void grid_ball_search(const GridView& g, float qx, float qy, float qz, float limit_d2, NnBest& best) {
  const float fx = (qx - g.ox) * g.inv_h, fy = (qy - g.oy) * g.inv_h, fz = (qz - g.oz) * g.inv_h;
  const float inv_h2 = g.inv_h * g.inv_h;
  // 0.001 cell >> the rounding of a cell coordinate (4 ulps of the largest one are added for very large grids)
  const float pad = 0.001f + 4.8e-7f * static_cast<float>(max(g.dx, max(g.dy, g.dz)));
  const float R = sqrtf(fminf(best.d2, limit_d2) * inv_h2) * 1.0001f + pad;
  const int y0 = grid_clamp_cell(fy - R, g.dy), y1 = grid_clamp_cell(fy + R, g.dy);
  const int z0 = grid_clamp_cell(fz - R, g.dz), z1 = grid_clamp_cell(fz + R, g.dz);
  for (int z = z0; z <= z1; ++z) {
    const float dz = grid_slab_dist_cells(fz, z);
    for (int y = y0; y <= y1; ++y) {
      const float dy = grid_slab_dist_cells(fy, y);
      const float dyz2 = dy * dy + dz * dz;
      const float cur = fminf(best.d2, limit_d2) * inv_h2;  // (cells^2; shrinks as better points are found)
      if (dyz2 > cur) continue;
      const float rx = sqrtf(cur - dyz2) * 1.0001f + pad;
      const int x0 = grid_clamp_cell(fx - rx, g.dx), x1 = grid_clamp_cell(fx + rx, g.dx);
      const int base = (z * g.dy + y) * g.dx;
      grid_scan_range(g, g.cell_start[base + x0], g.cell_start[base + x1 + 1], qx, qy, qz, best);
    }
  }
}

// Grid rows (fixed y, z) in the bounding box of the ball grid_ball_search would walk for a candidate at squared
// distance d2: the walk's trip count, known before any cell is looked at.  Scheduling only (icp.cu bins the queries of
// a block by it so that the lanes of a warp walk equally many rows); it never decides a result.
PEB_HD int grid_ball_rows(const GridView& g, float qy, float qz, float d2, float limit_d2) {
  const float fy = (qy - g.oy) * g.inv_h, fz = (qz - g.oz) * g.inv_h;
  const float pad = 0.001f + 4.8e-7f * static_cast<float>(max(g.dx, max(g.dy, g.dz)));
  const float R = sqrtf(fminf(d2, limit_d2) * (g.inv_h * g.inv_h)) * 1.0001f + pad;
  const int y0 = grid_clamp_cell(fy - R, g.dy), y1 = grid_clamp_cell(fy + R, g.dy);
  const int z0 = grid_clamp_cell(fz - R, g.dz), z1 = grid_clamp_cell(fz + R, g.dz);
  return (y1 - y0 + 1) * (z1 - z0 + 1);
}

// Exact 1-NN given one candidate (sorted position j_prev, e.g. last iteration's match)
PEB_HD NnBest grid_nn_warm(const GridView& g, float qx, float qy, float qz, int j_prev, float limit_d2) {
  NnBest best;
  const float4 p = g.pts[j_prev];
  best.d2 = l2_simple(qx, qy, qz, p.x, p.y, p.z);
  best.idx = point_index(p);
  best.j = j_prev;
  grid_ball_search(g, qx, qy, qz, limit_d2, best);
  return best;
}

// Exact 1-NN of q given the match (sorted position j_seed) of a NEARBY query q_seed: the seed's
// match shifted by (q - q_seed) predicts where q's own match lies; the 3 x 3 x 3 block around
// that prediction is probed first so that the ball to verify is as small as it can be.
PEB_HD NnBest grid_nn_seeded(const GridView& g, float qx, float qy, float qz, int j_seed, float sx, float sy, float sz,
                             float limit_d2) {
  NnBest best;
  const float4 t = g.pts[j_seed];
  best.d2 = l2_simple(qx, qy, qz, t.x, t.y, t.z);
  best.idx = point_index(t);
  best.j = j_seed;
  const int cx = grid_coord(t.x + (qx - sx), g.ox, g.inv_h, g.dx);
  const int cy = grid_coord(t.y + (qy - sy), g.oy, g.inv_h, g.dy);
  const int cz = grid_coord(t.z + (qz - sz), g.oz, g.inv_h, g.dz);
  grid_scan_ring(g, qx, qy, qz, cx, cy, cz, 1, true, 0, 1, best);
  grid_ball_search(g, qx, qy, qz, limit_d2, best);
  return best;
}

// The first half of grid_nn_seeded: the candidate only (an upper bound that still has to be verified
// by a ball search — the caller's own, or the warp-cooperative one of nn_search.cuh).
PEB_HD NnBest grid_nn_seed_probe(const GridView& g, float qx, float qy, float qz, int j_seed, float sx, float sy, float sz) {
  NnBest best;
  const float4 t = g.pts[j_seed];
  best.d2 = l2_simple(qx, qy, qz, t.x, t.y, t.z);
  best.idx = point_index(t);
  best.j = j_seed;
  const int cx = grid_coord(t.x + (qx - sx), g.ox, g.inv_h, g.dx);
  const int cy = grid_coord(t.y + (qy - sy), g.oy, g.inv_h, g.dy);
  const int cz = grid_coord(t.z + (qz - sz), g.oz, g.inv_h, g.dz);
  grid_scan_ring(g, qx, qy, qz, cx, cy, cz, 1, true, 0, 1, best);
  return best;
}

// The same search with a certificate.
// Certificate: the ball is grown by `margin`, and the search also tracks the runner-up distance.
// On return *slack_out is a lower bound on (distance of any OTHER target point) - (distance of the
// winner): every point within sqrt(best) + margin has been examined.  While the query has moved by
// less than slack / 2 since then, the winner is still the exact nearest neighbour and the next
// search can be skipped (icp.cu).  slack <= 0: no certificate (exact tie, or winner beyond limit).
PEB_HD NnBest grid_nn_warm_cert(const GridView& g, float qx, float qy, float qz, int j_prev, float limit_d2,
                                float margin, float* slack_out) {
  NnBest best;
  {
    const float4 p = g.pts[j_prev];
    best.d2 = l2_simple(qx, qy, qz, p.x, p.y, p.z);
#ifdef __CUDA_ARCH__
    best.idx = __float_as_int(p.w);
#else
    memcpy(&best.idx, &p.w, 4);
#endif
    best.j = j_prev;
  }
  float second = FLT_MAX;  // smallest squared distance among examined points other than the winner
  const float pad = 0.001f * g.h + margin;  // 0.001 h >> one ulp of any coordinate (h >= 1e-4 * max |coordinate|)
  const float R = sqrtf(fminf(best.d2, limit_d2)) * 1.0001f + pad;
  const int y0 = grid_coord(qy - R, g.oy, g.inv_h, g.dy), y1 = grid_coord(qy + R, g.oy, g.inv_h, g.dy);
  const int z0 = grid_coord(qz - R, g.oz, g.inv_h, g.dz), z1 = grid_coord(qz + R, g.oz, g.inv_h, g.dz);
  for (int z = z0; z <= z1; ++z) {
    const float dz = grid_slab_dist(qz, g.oz, g.h, z);
    for (int y = y0; y <= y1; ++y) {
      const float dy = grid_slab_dist(qy, g.oy, g.h, y);
      const float dyz2 = dy * dy + dz * dz;
      const float rc = sqrtf(fminf(best.d2, limit_d2)) * 1.0001f + pad;  // radius still to be covered
      const float rx2 = rc * rc - dyz2;
      if (rx2 < 0.0f) continue;
      const float rx = sqrtf(rx2) * 1.0001f;
      const int x0 = grid_coord(qx - rx, g.ox, g.inv_h, g.dx), x1 = grid_coord(qx + rx, g.ox, g.inv_h, g.dx);
      const int base = (z * g.dy + y) * g.dx;
      const uint32_t s = g.cell_start[base + x0], e = g.cell_start[base + x1 + 1];
      for (uint32_t j = s; j < e; ++j) {
        if (static_cast<int>(j) == best.j) continue;
        const float4 p = g.pts[j];
        const float d2 = l2_simple(qx, qy, qz, p.x, p.y, p.z);
#ifdef __CUDA_ARCH__
        const int id = __float_as_int(p.w);
#else
        int id;
        memcpy(&id, &p.w, 4);
#endif
        if (d2 < best.d2 || (d2 == best.d2 && id < best.idx)) {
          second = best.d2;
          best.d2 = d2;
          best.idx = id;
          best.j = static_cast<int>(j);
        } else {
          second = fminf(second, d2);
        }
      }
    }
  }
  if (slack_out) {
    float slack = -1.0f;
    if (best.d2 <= limit_d2) {
      const float db = sqrtf(best.d2);
      // examined points are at least sqrt(second) away, unexamined ones more than db + margin
      slack = fminf(sqrtf(second) - db, margin) - (1e-5f * g.h + 1e-6f * db);
    }
    *slack_out = slack;
  }
  return best;
}

// After this many rings the search gives up on the grid and scans every point (still exact):
// a query that far from all target points costs O(r^3) row visits on the grid, which beats a
// full scan only while r stays small.  Rings 1..16 visit ~6 k rows.
constexpr int kMaxRings = 16;

// First guess of the cell edge for a cloud of n finite points with sorted extents e0 >= e1 >= e2:
// surface-like clouds (area ~ e0 * e1) get `occupancy` points per occupied cell.  h_floor keeps
// cells far above the float resolution of the coordinates.
inline float grid_initial_cell(const float e[3], int n, float occupancy, float maxabs, float* h_floor_out) {
  const float h_floor = fmaxf(maxabs * 1e-4f, 1e-30f);
  float h;
  if (e[0] <= 0.0f) {
    h = fmaxf(h_floor, 1e-6f);  // all points identical
  } else if (e[1] <= e[0] * 1e-6f) {
    h = e[0] * occupancy / static_cast<float>(n);  // a line
  } else {
    h = sqrtf(e[0] * e[1] * occupancy / static_cast<float>(n));
  }
  if (h_floor_out) *h_floor_out = h_floor;
  return fmaxf(h, h_floor);
}

// ---- 3x3 SVD in double: two-sided Jacobi (the JacobiSVD scheme, see oracle/pcl_oracle.cpp) ----
struct Rot2 {
  double c, s;
};

// All indices below are compile-time constants (templates, unrolled loops) so that W, U, V live
// in registers: the solve runs in ONE thread at the end of every iteration launch and sits on the
// critical path of a single align (measured 10 us per iteration with indexed local arrays).
template <int P, int Q>
PEB_HD void rot_left(double (&W)[9], Rot2 j) {
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double xi = W[P * 3 + i], yi = W[Q * 3 + i];
    W[P * 3 + i] = j.c * xi + j.s * yi;
    W[Q * 3 + i] = -j.s * xi + j.c * yi;
  }
}
template <int P, int Q>
PEB_HD void rot_right(double (&W)[9], Rot2 j) {
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double xi = W[i * 3 + P], yi = W[i * 3 + Q];
    W[i * 3 + P] = j.c * xi - j.s * yi;
    W[i * 3 + Q] = j.s * xi + j.c * yi;
  }
}

PEB_HD double det3(const double* a) {
  return a[0] * (a[4] * a[8] - a[5] * a[7]) - a[1] * (a[3] * a[8] - a[5] * a[6]) + a[2] * (a[3] * a[7] - a[4] * a[6]);
}

// one (p, q) step of a two-sided Jacobi sweep ([EIGEN] JacobiSVD + real_2x2_jacobi_svd)
template <int P, int Q>
PEB_HD void jacobi_pair(double (&W)[9], double (&U)[9], double (&V)[9], double& maxDiag, bool& finished) {
  const double precision = 2.0 * DBL_EPSILON;
  const double thr = fmax(DBL_MIN, precision * maxDiag);
  if (!(fabs(W[P * 3 + Q]) > thr || fabs(W[Q * 3 + P]) > thr)) return;
  finished = false;
  const double m00 = W[P * 3 + P], m01 = W[P * 3 + Q], m10 = W[Q * 3 + P], m11 = W[Q * 3 + Q];
  // Same rotations as Eigen's real_2x2_jacobi_svd / makeJacobi, written with reciprocal square
  // roots instead of their divide-sqrt-divide chains: the solve is one thread's serial dependency
  // chain, and every double division or square root in it costs ~100 cycles of latency.
  Rot2 r1;
  const double t = m00 + m11, d = m10 - m01;
  if (fabs(d) < DBL_MIN) {
    r1.s = 0.0;
    r1.c = 1.0;
  } else {
    // u = t / d;  s = 1 / sqrt(1 + u^2) = |d| / hypot(t, d);  c = u * s = t * sign(d) / hypot(t, d)
    const double inv = rsqrt(t * t + d * d);
    r1.s = fabs(d) * inv;
    r1.c = copysign(t, t * d) * inv;
  }
  const double n00 = r1.c * m00 + r1.s * m10, n01 = r1.c * m01 + r1.s * m11, n11 = -r1.s * m01 + r1.c * m11;
  Rot2 jr;
  const double deno = 2.0 * fabs(n01);
  if (deno < DBL_MIN) {
    jr.c = 1.0;
    jr.s = 0.0;
  } else {
    // tan(theta) = sign(tau) / (|tau| + sqrt(tau^2 + 1)),  tau = (n00 - n11) / (2 |n01|)
    // multiply through by 2 |n01|:  tan(theta) = sign(a) * b / (|a| + hypot(a, b)),  a = n00 - n11, b = 2 |n01|
    const double a = n00 - n11;
    const double hyp = sqrt(a * a + deno * deno);
    const double tt = copysign(deno, a > 0.0 ? 1.0 : -1.0) / (fabs(a) + hyp);
    const double nn = rsqrt(tt * tt + 1.0);
    jr.s = -copysign(fabs(tt) * nn, tt) * copysign(1.0, n01);
    jr.c = nn;
  }
  const Rot2 jl{r1.c * jr.c + r1.s * jr.s, r1.s * jr.c - r1.c * jr.s};
  rot_left<P, Q>(W, jl);
  rot_right<P, Q>(U, Rot2{jl.c, -jl.s});
  rot_right<P, Q>(W, jr);
  rot_right<P, Q>(V, jr);
  maxDiag = fmax(maxDiag, fmax(fabs(W[P * 3 + P]), fabs(W[Q * 3 + Q])));
}

template <int I, int J>
PEB_HD void swap_columns(double (&sv)[3], double (&U)[9], double (&V)[9]) {
  const double ts = sv[I];
  sv[I] = sv[J];
  sv[J] = ts;
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const double tu = U[r * 3 + I];
    U[r * 3 + I] = U[r * 3 + J];
    U[r * 3 + J] = tu;
    const double tv = V[r * 3 + I];
    V[r * 3 + I] = V[r * 3 + J];
    V[r * 3 + J] = tv;
  }
}

// A (row-major) = U diag(sv) V^T, sv descending
PEB_HD void svd3(const double (&A)[9], double (&U)[9], double (&sv)[3], double (&V)[9]) {
  double scale = 0.0;
#pragma unroll
  for (int i = 0; i < 9; ++i) scale = fmax(scale, fabs(A[i]));
  if (scale == 0.0) scale = 1.0;
  double W[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    W[i] = A[i] / scale;
    U[i] = V[i] = (i % 4 == 0) ? 1.0 : 0.0;
  }
  double maxDiag = fmax(fabs(W[0]), fmax(fabs(W[4]), fabs(W[8])));
  bool finished = false;
  for (int sweep = 0; sweep < 64 && !finished; ++sweep) {
    finished = true;
    jacobi_pair<1, 0>(W, U, V, maxDiag, finished);  // (p, q) in JacobiSVD's order: (1,0) (2,0) (2,1)
    jacobi_pair<2, 0>(W, U, V, maxDiag, finished);
    jacobi_pair<2, 1>(W, U, V, maxDiag, finished);
  }
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double a = W[i * 3 + i];
    sv[i] = fabs(a) * scale;
    if (a < 0.0) {
#pragma unroll
      for (int r = 0; r < 3; ++r) U[r * 3 + i] = -U[r * 3 + i];
    }
  }
  // selection sort, descending, first maximum wins (Eigen's order of swaps), with constant indices
  {
    const bool one = sv[1] > sv[0];
    const double m01 = one ? sv[1] : sv[0];
    const bool two = sv[2] > m01;
    if ((two ? sv[2] : m01) == 0.0) return;
    if (two)
      swap_columns<0, 2>(sv, U, V);
    else if (one)
      swap_columns<0, 1>(sv, U, V);
    if (sv[2] > sv[1]) swap_columns<1, 2>(sv, U, V);
  }
}

// Orthogonal polar factor of A by scaled Newton iterations, X <- (g X + X^-T / g) / 2 (Higham).
// For det(A) > 0 it equals U V^T of the SVD — umeyama's rotation in the generic case — to double
// precision, at a fraction of the latency of the Jacobi sweeps: ~7 iterations of mostly independent
// multiplies with 3 dependent divide / square-root steps each, against ~12 plane rotations with 5.
// Returns false (caller takes the SVD path) for reflections, rank deficiency or no convergence.
PEB_HD bool polar_rotation3(const double (&A)[9], double (&R)[9]) {
  double n2 = 0.0;
#pragma unroll
  for (int i = 0; i < 9; ++i) n2 += A[i] * A[i];
  if (!(n2 > 0.0)) return false;
  const double inv_norm = rsqrt(n2);
  double X[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) X[i] = A[i] * inv_norm;
  if (!(det3(X) > 1e-15)) return false;  // |X|_F = 1: det = s1 s2 s3 <= 0.2; tiny or negative -> SVD path
  bool scaled = true;
  for (int it = 0; it < 16; ++it) {
    double Cf[9];  // cofactors: X^-T = Cf / det
    Cf[0] = X[4] * X[8] - X[5] * X[7];
    Cf[1] = X[5] * X[6] - X[3] * X[8];
    Cf[2] = X[3] * X[7] - X[4] * X[6];
    Cf[3] = X[2] * X[7] - X[1] * X[8];
    Cf[4] = X[0] * X[8] - X[2] * X[6];
    Cf[5] = X[1] * X[6] - X[0] * X[7];
    Cf[6] = X[1] * X[5] - X[2] * X[4];
    Cf[7] = X[2] * X[3] - X[0] * X[5];
    Cf[8] = X[0] * X[4] - X[1] * X[3];
    const double det = X[0] * Cf[0] + X[1] * Cf[1] + X[2] * Cf[2];
    if (!(det > 0.0)) return false;
    double a, b;  // X <- a X + b Cf
    if (scaled) {
      // Any positive scaling keeps the iteration on course; only its speed depends on g.  The
      // scaled steps therefore take g, 1/g and 1/det from single-precision MUFU operations
      // (~20 cycles each) instead of double divisions and square roots (~200 cycles each, in series).
      float nx2 = 0.0f, nc2 = 0.0f;
#pragma unroll
      for (int i = 0; i < 9; ++i) {
        nx2 += static_cast<float>(X[i]) * static_cast<float>(X[i]);
        nc2 += static_cast<float>(Cf[i]) * static_cast<float>(Cf[i]);
      }
      const float fdet = static_cast<float>(det);
      // g^4 = |X^-T|_F^2 / |X|_F^2 = nc2 / (det^2 nx2)
      const float g2 = sqrtf(nc2 / (fdet * fdet * nx2));
      const float g = sqrtf(g2);
      a = 0.5 * static_cast<double>(g);
      b = static_cast<double>(0.5f / (g * fdet));
    } else {
      a = 0.5;
      b = 0.5 / det;
    }
    double delta = 0.0;
#pragma unroll
    for (int i = 0; i < 9; ++i) {
      const double xn = a * X[i] + b * Cf[i];
      delta = fmax(delta, fabs(xn - X[i]));
      X[i] = xn;
    }
    if (delta < 1e-2) scaled = false;  // close to orthogonal: plain (exact) Newton converges quadratically
    if (delta < 1e-15) {
#pragma unroll
      for (int i = 0; i < 9; ++i) R[i] = X[i];
      return true;
    }
  }
  return false;
}

// Accumulator layouts of the two estimators (doubles):
//   SVD   : [0] n  [1..3] sum s  [4..6] sum t  [7..15] sum t_r*s_c (row-major)  [16] sum d2
//   LLS   : [0] n  [1..21] upper triangle of ATA (row-major)  [22..27] ATb  [28] sum d2
constexpr int kAccSvd = 17;
constexpr int kAccLls = 29;
constexpr int kAccMax = 32;

// umeyama's rotation through the SVD, with its reflection and rank-2 cases
// ([PCL] common/impl/eigen.hpp : pcl::umeyama): the path for everything polar_rotation3 declines.
PEB_HD void umeyama_rotation_svd(const double (&sigma)[9], double (&R)[9]) {
  double U[9], V[9], sv[3];
  svd3(sigma, U, sv, V);
  double S[3] = {1.0, 1.0, 1.0};
  if (det3(sigma) < 0.0) S[2] = -1.0;
  int rank = 0;
#pragma unroll
  for (int i = 0; i < 3; ++i)
    if (!(fabs(sv[i]) <= fabs(sv[0]) * 1e-12)) ++rank;
  if (rank == 2) {
    if (det3(U) * det3(V) > 0.0) {
      S[2] = 1.0;
    } else {
      S[2] = -1.0;
    }
  }
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      double a = 0.0;
#pragma unroll
      for (int k = 0; k < 3; ++k) a += U[r * 3 + k] * S[k] * V[c * 3 + k];
      R[r * 3 + c] = a;
    }
}

// T = [R | dst_mean - R src_mean], cast to float like umeyama's Matrix4f result
PEB_HD Mat4 umeyama_pack(const double (&R)[9], const double (&sm)[3], const double (&tm)[3]) {
  Mat4 T = mat4_identity();
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    double a = 0.0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      T.m[c * 4 + r] = static_cast<float>(R[r * 3 + c]);
      a += R[r * 3 + c] * sm[c];
    }
    T.m[12 + r] = static_cast<float>(tm[r] - a);
  }
  return T;
}

// [PCL] common/impl/eigen.hpp : pcl::umeyama (no scaling) from the moment sums, in double.
// PCL runs it in float on demeaned 3 x n matrices; sums of the raw moments in double carry
// ~1e-13 relative error, far below PCL's own float noise (SURVEY.md H2b).
PEB_HD Mat4 umeyama_from_sums(const double* acc) {
  const double n = acc[0];
  const double inv_n = 1.0 / n;
  double sm[3], tm[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    sm[i] = acc[1 + i] * inv_n;
    tm[i] = acc[4 + i] * inv_n;
  }
  double sigma[9];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) sigma[r * 3 + c] = acc[7 + r * 3 + c] * inv_n - tm[r] * sm[c];
  double R[9];
  if (!polar_rotation3(sigma, R)) umeyama_rotation_svd(sigma, R);
  return umeyama_pack(R, sm, tm);
}

// x = ATA^-1 ATb by LU with partial pivoting ([EIGEN] fixed 6x6 inverse() goes through
// PartialPivLU), then [PCL] constructTransformationMatrix (double trig, cast to float).
PEB_HD Mat4 lls_from_sums(const double* acc) {
  double A[36], b[6];
  int k = 1;
  for (int r = 0; r < 6; ++r)
    for (int c = r; c < 6; ++c) {
      A[r * 6 + c] = acc[k];
      A[c * 6 + r] = acc[k];
      ++k;
    }
  for (int r = 0; r < 6; ++r) b[r] = acc[22 + r];
  for (int col = 0; col < 6; ++col) {
    int piv = col;
    double bestv = fabs(A[col * 6 + col]);
    for (int r = col + 1; r < 6; ++r)
      if (fabs(A[r * 6 + col]) > bestv) {
        bestv = fabs(A[r * 6 + col]);
        piv = r;
      }
    if (piv != col) {
      for (int c = 0; c < 6; ++c) {
        double t = A[col * 6 + c];
        A[col * 6 + c] = A[piv * 6 + c];
        A[piv * 6 + c] = t;
      }
      double t = b[col];
      b[col] = b[piv];
      b[piv] = t;
    }
    if (A[col * 6 + col] == 0.0) continue;
    for (int r = col + 1; r < 6; ++r) {
      double f = A[r * 6 + col] / A[col * 6 + col];
      for (int c = col + 1; c < 6; ++c) A[r * 6 + c] -= f * A[col * 6 + c];
      b[r] -= f * b[col];
    }
  }
  double x[6];
  for (int r = 5; r >= 0; --r) {
    double v = b[r];
    for (int c = r + 1; c < 6; ++c) v -= A[r * 6 + c] * x[c];
    x[r] = v / A[r * 6 + r];
  }
  const double alpha = x[0], beta = x[1], gamma = x[2];
  const double ca = cos(alpha), sa = sin(alpha), cb = cos(beta), sb = sin(beta), cg = cos(gamma), sg = sin(gamma);
  Mat4 T;
  for (int i = 0; i < 16; ++i) T.m[i] = 0.0f;
  T.m[0] = static_cast<float>(cg * cb);
  T.m[4] = static_cast<float>(-sg * ca + cg * sb * sa);
  T.m[8] = static_cast<float>(sg * sa + cg * sb * ca);
  T.m[1] = static_cast<float>(sg * cb);
  T.m[5] = static_cast<float>(cg * ca + sg * sb * sa);
  T.m[9] = static_cast<float>(-cg * sa + sg * sb * ca);
  T.m[2] = static_cast<float>(-sb);
  T.m[6] = static_cast<float>(cb * sa);
  T.m[10] = static_cast<float>(cb * ca);
  T.m[12] = static_cast<float>(x[3]);
  T.m[13] = static_cast<float>(x[4]);
  T.m[14] = static_cast<float>(x[5]);
  T.m[15] = 1.0f;
  return T;
}

// ---- per-hypothesis ICP state, advanced on the device ---------------------------------------
struct IcpState {
  Mat4 inc;        // transformation_ (increment of the last completed iteration)
  Mat4 final_t;    // final_transformation_
  double prev_mse, cur_mse;
  double fit_sum;
  int iterations, state, converged, similar;
  int ncorr, active, fit_n, pad0;
  unsigned ticket, ticket_fit;
  unsigned ticket_search;  // split iterations of a batch (icp.cu : icp_search_kernel): search blocks of the launch done
  int searched;            // ... and search launches of this hypothesis completed
};

struct IcpCriteria {
  int max_iterations, min_correspondences, max_similar, estimator;
  double rotation_threshold, translation_threshold, mse_rel, mse_abs;
};

// [PCL] registration/impl/icp.hpp (loop body after the correspondences are known) +
// registration/impl/default_convergence_criteria.hpp : hasConverged.  inc = the estimator's
// transformation_, sum_d2 / n = this iteration's correspondences.
PEB_HD void icp_finish_iteration_scripted(IcpState& st, const IcpCriteria& cr, const Mat4& inc, double sum_d2, int n) {
  st.ncorr = n;
  if (n < cr.min_correspondences) {
    st.state = PEB_NO_CORRESPONDENCES;
    st.converged = 0;
    st.active = 0;
    return;
  }
  st.inc = inc;
  st.final_t = mat4_mul(st.inc, st.final_t);
  st.iterations += 1;
  // hasConverged()
  bool is_similar = false;
  bool ret = false;
  int state = PEB_NOT_CONVERGED;
  const float* t = st.inc.m;
  do {
    if (st.iterations >= cr.max_iterations) {
      state = PEB_ITERATIONS;
      ret = true;
      break;
    }
    double cos_angle = 0.5 * static_cast<double>(t[0] + t[5] + t[10] - 1.0f);
    double translation_sqr = static_cast<double>(t[12] * t[12] + t[13] * t[13] + t[14] * t[14]);
    if (cos_angle >= cr.rotation_threshold && translation_sqr <= cr.translation_threshold) {
      if (st.similar >= cr.max_similar) {
        state = PEB_TRANSFORM;
        ret = true;
        break;
      }
      is_similar = true;
    }
    st.cur_mse = sum_d2 / static_cast<double>(n);
    if (fabs(st.cur_mse - st.prev_mse) < cr.mse_abs) {
      if (st.similar >= cr.max_similar) {
        state = PEB_ABS_MSE;
        ret = true;
        break;
      }
      is_similar = true;
    }
    if (fabs(st.cur_mse - st.prev_mse) / st.prev_mse < cr.mse_rel) {
      if (st.similar >= cr.max_similar) {
        state = PEB_REL_MSE;
        ret = true;
        break;
      }
      is_similar = true;
    }
    if (is_similar)
      st.similar += 1;
    else
      st.similar = 0;
    st.prev_mse = st.cur_mse;
  } while (false);
  st.state = state;
  st.converged = ret ? 1 : 0;
  st.active = (state == PEB_NOT_CONVERGED) ? 1 : 0;
}

// acc = the reduced moment sums of the iteration (layouts above)
PEB_HD void icp_finish_iteration(IcpState& st, const IcpCriteria& cr, const double* acc) {
  const int n = static_cast<int>(acc[0]);
  Mat4 inc = st.inc;
  if (n >= cr.min_correspondences)
    inc = (cr.estimator == PEB_ESTIMATOR_SVD) ? umeyama_from_sums(acc) : lls_from_sums(acc);
  icp_finish_iteration_scripted(st, cr, inc, acc[cr.estimator == PEB_ESTIMATOR_SVD ? 16 : 28], n);
}

// ---- [PCL] common/impl/eigen.hpp : computeRoots2 / computeRoots / eigen33, float -------------
PEB_HD void compute_roots2(float b, float c, float* roots) {
  roots[0] = 0.0f;
  float d = static_cast<float>(static_cast<double>(b * b) - 4.0 * static_cast<double>(c));
  if (d < 0.0f) d = 0.0f;
  float sd = sqrtf(d);
  roots[2] = 0.5f * (b + sd);
  roots[1] = 0.5f * (b - sd);
}

PEB_HD void compute_roots(const float* m, float* roots) {
  float c0 = m[0] * m[4] * m[8] + 2.0f * m[1] * m[2] * m[5] - m[0] * m[5] * m[5] - m[4] * m[2] * m[2] -
             m[8] * m[1] * m[1];
  float c1 = m[0] * m[4] - m[1] * m[1] + m[0] * m[8] - m[2] * m[2] + m[4] * m[8] - m[5] * m[5];
  float c2 = m[0] + m[4] + m[8];
  if (fabsf(c0) < FLT_EPSILON) {
    compute_roots2(c2, c1, roots);
  } else {
    const float s_inv3 = static_cast<float>(1.0 / 3.0);
    const float s_sqrt3 = sqrtf(3.0f);
    float c2_over_3 = c2 * s_inv3;
    float a_over_3 = (c1 - c2 * c2_over_3) * s_inv3;
    if (a_over_3 > 0.0f) a_over_3 = 0.0f;
    float half_b = 0.5f * (c0 + c2_over_3 * (2.0f * c2_over_3 * c2_over_3 - c1));
    float q = half_b * half_b + a_over_3 * a_over_3 * a_over_3;
    if (q > 0.0f) q = 0.0f;
    float rho = sqrtf(-a_over_3);
    float theta = atan2f(sqrtf(-q), half_b) * s_inv3;
    float cos_theta = cosf(theta);
    float sin_theta = sinf(theta);
    roots[0] = c2_over_3 + 2.0f * rho * cos_theta;
    roots[1] = c2_over_3 - rho * (cos_theta + s_sqrt3 * sin_theta);
    roots[2] = c2_over_3 - rho * (cos_theta - s_sqrt3 * sin_theta);
    float t;
    if (roots[0] >= roots[1]) {
      t = roots[0];
      roots[0] = roots[1];
      roots[1] = t;
    }
    if (roots[1] >= roots[2]) {
      t = roots[1];
      roots[1] = roots[2];
      roots[2] = t;
      if (roots[0] >= roots[1]) {
        t = roots[0];
        roots[0] = roots[1];
        roots[1] = t;
      }
    }
    if (roots[0] <= 0.0f) compute_roots2(c2, c1, roots);
  }
}

PEB_HD void eigen33_smallest(const float* mat, float& eigenvalue, float* ev) {
  float scale = 0.0f;
  for (int i = 0; i < 9; ++i) scale = fmaxf(scale, fabsf(mat[i]));
  if (scale <= FLT_MIN) scale = 1.0f;
  float s[9];
  for (int i = 0; i < 9; ++i) s[i] = mat[i] / scale;
  float roots[3];
  compute_roots(s, roots);
  eigenvalue = roots[0] * scale;
  s[0] -= roots[0];
  s[4] -= roots[0];
  s[8] -= roots[0];
  float v1[3], v2[3], v3[3];
  v1[0] = s[1] * s[5] - s[2] * s[4];
  v1[1] = s[2] * s[3] - s[0] * s[5];
  v1[2] = s[0] * s[4] - s[1] * s[3];
  v2[0] = s[1] * s[8] - s[2] * s[7];
  v2[1] = s[2] * s[6] - s[0] * s[8];
  v2[2] = s[0] * s[7] - s[1] * s[6];
  v3[0] = s[4] * s[8] - s[5] * s[7];
  v3[1] = s[5] * s[6] - s[3] * s[8];
  v3[2] = s[3] * s[7] - s[4] * s[6];
  float l1 = v1[0] * v1[0] + v1[1] * v1[1] + v1[2] * v1[2];
  float l2 = v2[0] * v2[0] + v2[1] * v2[1] + v2[2] * v2[2];
  float l3 = v3[0] * v3[0] + v3[1] * v3[1] + v3[2] * v3[2];
  const float* v;
  float l;
  if (l1 >= l2 && l1 >= l3) {
    v = v1;
    l = l1;
  } else if (l2 >= l1 && l2 >= l3) {
    v = v2;
    l = l2;
  } else {
    v = v3;
    l = l3;
  }
  float sl = sqrtf(l);
  ev[0] = v[0] / sl;
  ev[1] = v[1] / sl;
  ev[2] = v[2] / sl;
}

// [PCL] common/impl/centroid.hpp (computeMeanAndCovarianceMatrix tail) + features/impl/feature.hpp
// (solvePlaneParameters) + features/normal_3d.h (flipNormalTowardsViewpoint).
// accu = the nine float sums (xx xy xz yy yz zz x y z) over cnt neighbours, already accumulated
// in neighbour order.  out8 = pcl::Normal image.
PEB_HD void normal_from_accu(float* accu, int cnt, float px, float py, float pz, float vx, float vy, float vz,
                             float* out8) {
  const float fc = static_cast<float>(cnt);
  for (int i = 0; i < 9; ++i) accu[i] = accu[i] / fc;
  float cov[9];
  cov[0] = accu[0] - accu[6] * accu[6];
  cov[1] = accu[1] - accu[6] * accu[7];
  cov[2] = accu[2] - accu[6] * accu[8];
  cov[4] = accu[3] - accu[7] * accu[7];
  cov[5] = accu[4] - accu[7] * accu[8];
  cov[8] = accu[5] - accu[8] * accu[8];
  cov[3] = cov[1];
  cov[6] = cov[2];
  cov[7] = cov[5];
  float ev, vec[3];
  eigen33_smallest(cov, ev, vec);
  float eig_sum = cov[0] + cov[4] + cov[8];
  float curvature = (eig_sum != 0.0f) ? fabsf(ev / eig_sum) : 0.0f;
  float dx = vx - px, dy = vy - py, dz = vz - pz;
  float cos_theta = (dx * vec[0] + dy * vec[1] + dz * vec[2]);
  if (cos_theta < 0.0f) {
    vec[0] *= -1.0f;
    vec[1] *= -1.0f;
    vec[2] *= -1.0f;
  }
  out8[0] = vec[0];
  out8[1] = vec[1];
  out8[2] = vec[2];
  out8[3] = 0.0f;
  out8[4] = curvature;
  out8[5] = out8[6] = out8[7] = 0.0f;
}

// ---- cv::ppf_match_3d::computeNormalsPC3d (DESIGN.md §13) -----------------------------------
// [CV] core/src/lapack.cpp : hypot<double> — mul, div and sqrt only, so -fmad=false / -ffp-contract=off make the
// device and the host round every step alike
PEB_HD double cv_hypot(double a, double b) {
  a = fabs(a);
  b = fabs(b);
  if (a > b) {
    b /= a;
    return a * sqrt(1 + b * b);
  }
  if (b > 0) {
    a /= b;
    return b * sqrt(1 + a * a);
  }
  return 0;
}

// JacobiImpl_'s rotate(v0, v1)
PEB_HD void cv_rotate(double& v0, double& v1, double c, double s) {
  const double a0 = v0, b0 = v1;
  v0 = a0 * c - b0 * s;
  v1 = a0 * s + b0 * c;
}

template <int K, int L>
PEB_HD void cv_rotate_rows(double (&V)[9], double c, double s) {
#pragma unroll
  for (int i = 0; i < 3; ++i) cv_rotate(V[K * 3 + i], V[L * 3 + i], c, s);
}

template <int K, int M>
PEB_HD void cv_swap_rows(double (&W)[3], double (&V)[9]) {
  const double tw = W[K];
  W[K] = W[M];
  W[M] = tw;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const double tv = V[K * 3 + i];
    V[K * 3 + i] = V[M * 3 + i];
    V[M * 3 + i] = tv;
  }
}

// cv::eigen(A, W, V) for a symmetric 3 x 3 double matrix in an OpenCV built without Eigen: [CV] core/src/lapack.cpp :
// JacobiImpl_<double> with n = 3 (cyclic-by-largest Jacobi, at most n * n * 30 rotations, eps = DBL_EPSILON).
// A is row-major; only its upper triangle is read.  W: eigenvalues, descending; V: eigenvectors as ROWS.
// The three off-diagonal entries and the two pivot indices that vary for n = 3 (indR[0], indC[2]; indR[1] = 2 and
// indC[1] = 0 always) are scalars, so the solver lives in registers.  Like upstream, a pivot index is recomputed only
// for the row / column a rotation touches: a stale indR[0] after a (1, 2) rotation is part of the pivot sequence.
PEB_HD void cv_eigen_sym3(const double (&A)[9], double (&W)[3], double (&V)[9]) {
  const double eps = DBL_EPSILON;
  double a01 = A[1], a02 = A[2], a12 = A[5];
  W[0] = A[0];
  W[1] = A[4];
  W[2] = A[8];
#pragma unroll
  for (int i = 0; i < 9; ++i) V[i] = (i % 4 == 0) ? 1.0 : 0.0;
  int r0 = fabs(a01) < fabs(a02) ? 2 : 1;  // indR[0]: argmax over m > 0 of |A[0][m]|, first maximum wins
  int c2 = fabs(a02) < fabs(a12) ? 1 : 0;  // indC[2]: argmax over m < 2 of |A[m][2]|
  for (int iters = 0; iters < 3 * 3 * 30; ++iters) {
    // pivot (k, l): rows by indR first, then columns by indC, strict < so the first maximum wins
    int k = 0, l;
    double mv = fabs(r0 == 1 ? a01 : a02);
    if (mv < fabs(a12)) {
      mv = fabs(a12);
      k = 1;
    }
    l = k == 0 ? r0 : 2;
    if (mv < fabs(a01)) {
      mv = fabs(a01);
      k = 0;
      l = 1;
    }
    const double a_c2 = c2 == 0 ? a02 : a12;
    if (mv < fabs(a_c2)) {
      k = c2;
      l = 2;
    }
    const double p = k == 1 ? a12 : (l == 1 ? a01 : a02);
    if (fabs(p) <= eps) break;
    const double wk = k == 0 ? W[0] : W[1];
    const double wl = l == 1 ? W[1] : W[2];
    const double y = (wl - wk) * 0.5;
    double t = fabs(y) + cv_hypot(p, y);
    double s = cv_hypot(p, t);
    const double c = t / s;
    s = p / s;
    t = (p / t) * p;
    if (y < 0) {
      s = -s;
      t = -t;
    }
    if (k == 0 && l == 1) {
      a01 = 0;
      W[0] -= t;
      W[1] += t;
      cv_rotate(a02, a12, c, s);  // i > l: (A[k][i], A[l][i])
      cv_rotate_rows<0, 1>(V, c, s);
      r0 = fabs(a01) < fabs(a02) ? 2 : 1;
    } else if (k == 0) {  // (0, 2)
      a02 = 0;
      W[0] -= t;
      W[2] += t;
      cv_rotate(a01, a12, c, s);  // k < i < l: (A[k][i], A[i][l])
      cv_rotate_rows<0, 2>(V, c, s);
      r0 = fabs(a01) < fabs(a02) ? 2 : 1;
      c2 = fabs(a02) < fabs(a12) ? 1 : 0;
    } else {  // (1, 2)
      a12 = 0;
      W[1] -= t;
      W[2] += t;
      cv_rotate(a01, a02, c, s);  // i < k: (A[i][k], A[i][l])
      cv_rotate_rows<1, 2>(V, c, s);
      c2 = fabs(a02) < fabs(a12) ? 1 : 0;
    }
  }
  // selection sort, descending (first maximum wins), rows of V move with W
  {
    int m = 0;
    if (W[0] < W[1]) m = 1;
    if (W[m] < W[2]) m = 2;
    if (m == 1) cv_swap_rows<0, 1>(W, V);
    else if (m == 2) cv_swap_rows<0, 2>(W, V);
    if (W[1] < W[2]) cv_swap_rows<1, 2>(W, V);
  }
}

// [CV] surface_matching/src/ppf_helpers.cpp : meanCovLocalPCInd, one neighbour.  acc = the six distinct products
// (xx xy xz yy yz zz) and the three coordinates, double; every product is formed in float, then widened.  The matrix is
// symmetric bit for bit (a float product commutes), so the six sums stand for upstream's nine.
PEB_HD void cv_moments_add(double (&acc)[9], float x, float y, float z) {
  acc[0] += static_cast<double>(x * x);
  acc[1] += static_cast<double>(x * y);
  acc[2] += static_cast<double>(x * z);
  acc[3] += static_cast<double>(y * y);
  acc[4] += static_cast<double>(y * z);
  acc[5] += static_cast<double>(z * z);
  acc[6] += static_cast<double>(x);
  acc[7] += static_cast<double>(y);
  acc[8] += static_cast<double>(z);
}

// meanCovLocalPCInd's tail (mean and covariance scaled by the reciprocal 1.0 / k, then C -= mu mu^T), cv::eigen, row 2
// of the eigenvectors rounded to float and — flip — flipNormalViewpoint: d = vp - p and d . n in float, left to right.
PEB_HD void cv_normal_from_moments(const double (&acc)[9], int k, float px, float py, float pz, bool flip, float vx, float vy,
                                   float vz, float (&n)[3]) {
  const double inv = 1.0 / k;
  const double mu[3] = {acc[6] * inv, acc[7] * inv, acc[8] * inv};
  double C[9];
  C[0] = acc[0] * inv - mu[0] * mu[0];
  C[1] = acc[1] * inv - mu[0] * mu[1];
  C[2] = acc[2] * inv - mu[0] * mu[2];
  C[4] = acc[3] * inv - mu[1] * mu[1];
  C[5] = acc[4] * inv - mu[1] * mu[2];
  C[8] = acc[5] * inv - mu[2] * mu[2];
  C[3] = C[1];
  C[6] = C[2];
  C[7] = C[5];
  double W[3], V[9];
  cv_eigen_sym3(C, W, V);
  n[0] = static_cast<float>(V[6]);
  n[1] = static_cast<float>(V[7]);
  n[2] = static_cast<float>(V[8]);
  if (flip) {
    const float dx = vx - px, dy = vy - py, dz = vz - pz;
    const float cos_theta = dx * n[0] + dy * n[1] + dz * n[2];
    if (cos_theta < 0) {
      n[0] *= -1;
      n[1] *= -1;
      n[2] *= -1;
    }
  }
}

}  // namespace peb
