// cvicp.cu — cv::ppf_match_3d::ICP::registerModelToScene(model, scene, poses) on the device
// (SURVEY.md 8f rank 2: what the reference runs in the refinement slot,
//  pose_estimation/src/opencv_surface_match.cpp:85-94: ICP icp(250, 0.005f, 2.5f, 8)).
// [CV] opencv_contrib/modules/surface_matching/src/icp.cpp — restated from recollection (DESIGN.md section 9;
// the contrib sources are in neither the reference tree nor this image), the arithmetic OpenCV uses: float clouds,
// double poses and sums.
//
// All poses of a call advance together: one kernel per step of the algorithm with blockIdx.y = pose, the pyramid
// and the per-level iteration loop run on the host (one 8 x n_poses-double read-back per iteration: the
// convergence test of every pose decides whether it takes part in the next one).
//   cv_move_model      model through the pose (double), column sums                 -> meanAvg
//   cv_center_src      subtract meanAvg (float), sum of norms of both clouds        -> scale
//   cv_scale_src       the normalised model of every pose
//   per level:  grid over every step-th scene point (ORIGINAL coordinates, shared by all poses: the exact 1-NN of
//               nn_search.cuh; the query is mapped back from the pose's normalised frame, the squared distance is
//               then taken in the normalised frame in float as FLANN would)
//   cv_level_init      srcPCT = every step-th point of (pose * normalised model)
//   per iteration:
//     cv_nn            nearest scene point + normalised squared distance
//     cv_threshold     median + scale * 1.48257968 * MAD (two exact radix selects at index m / 2), one block per pose
//     cv_pick          per scene point the closest accepted source (atomicMin on (distance, source) keys)
//     cv_accumulate    the 6 x 6 normal equations of the linearised point-to-plane step over the winners + the
//                      Frobenius error: one record per block, the host adds them in block order
//     host             solve, PoseX = [Rx (Ry Rz) | t], fval / fval_old against the level's tolerance
//     cv_move          Src_Moved = PoseX * srcPCT
// Clouds are expected finite: a NaN row makes meanAvg NaN, here as in OpenCV.
#include <algorithm>
#include <cmath>
#include <vector>

#include "block_select.cuh"
#include "nn_search.cuh"

namespace peb {

namespace {

constexpr double kCvEps = 1.192092896e-07;  // OpenCV's EPS
constexpr int kCvAcc = 44;                  // 36 (N) + 6 (r) + fsum + count

struct CvPoseDev {  // per pose, read by the kernels
  double pose[16];  // the transform the next kernel applies (row-major 4x4)
  double mean_avg[3];
  double scale;
  int active;
  int pad;
};

__device__ __forceinline__ void cv_transform(const double* P, const float* r, float* o) {
  // [CV] ppf_helpers.cpp : transformPCPose — homogeneous divide for the point, 3x3 + renormalisation for the normal
  double p[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) p[k] = P[4 * k] * r[0] + P[4 * k + 1] * r[1] + P[4 * k + 2] * r[2] + P[4 * k + 3];
  if (fabs(p[3]) > kCvEps) {
    o[0] = static_cast<float>(p[0] / p[3]);
    o[1] = static_cast<float>(p[1] / p[3]);
    o[2] = static_cast<float>(p[2] / p[3]);
  } else {
    o[0] = o[1] = o[2] = 0.0f;
  }
  double nn[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) nn[k] = P[4 * k] * r[3] + P[4 * k + 1] * r[4] + P[4 * k + 2] * r[5];
  const double norm = sqrt(nn[0] * nn[0] + nn[1] * nn[1] + nn[2] * nn[2]);
  if (norm > kCvEps) {
    o[3] = static_cast<float>(nn[0] / norm);
    o[4] = static_cast<float>(nn[1] / norm);
    o[5] = static_cast<float>(nn[2] / norm);
  } else {
    o[3] = o[4] = o[5] = 0.0f;
  }
}

// block-wide sum of K doubles per thread, fixed order; result in out[0..K) (shared), valid after the call for all threads
template <int K, int T>
__device__ __forceinline__ void block_sum(double (&v)[K], double* sm /* [T/32][K] */, double* out /* [K] */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) {
    double x = v[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xFFFFFFFFu, x, o);
    if (lane == 0) sm[warp * K + k] = x;
  }
  __syncthreads();
  if (threadIdx.x < K) {
    double r = 0.0;
    for (int w = 0; w < T / 32; ++w) r += sm[w * K + threadIdx.x];
    out[threadIdx.x] = r;
  }
  __syncthreads();
}

constexpr int kCvT = 256;

// model through the pose of blockIdx.y; per-block column sums (host adds the blocks in order)
__global__ void __launch_bounds__(kCvT) cv_move_model(const float* __restrict__ model, int n, const CvPoseDev* __restrict__ poses,
                                                      float* __restrict__ src0, double* __restrict__ sums /* [H][blocks][4] */) {
  __shared__ double sm[(kCvT / 32) * 4], tot[4];
  const int h = blockIdx.y;
  const int i = blockIdx.x * kCvT + threadIdx.x;
  double v[4] = {0, 0, 0, 0};
  if (i < n) {
    float o[6];
    cv_transform(poses[h].pose, model + 6 * static_cast<size_t>(i), o);
    float* d = src0 + (static_cast<size_t>(h) * n + i) * 6;
#pragma unroll
    for (int k = 0; k < 6; ++k) d[k] = o[k];
    v[0] = o[0];
    v[1] = o[1];
    v[2] = o[2];
  }
  block_sum<4, kCvT>(v, sm, tot);
  if (threadIdx.x < 4) sums[(static_cast<size_t>(h) * gridDim.x + blockIdx.x) * 4 + threadIdx.x] = tot[threadIdx.x];
}

// column sums of the scene (once per call; blockIdx.y unused)
__global__ void __launch_bounds__(kCvT) cv_scene_sums(const float* __restrict__ scene, int ns, double* __restrict__ sums) {
  __shared__ double sm[(kCvT / 32) * 4], tot[4];
  const int i = blockIdx.x * kCvT + threadIdx.x;
  double v[4] = {0, 0, 0, 0};
  if (i < ns) {
    v[0] = scene[6 * static_cast<size_t>(i)];
    v[1] = scene[6 * static_cast<size_t>(i) + 1];
    v[2] = scene[6 * static_cast<size_t>(i) + 2];
  }
  block_sum<4, kCvT>(v, sm, tot);
  if (threadIdx.x < 4) sums[static_cast<size_t>(blockIdx.x) * 4 + threadIdx.x] = tot[threadIdx.x];
}

// subtractColumns (float) in place for the moved model, and the per-block sums of norms of the centred model
// (x < src_blocks) or of the centred scene (the other blocks); the scene itself is never stored centred
__global__ void __launch_bounds__(kCvT) cv_center(float* __restrict__ src0, int n, const float* __restrict__ scene, int ns,
                                                  const CvPoseDev* __restrict__ poses, int src_blocks,
                                                  double* __restrict__ sums /* [H][blocks][4] */) {
  __shared__ double sm[(kCvT / 32) * 4], tot[4];
  const int h = blockIdx.y;
  const float mx = static_cast<float>(poses[h].mean_avg[0]), my = static_cast<float>(poses[h].mean_avg[1]),
              mz = static_cast<float>(poses[h].mean_avg[2]);
  double v[4] = {0, 0, 0, 0};
  if (static_cast<int>(blockIdx.x) < src_blocks) {
    const int i = blockIdx.x * kCvT + threadIdx.x;
    if (i < n) {
      float* d = src0 + (static_cast<size_t>(h) * n + i) * 6;
      const float x = d[0] - mx, y = d[1] - my, z = d[2] - mz;
      d[0] = x;
      d[1] = y;
      d[2] = z;
      const double dx = x, dy = y, dz = z;
      v[0] = sqrt(dx * dx + dy * dy + dz * dz);
    }
  } else {
    const int i = (blockIdx.x - src_blocks) * kCvT + threadIdx.x;
    if (i < ns) {
      const float* s = scene + 6 * static_cast<size_t>(i);
      const double dx = s[0] - mx, dy = s[1] - my, dz = s[2] - mz;  // float subtraction, widened
      v[1] = sqrt(dx * dx + dy * dy + dz * dz);
    }
  }
  block_sum<4, kCvT>(v, sm, tot);
  if (threadIdx.x < 4) sums[(static_cast<size_t>(h) * gridDim.x + blockIdx.x) * 4 + threadIdx.x] = tot[threadIdx.x];
}

__global__ void __launch_bounds__(kCvT) cv_scale_src(float* __restrict__ src0, int n, const CvPoseDev* __restrict__ poses) {
  const int h = blockIdx.y;
  const int i = blockIdx.x * kCvT + threadIdx.x;
  if (i >= n) return;
  const double s = poses[h].scale;
  float* d = src0 + (static_cast<size_t>(h) * n + i) * 6;
#pragma unroll
  for (int k = 0; k < 3; ++k) d[k] = static_cast<float>(d[k] * s);  // Mat *= double
}

// srcPCT = every step-th row of (pose * src0); Src_Moved starts as a copy
__global__ void __launch_bounds__(kCvT) cv_level_init(const float* __restrict__ src0, int n, int step, int m,
                                                      const CvPoseDev* __restrict__ poses, float* __restrict__ pct,
                                                      float* __restrict__ moved) {
  const int h = blockIdx.y;
  const int s = blockIdx.x * kCvT + threadIdx.x;
  if (s >= m) return;
  float o[6];
  cv_transform(poses[h].pose, src0 + (static_cast<size_t>(h) * n + static_cast<size_t>(s) * step) * 6, o);
  float* a = pct + (static_cast<size_t>(h) * m + s) * 6;
  float* b = moved + (static_cast<size_t>(h) * m + s) * 6;
#pragma unroll
  for (int k = 0; k < 6; ++k) {
    a[k] = o[k];
    b[k] = o[k];
  }
}

__global__ void __launch_bounds__(kCvT) cv_move(const float* __restrict__ pct, int m, const CvPoseDev* __restrict__ poses,
                                                float* __restrict__ moved) {
  const int h = blockIdx.y;
  if (!poses[h].active) return;
  const int s = blockIdx.x * kCvT + threadIdx.x;
  if (s >= m) return;
  float o[6];
  cv_transform(poses[h].pose, pct + (static_cast<size_t>(h) * m + s) * 6, o);
  float* b = moved + (static_cast<size_t>(h) * m + s) * 6;
#pragma unroll
  for (int k = 0; k < 6; ++k) b[k] = o[k];
}

// the level's scene point j in the normalised frame of pose h: ((float)(s - (float)mean)) * scale -> float
__device__ __forceinline__ void cv_scene_norm(const float* __restrict__ s, const CvPoseDev& p, float* o) {
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float c = s[k] - static_cast<float>(p.mean_avg[k]);
    o[k] = static_cast<float>(c * p.scale);
  }
}

__global__ void __launch_bounds__(128) cv_nn(const GridView g, const float* __restrict__ scene, int step,
                                             const float* __restrict__ moved, int m, const CvPoseDev* __restrict__ poses,
                                             int* __restrict__ idx, float* __restrict__ dist) {
  const int h = blockIdx.y;
  if (!poses[h].active) return;
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= m) return;
  const CvPoseDev& P = poses[h];
  const float* q = moved + (static_cast<size_t>(h) * m + s) * 6;
  // back to the scene's own coordinates for the search
  const float ox = static_cast<float>(q[0] / P.scale + P.mean_avg[0]);
  const float oy = static_cast<float>(q[1] / P.scale + P.mean_avg[1]);
  const float oz = static_cast<float>(q[2] / P.scale + P.mean_avg[2]);
  const NnBest best = grid_nn<1>(g, ox, oy, oz, pos_inf());
  float d2 = 0.0f;
  if (best.idx >= 0) {
    float t[3];
    cv_scene_norm(scene + 6 * static_cast<size_t>(best.idx) * step, P, t);
    d2 = l2_simple(q[0], q[1], q[2], t[0], t[1], t[2]);  // FLANN L2 in the normalised frame, float
  }
  idx[static_cast<size_t>(h) * m + s] = best.idx;
  dist[static_cast<size_t>(h) * m + s] = d2;
}

// The same for a coarse pyramid level: the few thousand scene points of the level are scanned directly from shared-memory
// tiles (no grid to build); same distance arithmetic and tie rule (smaller distance, then lower index) as the grid search.
constexpr int kCvBruteMax = 4096;     // level scene points up to which no grid is built
__global__ void __launch_bounds__(128) cv_nn_brute(const float4* __restrict__ lvl, int msl, const float* __restrict__ scene, int step,
                                                   const float* __restrict__ moved, int m, const CvPoseDev* __restrict__ poses,
                                                   int* __restrict__ idx, float* __restrict__ dist) {
  __shared__ float4 tile[512];
  const int h = blockIdx.y;
  if (!poses[h].active) return;
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  const CvPoseDev& P = poses[h];
  float q[3] = {0.f, 0.f, 0.f}, ox = 0.f, oy = 0.f, oz = 0.f;
  if (s < m) {
    const float* qq = moved + (static_cast<size_t>(h) * m + s) * 6;
    q[0] = qq[0];
    q[1] = qq[1];
    q[2] = qq[2];
    ox = static_cast<float>(q[0] / P.scale + P.mean_avg[0]);
    oy = static_cast<float>(q[1] / P.scale + P.mean_avg[1]);
    oz = static_cast<float>(q[2] / P.scale + P.mean_avg[2]);
  }
  float best_d = pos_inf();
  int best_j = -1;
  for (int t0 = 0; t0 < msl; t0 += 512) {
    const int cnt = min(512, msl - t0);
    __syncthreads();
    for (int k = threadIdx.x; k < cnt; k += blockDim.x) tile[k] = lvl[t0 + k];
    __syncthreads();
    for (int k = 0; k < cnt; ++k) {
      const float4 p = tile[k];
      if (!finite3(p.x, p.y, p.z)) continue;  // (the grid leaves non-finite points out as well)
      const float d2 = l2_simple(ox, oy, oz, p.x, p.y, p.z);
      if (d2 < best_d) {  // ascending index: the first of equal distances stays
        best_d = d2;
        best_j = t0 + k;
      }
    }
  }
  if (s >= m) return;
  float d2 = 0.0f;
  if (best_j >= 0) {
    float t[3];
    cv_scene_norm(scene + 6 * static_cast<size_t>(best_j) * step, P, t);
    d2 = l2_simple(q[0], q[1], q[2], t[0], t[1], t[2]);
  }
  idx[static_cast<size_t>(h) * m + s] = best_j;
  dist[static_cast<size_t>(h) * m + s] = d2;
}

// [CV] icp.cpp : getRejectionThreshold — one block per pose
__global__ void __launch_bounds__(1024) cv_threshold(const float* __restrict__ dist, int m, float rejection_scale,
                                                     const CvPoseDev* __restrict__ poses, float* __restrict__ thr) {
  __shared__ unsigned hist[2048];
  __shared__ unsigned st[2];
  __shared__ unsigned wsum[32];
  const int h = blockIdx.x;
  if (!poses[h].active) return;
  const float* d = dist + static_cast<size_t>(h) * m;
  const float med = block_select_nth([&](int i) { return d[i]; }, m, m / 2, hist, st, wsum);
  const float mad = block_select_nth([&](int i) { return fabsf(d[i] - med); }, m, m / 2, hist, st, wsum);
  if (threadIdx.x == 0) {
    const float sgm = 1.48257968f * mad;
    thr[h] = rejection_scale * sgm + med;
  }
}

// "picky ICP": per scene point the closest accepted source; ties go to the smaller source index
__global__ void __launch_bounds__(kCvT) cv_pick(const int* __restrict__ idx, const float* __restrict__ dist, int m, int ms,
                                                const float* __restrict__ thr, int robust, const CvPoseDev* __restrict__ poses,
                                                unsigned long long* __restrict__ keys) {
  const int h = blockIdx.y;
  if (!poses[h].active) return;
  const int s = blockIdx.x * kCvT + threadIdx.x;
  if (s >= m) return;
  const int j = idx[static_cast<size_t>(h) * m + s];
  const float d = dist[static_cast<size_t>(h) * m + s];
  if (j < 0) return;
  if (robust && !(d < thr[h])) return;
  const unsigned long long key = (static_cast<unsigned long long>(__float_as_uint(d)) << 32) | static_cast<unsigned>(s);
  atomicMin(&keys[static_cast<size_t>(h) * ms + j], key);
}

// normal equations of the linearised point-to-plane step over the winners: kCvAccBlocks blocks per pose, one record of
// kCvAcc doubles per block (the host adds the records in block order: fixed summation order)
constexpr int kCvAccBlocks = 48;
__global__ void __launch_bounds__(kCvT) cv_accumulate(const float* __restrict__ pct, const float* __restrict__ scene, int step,
                                                      const int* __restrict__ idx, const float* __restrict__ dist, int m, int ms,
                                                      const unsigned long long* __restrict__ keys,
                                                      const CvPoseDev* __restrict__ poses, double* __restrict__ acc_out) {
  __shared__ double sm[(kCvT / 32) * 4], tot[4];
  const int h = blockIdx.y;
  if (!poses[h].active) return;
  const CvPoseDev& P = poses[h];
  double v[kCvAcc];
#pragma unroll
  for (int e = 0; e < kCvAcc; ++e) v[e] = 0.0;
  for (int s = blockIdx.x * kCvT + threadIdx.x; s < m; s += gridDim.x * kCvT) {
    const int j = idx[static_cast<size_t>(h) * m + s];
    if (j < 0) continue;
    const unsigned long long key =
        (static_cast<unsigned long long>(__float_as_uint(dist[static_cast<size_t>(h) * m + s])) << 32) | static_cast<unsigned>(s);
    if (keys[static_cast<size_t>(h) * ms + j] != key) continue;  // not the winner of its scene point (or rejected)
    const float* sp = pct + (static_cast<size_t>(h) * m + s) * 6;
    const float* dr = scene + 6 * static_cast<size_t>(j) * step;
    float dn[3];
    cv_scene_norm(dr, P, dn);
    const double sx = sp[0], sy = sp[1], sz = sp[2], dx = dn[0], dy = dn[1], dz = dn[2], nx = dr[3], ny = dr[4], nz = dr[5];
    const double row[6] = {sy * nz - sz * ny, sz * nx - sx * nz, sx * ny - sy * nx, nx, ny, nz};
    const double b = (dx - sx) * nx + (dy - sy) * ny + (dz - sz) * nz;
#pragma unroll
    for (int a = 0; a < 6; ++a) {
#pragma unroll
      for (int c = 0; c < 6; ++c) v[6 * a + c] += row[a] * row[c];
      v[36 + a] += row[a] * b;
    }
    const double e0 = sx - dx, e1 = sy - dy, e2 = sz - dz, e3 = static_cast<double>(sp[3]) - nx,
                 e4 = static_cast<double>(sp[4]) - ny, e5 = static_cast<double>(sp[5]) - nz;
    v[42] += e0 * e0 + e1 * e1 + e2 * e2 + e3 * e3 + e4 * e4 + e5 * e5;
    v[43] += 1.0;
  }
  double* out = acc_out + (static_cast<size_t>(h) * gridDim.x + blockIdx.x) * kCvAcc;
#pragma unroll
  for (int g0 = 0; g0 < kCvAcc; g0 += 4) {
    double w[4] = {v[g0], v[g0 + 1], v[g0 + 2], v[g0 + 3]};
    block_sum<4, kCvT>(w, sm, tot);
    if (threadIdx.x < 4) out[g0 + threadIdx.x] = tot[threadIdx.x];
    __syncthreads();
  }
}

__global__ void cv_gather_xyz(const float* __restrict__ scene, int step, int ms, float4* __restrict__ out) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= ms) return;
  const float* s = scene + 6 * static_cast<size_t>(j) * step;
  out[j] = make_float4(s[0], s[1], s[2], 1.0f);
}

// ---- host side ------------------------------------------------------------------------------------
int cv_round(double v) { return static_cast<int>(std::lrint(v)); }  // cvRound

void mat44_mul(const double* A, const double* B, double* C) {
  double t[16];
  for (int r = 0; r < 4; ++r)
    for (int c = 0; c < 4; ++c) {
      double a = 0.0;
      for (int k = 0; k < 4; ++k) a += A[4 * r + k] * B[4 * k + c];
      t[4 * r + c] = a;
    }
  std::copy(t, t + 16, C);
}

// [CV] c_utils.hpp : eulerToDCM (R = Rx (Ry Rz)) + rtToPose
void pose_from_euler(const double* e, const double* t, double* P) {
  const double cx = std::cos(e[0]), sx = std::sin(e[0]), cy = std::cos(e[1]), sy = std::sin(e[1]), cz = std::cos(e[2]),
               sz = std::sin(e[2]);
  const double Rx[9] = {1, 0, 0, 0, cx, -sx, 0, sx, cx};
  const double Ry[9] = {cy, 0, sy, 0, 1, 0, -sy, 0, cy};
  const double Rz[9] = {cz, -sz, 0, sz, cz, 0, 0, 0, 1};
  double T[9], R[9];
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) T[3 * r + c] = Ry[3 * r] * Rz[c] + Ry[3 * r + 1] * Rz[3 + c] + Ry[3 * r + 2] * Rz[6 + c];
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) R[3 * r + c] = Rx[3 * r] * T[c] + Rx[3 * r + 1] * T[3 + c] + Rx[3 * r + 2] * T[6 + c];
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) P[4 * r + c] = R[3 * r + c];
    P[4 * r + 3] = t[r];
  }
  P[12] = P[13] = P[14] = 0.0;
  P[15] = 1.0;
}

// the minimiser of |A x - b| through the normal equations (elimination with partial pivoting, double)
bool solve6(double* N, double* r, double* x) {
  for (int c = 0; c < 6; ++c) {
    int best = c;
    for (int rr = c + 1; rr < 6; ++rr)
      if (std::fabs(N[6 * rr + c]) > std::fabs(N[6 * best + c])) best = rr;
    if (!(std::fabs(N[6 * best + c]) > 0.0)) return false;
    if (best != c) {
      for (int k = 0; k < 6; ++k) std::swap(N[6 * c + k], N[6 * best + k]);
      std::swap(r[c], r[best]);
    }
    for (int rr = c + 1; rr < 6; ++rr) {
      const double f = N[6 * rr + c] / N[6 * c + c];
      for (int k = c; k < 6; ++k) N[6 * rr + k] -= f * N[6 * c + k];
      r[rr] -= f * r[c];
    }
  }
  for (int c = 5; c >= 0; --c) {
    double a = r[c];
    for (int k = c + 1; k < 6; ++k) a -= N[6 * c + k] * x[k];
    x[c] = a / N[6 * c + c];
  }
  return true;
}

void identity44(double* P) {
  for (int i = 0; i < 16; ++i) P[i] = (i % 5 == 0) ? 1.0 : 0.0;
}

}  // namespace

// the argument checks, before anything is uploaded
static int cvicp_check(peb_ctx* ctx, size_t n_model, size_t n_scene, const peb_cvicp_params* prm, size_t n_poses) {
  if (prm->iterations < 0 || prm->num_levels < 1 || prm->num_levels > 16)
    return fail(ctx, PEB_E_INVALID_ARG, "cvicp: iterations >= 0 and 1 <= num_levels <= 16 expected");
  if (n_poses == 0) return PEB_OK;
  if (n_model == 0 || n_scene == 0) return fail(ctx, PEB_E_INVALID_ARG, "cvicp: empty model or scene");
  if (n_poses > 4096) return fail(ctx, PEB_E_UNSUPPORTED, "cvicp: at most 4096 poses per call");
  if (n_model > (1u << 26) || n_scene > (1u << 26)) return fail(ctx, PEB_E_INVALID_ARG, "cvicp: cloud too large");
  return PEB_OK;
}

int cvicp_register_device(peb_ctx* ctx, const float* h_model, size_t n_model, const float* h_scene, size_t n_scene,
                          const peb_cvicp_params* prm, double* poses, size_t n_poses, double* residuals) {
  PEB_TRY(cvicp_check(ctx, n_model, n_scene, prm, n_poses));
  if (n_poses == 0) return PEB_OK;
  // the two uploads: model and scene one after the other in ctx->cv_in
  const size_t model_bytes = (sizeof(float) * 6 * n_model + 255) & ~static_cast<size_t>(255);
  PEB_CUDA(ctx, ctx->cv_in.ensure(model_bytes + sizeof(float) * 6 * n_scene));
  float* d_model = ctx->cv_in.as<float>();
  float* d_scene = reinterpret_cast<float*>(ctx->cv_in.as<char>() + model_bytes);
  PEB_CUDA(ctx, cudaMemcpyAsync(d_model, h_model, sizeof(float) * 6 * n_model, cudaMemcpyHostToDevice, ctx->stream));
  PEB_CUDA(ctx, cudaMemcpyAsync(d_scene, h_scene, sizeof(float) * 6 * n_scene, cudaMemcpyHostToDevice, ctx->stream));
  return cvicp_register_core(ctx, d_model, n_model, d_scene, n_scene, prm, poses, n_poses, residuals);
}

int cvicp_register_core(peb_ctx* ctx, const float* d_model, size_t n_model, const float* d_scene, size_t n_scene,
                        const peb_cvicp_params* prm, double* poses, size_t n_poses, double* residuals) {
  PEB_TRY(cvicp_check(ctx, n_model, n_scene, prm, n_poses));
  if (n_poses == 0) return PEB_OK;
  const int n = static_cast<int>(n_model), ns = static_cast<int>(n_scene), H = static_cast<int>(n_poses);
  cudaStream_t st = ctx->stream;
  const bool robust = prm->rejection_scale > 0.0f;

  // ---- device buffers (one arena; sizes for level 0, the largest) ----
  const int sblocks = ceil_div(n, kCvT), dblocks = ceil_div(ns, kCvT);
  size_t off = 0;
  auto carve = [&](size_t bytes) {
    const size_t o = off;
    off += (bytes + 255) & ~static_cast<size_t>(255);
    return o;
  };
  const size_t o_src0 = carve(sizeof(float) * 6 * n * static_cast<size_t>(H));
  const size_t o_pct = carve(sizeof(float) * 6 * n * static_cast<size_t>(H)), o_moved = carve(sizeof(float) * 6 * n * static_cast<size_t>(H));
  const size_t o_idx = carve(sizeof(int) * n * static_cast<size_t>(H)), o_dist = carve(sizeof(float) * n * static_cast<size_t>(H));
  const size_t o_keys = carve(sizeof(unsigned long long) * ns * static_cast<size_t>(H));
  const size_t o_lvl = carve(sizeof(float4) * ns);
  const size_t o_poses = carve(sizeof(CvPoseDev) * H);
  const size_t o_sums = carve(sizeof(double) * 4 * static_cast<size_t>(H) * (sblocks + dblocks));
  const size_t o_acc = carve(sizeof(double) * kCvAcc * kCvAccBlocks * H), o_thr = carve(sizeof(float) * H);
  PEB_CUDA(ctx, ctx->cv_arena.ensure(off));
  char* base = ctx->cv_arena.as<char>();
  float* d_src0 = reinterpret_cast<float*>(base + o_src0);
  float* d_pct = reinterpret_cast<float*>(base + o_pct);
  float* d_moved = reinterpret_cast<float*>(base + o_moved);
  int* d_idx = reinterpret_cast<int*>(base + o_idx);
  float* d_dist = reinterpret_cast<float*>(base + o_dist);
  unsigned long long* d_keys = reinterpret_cast<unsigned long long*>(base + o_keys);
  float4* d_lvl = reinterpret_cast<float4*>(base + o_lvl);
  CvPoseDev* d_poses = reinterpret_cast<CvPoseDev*>(base + o_poses);
  double* d_sums = reinterpret_cast<double*>(base + o_sums);
  double* d_acc = reinterpret_cast<double*>(base + o_acc);
  float* d_thr = reinterpret_cast<float*>(base + o_thr);

  // pinned staging: two pose tables used alternately (every iteration ends with a synchronising read-back, so a table is
  // never rewritten while its upload is in flight), and the accumulator read-back
  const size_t pose_bytes = (sizeof(CvPoseDev) * H + 255) & ~static_cast<size_t>(255);
  PEB_CUDA(ctx, ctx->h_cv.ensure(2 * pose_bytes + sizeof(double) * kCvAcc * kCvAccBlocks * H));
  CvPoseDev* stage[2] = {reinterpret_cast<CvPoseDev*>(ctx->h_cv.as<char>()), reinterpret_cast<CvPoseDev*>(ctx->h_cv.as<char>() + pose_bytes)};
  double* h_acc = reinterpret_cast<double*>(ctx->h_cv.as<char>() + 2 * pose_bytes);
  int stage_k = 0;
  std::vector<CvPoseDev> hp(H);
  std::vector<double> h_sums(4 * static_cast<size_t>(H) * (sblocks + dblocks));
  auto push_poses = [&]() -> int {
    std::copy(hp.begin(), hp.end(), stage[stage_k]);
    PEB_CUDA(ctx, cudaMemcpyAsync(d_poses, stage[stage_k], sizeof(CvPoseDev) * H, cudaMemcpyHostToDevice, st));
    stage_k ^= 1;
    return PEB_OK;
  };

  // ---- the model through every input pose, meanAvg ----
  for (int h = 0; h < H; ++h) {
    std::copy(poses + 16 * h, poses + 16 * h + 16, hp[h].pose);
    hp[h].active = 1;
    hp[h].scale = 1.0;
    hp[h].mean_avg[0] = hp[h].mean_avg[1] = hp[h].mean_avg[2] = 0.0;
  }
  PEB_TRY(push_poses());
  PEB_LAUNCH(ctx, cv_move_model, dim3(sblocks, H), kCvT, 0, d_model, n, d_poses, d_src0, d_sums);
  double* d_scene_sums = d_sums + 4 * static_cast<size_t>(H) * sblocks;
  PEB_LAUNCH(ctx, cv_scene_sums, dim3(dblocks), kCvT, 0, d_scene, ns, d_scene_sums);
  PEB_CUDA(ctx, cudaMemcpyAsync(h_sums.data(), d_sums, sizeof(double) * 4 * (static_cast<size_t>(H) * sblocks + dblocks),
                                cudaMemcpyDeviceToHost, st));
  PEB_CUDA(ctx, cudaStreamSynchronize(st));
  double mean_dst[3] = {0, 0, 0};
  for (int b = 0; b < dblocks; ++b)
    for (int k = 0; k < 3; ++k) mean_dst[k] += h_sums[4 * (static_cast<size_t>(H) * sblocks + b) + k];
  for (int k = 0; k < 3; ++k) mean_dst[k] /= static_cast<double>(ns);
  for (int h = 0; h < H; ++h) {
    double ms_[3] = {0, 0, 0};
    for (int b = 0; b < sblocks; ++b)
      for (int k = 0; k < 3; ++k) ms_[k] += h_sums[4 * (static_cast<size_t>(h) * sblocks + b) + k];
    for (int k = 0; k < 3; ++k) hp[h].mean_avg[k] = 0.5 * (ms_[k] / static_cast<double>(n) + mean_dst[k]);
  }
  PEB_TRY(push_poses());
  // ---- centre, scale ----
  PEB_LAUNCH(ctx, cv_center, dim3(sblocks + dblocks, H), kCvT, 0, d_src0, n, d_scene, ns, d_poses, sblocks, d_sums);
  PEB_CUDA(ctx, cudaMemcpyAsync(h_sums.data(), d_sums, sizeof(double) * 4 * static_cast<size_t>(H) * (sblocks + dblocks),
                                cudaMemcpyDeviceToHost, st));
  PEB_CUDA(ctx, cudaStreamSynchronize(st));
  for (int h = 0; h < H; ++h) {
    double ds = 0.0, dd = 0.0;
    const size_t row = static_cast<size_t>(h) * (sblocks + dblocks);
    for (int b = 0; b < sblocks; ++b) ds += h_sums[4 * (row + b)];
    for (int b = sblocks; b < sblocks + dblocks; ++b) dd += h_sums[4 * (row + b) + 1];
    hp[h].scale = static_cast<double>(n) / ((ds + dd) * 0.5);
    identity44(hp[h].pose);
  }
  PEB_TRY(push_poses());
  PEB_LAUNCH(ctx, cv_scale_src, dim3(sblocks, H), kCvT, 0, d_src0, n, d_poses);

  // ---- the pyramid ----
  std::vector<double> pose(16 * static_cast<size_t>(H)), pose_x(16 * static_cast<size_t>(H));
  std::vector<double> fval_old(H), fval_perc(H), fval_min(H), temp_res(H, 0.0);
  std::vector<int> it(H), running(H);
  for (int h = 0; h < H; ++h) identity44(&pose[16 * h]);
  for (int level = prm->num_levels - 1; level >= 0; --level) {
    const double div = std::pow(2.0, static_cast<double>(level));
    const int num_samples = cv_round(static_cast<double>(n) / div);
    const double tol_p = static_cast<double>(prm->tolerance) * static_cast<double>(level + 1) * (level + 1);
    const int max_it = cv_round(static_cast<double>(prm->iterations) / (level + 1));
    const int step = std::max(1, cv_round(static_cast<double>(n) / static_cast<double>(std::max(num_samples, 1))));
    // [CV] samplePCUniform: rows / sampleStep (integer division) rows, taken at 0, step, 2 step, ...
    const int m = n / step, msl = ns / step;
    if (m == 0 || msl == 0) continue;  // a level coarser than the clouds: nothing to iterate on (PoseX = I)
    // the level's scene grid (original coordinates, shared by all poses)
    PEB_LAUNCH(ctx, cv_gather_xyz, ceil_div(msl, 256), 256, 0, d_scene, step, msl, d_lvl);
    const bool brute = msl <= kCvBruteMax;  // coarse levels: scanning the level's scene beats building a grid for it
    GridView g{};
    if (!brute) {
      PEB_TRY(grid_build(ctx, &ctx->aux_grid, d_lvl, nullptr, msl, 2.0f));
      g = ctx->aux_grid.view;
    }
    for (int h = 0; h < H; ++h) {
      std::copy(&pose[16 * h], &pose[16 * h] + 16, hp[h].pose);
      hp[h].active = 1;
      fval_old[h] = 9999999999.0;
      fval_perc[h] = 0.0;
      fval_min[h] = 9999999999.0;
      it[h] = 0;
      identity44(&pose_x[16 * h]);
    }
    PEB_TRY(push_poses());
    PEB_LAUNCH(ctx, cv_level_init, dim3(ceil_div(m, kCvT), H), kCvT, 0, d_src0, n, step, m, d_poses, d_pct, d_moved);
    // while (!(fval_perc within 1 -/+ TolP) && i < MaxIterationsPyr): fval_perc starts at 0, so every pose enters if max_it > 0
    int any = 0;
    for (int h = 0; h < H; ++h) {
      running[h] = max_it > 0;
      hp[h].active = running[h];
      any |= running[h];
    }
    if (any) PEB_TRY(push_poses());  // (the kernels of an iteration only read `active`; cv_move also the pose = PoseX)
    while (any) {
      if (brute)
        PEB_LAUNCH(ctx, cv_nn_brute, dim3(ceil_div(m, 128), H), 128, 0, d_lvl, msl, d_scene, step, d_moved, m, d_poses, d_idx, d_dist);
      else
        PEB_LAUNCH(ctx, cv_nn, dim3(ceil_div(m, 128), H), 128, 0, g, d_scene, step, d_moved, m, d_poses, d_idx, d_dist);
      if (robust) PEB_LAUNCH(ctx, cv_threshold, H, 1024, 0, d_dist, m, prm->rejection_scale, d_poses, d_thr);
      PEB_CUDA(ctx, cudaMemsetAsync(d_keys, 0xFF, sizeof(unsigned long long) * msl * static_cast<size_t>(H), st));
      PEB_LAUNCH(ctx, cv_pick, dim3(ceil_div(m, kCvT), H), kCvT, 0, d_idx, d_dist, m, msl, d_thr, robust ? 1 : 0, d_poses, d_keys);
      const int ablocks = std::max(1, std::min(kCvAccBlocks, ceil_div(m, kCvT)));
      PEB_LAUNCH(ctx, cv_accumulate, dim3(ablocks, H), kCvT, 0, d_pct, d_scene, step, d_idx, d_dist, m, msl, d_keys, d_poses, d_acc);
      PEB_CUDA(ctx, cudaMemcpyAsync(h_acc, d_acc, sizeof(double) * kCvAcc * ablocks * H, cudaMemcpyDeviceToHost, st));
      PEB_CUDA(ctx, cudaStreamSynchronize(st));
      any = 0;
      for (int h = 0; h < H; ++h) {
        int next = 0;
        if (running[h]) {
          double a[kCvAcc];
          for (int e = 0; e < kCvAcc; ++e) a[e] = 0.0;
          for (int blk = 0; blk < ablocks; ++blk)  // (records of inactive poses are stale: only running poses are read)
            for (int e = 0; e < kCvAcc; ++e) a[e] += h_acc[(static_cast<size_t>(h) * ablocks + blk) * kCvAcc + e];
          const int sel = static_cast<int>(a[43]);
          double N[36], r[6], x[6];
          std::copy(a, a + 36, N);
          std::copy(a + 36, a + 42, r);
          bool ok = sel >= 6 && solve6(N, r, x);
          if (ok)
            for (int k = 0; k < 6; ++k) ok = ok && !std::isnan(x[k]);
          if (ok) {  // (else: "break" — the level ends for this pose with the PoseX it has)
            pose_from_euler(x, x + 3, &pose_x[16 * h]);
            const double fval = std::sqrt(a[42]) / static_cast<double>(m);
            fval_perc[h] = fval / fval_old[h];
            fval_old[h] = fval;
            if (fval < fval_min[h]) fval_min[h] = fval;
            ++it[h];
            next = !(fval_perc[h] < (1.0 + tol_p) && fval_perc[h] > (1.0 - tol_p)) && it[h] < max_it;
          }
        }
        running[h] = next;
        hp[h].active = next;
        std::copy(&pose_x[16 * h], &pose_x[16 * h] + 16, hp[h].pose);
        any |= next;
      }
      if (any) {
        PEB_TRY(push_poses());
        // Src_Moved = PoseX * srcPCT for the poses that iterate again (a pose that stops does not use it any more)
        PEB_LAUNCH(ctx, cv_move, dim3(ceil_div(m, kCvT), H), kCvT, 0, d_pct, m, d_poses, d_moved);
      }
    }
    for (int h = 0; h < H; ++h) {
      mat44_mul(&pose_x[16 * h], &pose[16 * h], &pose[16 * h]);
      temp_res[h] = fval_min[h];
    }
  }
  PEB_CUDA(ctx, cudaStreamSynchronize(st));
  // ---- undo the normalisation, append to the input poses ----
  for (int h = 0; h < H; ++h) {
    double* P = &pose[16 * h];
    for (int r = 0; r < 3; ++r) {
      const double rm = P[4 * r] * hp[h].mean_avg[0] + P[4 * r + 1] * hp[h].mean_avg[1] + P[4 * r + 2] * hp[h].mean_avg[2];
      P[4 * r + 3] = P[4 * r + 3] / hp[h].scale + hp[h].mean_avg[r] - rm;
    }
    mat44_mul(P, poses + 16 * h, poses + 16 * h);
    if (residuals) residuals[h] = temp_res[h];
  }
  return PEB_OK;
}

}  // namespace peb
