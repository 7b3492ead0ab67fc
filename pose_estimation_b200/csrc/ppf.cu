// ppf.cu — cv::ppf_match_3d::PPF3DDetector (trainModel / match) on the device: the coarse matcher that produces the
// hypotheses the refinement slot consumes (SURVEY.md 8f rank 4;
// pose_estimation/src/opencv_surface_match.cpp:37-51 trainModel, :65 match(pc, results, 1.0, 0.03)).
// [CV] opencv_contrib/modules/surface_matching/src/ppf_match_3d.cpp, ppf_helpers.cpp, pose_3d.cpp, c_utils.hpp —
// restated from recollection (the sources are in neither the reference tree nor this image), parity unpinned; the
// oracle (oracle/ppf_oracle.cpp) restates the same functions on the CPU and the tests compare the two.
//
//   sampling   samplePCByQuantization: cell key per point (upstream's float expression) -> stable radix sort ->
//              one warp per occupied cell adds the cell's points and normals SEQUENTIALLY in double in input order
//              (upstream's order; the loads of a chunk of 32 are parallel, the adds are not) -> lattice order
//   frames     computeTransformRT of every sampled point (the rotation that takes its normal onto x), once
//   training   every ordered pair of sampled model points: four-component feature, quantised -> a DIRECT-ADDRESS table
//              over the quantised feature (angle bins^3 x distance bins, < 1 M entries for the reference's
//              parameters) built by counting sort: count, scan, fill.  OpenCV's chained MurmurHash table is replaced
//              by the key itself: a scene pair votes for the model pairs with the same quantised feature and for no
//              hash-collision neighbours (pe_b200.h / DESIGN.md section 11: the one deliberate difference).
//   voting     one block per scene reference point.  Its accumulator (model reference x alpha bin) lives in SHARED
//              memory, a range of model reference points at a time: the pairs of a feature bin are stored sorted by
//              that range, so a pass walks exactly its own nodes.  Buckets are very uneven (on a smooth object a few
//              feature bins hold most pairs), so the (scene pair, model pair) items of a tile of 256 scene points are
//              FLATTENED — block scan of the bucket lengths, every thread takes items t, t + 256, ... and finds its
//              scene pair by binary search — which also makes the node loads coalesced.  Block argmax with upstream's
//              first-maximum rule.
//   poses      one thread per reference point: Tsg^-1 * Rx(alpha) * Tmg, Pose3D::updatePose (angle, quaternion), double
//   clustering PPF3DDetector::clusterPoses on the host: a greedy, order-dependent pass over at most a few thousand
//              poses (sorted by votes) — sequential by definition, microseconds of work.
// Double precision throughout the feature / alpha / pose arithmetic like upstream (Vec3d); sin / cos / acos / atan2 are
// CUDA's double functions (<= 2 ulp from glibc's): a feature within an ulp of a bin edge may quantise differently
// than on the CPU (tests/test_ppf.py counts such cases; none in the committed cases; tests/test_gpu_ppf_edges.py fails on
// any disagreement with the oracle that no quotient within 1e-12 of a bin edge explains).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>

#include "common.cuh"
#include "sort_scan.cuh"

struct peb_ppf_model {
  peb_ctx* ctx = nullptr;
  int device = 0;              // ctx's device, kept here: destroying the model never reads ctx (it may be gone already)
  peb_ppf_params prm{};
  double angle_step = 0.0;     // radians
  float distance_step = 0.0f;  // float like upstream
  double position_threshold = 0.0, rotation_threshold = 0.0;
  int num_angles = 0;          // alpha bins
  int n = 0;                   // sampled model points
  int na = 0, nd = 0;          // angle bins per component, distance bins
  int chunk = 0, ranges = 0;   // voting: model reference points per shared-memory pass, number of passes
  peb::DevBuf sampled;         // n x 6 float
  peb::DevBuf frames;          // n x 12 double (R row-major, t)
  peb::DevBuf bucket_start;    // (na^3 * nd) * ranges + 1: the pairs of a feature bin, by range of the model reference point
  peb::DevBuf nodes;           // uint2 (model reference, alpha bits) per stored pair
  peb::DevBuf rows;            // n_rows x 6 float: the rows trained on, resident for the cv ICP of peb_surface_match
  size_t n_rows = 0;
  std::vector<float> h_sampled;
};

namespace peb {
namespace {

constexpr double kPpfEps = 1.192092896e-07;  // [CV] c_utils.hpp : EPS
constexpr double kPi = 3.14159265358979323846;
constexpr size_t kVoteSmemBytes = 48 * 1024;  // shared-memory accumulator of the voting kernel (four blocks per SM)

// ---- sampling ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned f32_ordered(float f) {
  const unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ inline float f32_from_ordered(unsigned u) {
  const unsigned b = (u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u;
  float f;
#ifdef __CUDA_ARCH__
  f = __uint_as_float(b);
#else
  memcpy(&f, &b, 4);
#endif
  return f;
}

// [CV] computeBboxStd over the rows with finite coordinates: box[0..2] = min, box[3..5] = max (ordered-int encoding)
__global__ void ppf_bbox_kernel(const float* __restrict__ pc6, int n, unsigned* __restrict__ box) {
  unsigned lo[3] = {0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu}, hi[3] = {0u, 0u, 0u};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float x = pc6[6 * static_cast<size_t>(i)], y = pc6[6 * static_cast<size_t>(i) + 1], z = pc6[6 * static_cast<size_t>(i) + 2];
    if (!(isfinite(x) && isfinite(y) && isfinite(z))) continue;
    const unsigned e[3] = {f32_ordered(x), f32_ordered(y), f32_ordered(z)};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      lo[a] = min(lo[a], e[a]);
      hi[a] = max(hi[a], e[a]);
    }
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lo[a] = min(lo[a], __shfl_xor_sync(0xFFFFFFFFu, lo[a], o));
      hi[a] = max(hi[a], __shfl_xor_sync(0xFFFFFFFFu, hi[a], o));
    }
    if ((threadIdx.x & 31) == 0) {
      atomicMin(box + a, lo[a]);
      atomicMax(box + 3 + a, hi[a]);
    }
  }
}

struct SampleParams {
  float lo[3], range[3];
  int nsd;
  uint32_t sentinel;
};

// [CV] samplePCByQuantization: (int)((float)numSamplesDim * (p - lo) / range) per axis, index = x nsd^2 + y nsd + z
__global__ void ppf_cell_key_kernel(const float* __restrict__ pc6, int n, SampleParams sp, uint32_t* __restrict__ keys,
                                    uint32_t* __restrict__ vals) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float x = pc6[6 * static_cast<size_t>(i)], y = pc6[6 * static_cast<size_t>(i) + 1], z = pc6[6 * static_cast<size_t>(i) + 2];
  uint32_t key = sp.sentinel;
  if (isfinite(x) && isfinite(y) && isfinite(z)) {
    const float fn = static_cast<float>(sp.nsd);
    const int xc = static_cast<int>(fn * (x - sp.lo[0]) / sp.range[0]);
    const int yc = static_cast<int>(fn * (y - sp.lo[1]) / sp.range[1]);
    const int zc = static_cast<int>(fn * (z - sp.lo[2]) / sp.range[2]);
    const int index = xc * sp.nsd * sp.nsd + yc * sp.nsd + zc;
    key = (index >= 0 && static_cast<uint32_t>(index) < sp.sentinel) ? static_cast<uint32_t>(index) : sp.sentinel;
  }
  keys[i] = key;
  vals[i] = static_cast<uint32_t>(i);
}

__global__ void ppf_run_flag_kernel(const uint32_t* __restrict__ sorted_keys, int n, uint32_t sentinel, uint32_t* __restrict__ flags) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const uint32_t k = sorted_keys[j];
  flags[j] = (k != sentinel && (j == 0 || sorted_keys[j - 1] != k)) ? 1u : 0u;
}
__global__ void ppf_run_start_kernel(const uint32_t* __restrict__ flags, const uint32_t* __restrict__ slots, int n,
                                     uint32_t* __restrict__ run_start) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n && flags[j]) run_start[slots[j]] = static_cast<uint32_t>(j);
}

// one warp per occupied cell: chunks of 32 members are loaded in parallel and added one after the other (every lane
// keeps the same running sums), in sorted order = ascending input index (the sort is stable)
__global__ void __launch_bounds__(128) ppf_cell_mean_kernel(const float* __restrict__ pc6, const uint32_t* __restrict__ sorted_keys,
                                                            const uint32_t* __restrict__ sorted_vals, int n_sorted,
                                                            const uint32_t* __restrict__ run_start, int n_runs,
                                                            float* __restrict__ out6) {
  const int run = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (run >= n_runs) return;
  const uint32_t s = run_start[run];
  const uint32_t key = sorted_keys[s];
  double sum[6] = {0, 0, 0, 0, 0, 0};
  int cn = 0;
  for (uint32_t base = s;; base += 32) {
    const uint32_t j = base + lane;
    const bool mine = j < static_cast<uint32_t>(n_sorted) && sorted_keys[j] == key;
    float v[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (mine) {
      const float* p = pc6 + 6 * static_cast<size_t>(sorted_vals[j]);
#pragma unroll
      for (int a = 0; a < 6; ++a) v[a] = p[a];
    }
    const unsigned members = __ballot_sync(0xFFFFFFFFu, mine);  // a prefix of the lanes: the run is contiguous
    const int cnt = __popc(members);
    for (int l = 0; l < cnt; ++l) {
#pragma unroll
      for (int a = 0; a < 6; ++a) sum[a] += static_cast<double>(__shfl_sync(0xFFFFFFFFu, v[a], l));
    }
    cn += cnt;
    if (cnt < 32) break;
  }
  if (lane == 0) {
    const double dn = static_cast<double>(cn);
    const double px = sum[0] / dn, py = sum[1] / dn, pz = sum[2] / dn;
    const double nx = sum[3] / dn, ny = sum[4] / dn, nz = sum[5] / dn;
    float* o = out6 + 6 * static_cast<size_t>(run);
    o[0] = static_cast<float>(px);
    o[1] = static_cast<float>(py);
    o[2] = static_cast<float>(pz);
    const double nn = sqrt(nx * nx + ny * ny + nz * nz);
    const bool ok = nn > kPpfEps;
    o[3] = ok ? static_cast<float>(nx / nn) : 0.0f;
    o[4] = ok ? static_cast<float>(ny / nn) : 0.0f;
    o[5] = ok ? static_cast<float>(nz / nn) : 0.0f;
  }
}

// ---- frames, features ---------------------------------------------------------------------------------------------
struct D3 {
  double x, y, z;
};
__device__ __forceinline__ double dot3(const D3& a, const D3& b) { return a.x * b.x + a.y * b.y + a.z * b.z; }

// [CV] computeTransformRT + aaToR
__device__ void ppf_transform_rt(const D3& p1, const D3& n1, double* R, double* t) {
  const double angle = acos(n1.x);
  D3 axis = {0.0, n1.z, -n1.y};
  if (n1.y == 0.0 && n1.z == 0.0) {
    axis.y = 1.0;
    axis.z = 0.0;
  } else {
    const double nn = sqrt(dot3(axis, axis));
    if (nn > kPpfEps) {
      const double inv = 1.0 / nn;
      axis.x *= inv;
      axis.y *= inv;
      axis.z *= inv;
    }
  }
  const double c = cos(angle), s = sin(angle), omc = 1.0 - c;
  R[0] = c + omc * axis.x * axis.x;
  R[1] = omc * axis.x * axis.y - s * axis.z;
  R[2] = omc * axis.x * axis.z + s * axis.y;
  R[3] = omc * axis.y * axis.x + s * axis.z;
  R[4] = c + omc * axis.y * axis.y;
  R[5] = omc * axis.y * axis.z - s * axis.x;
  R[6] = omc * axis.z * axis.x - s * axis.y;
  R[7] = omc * axis.z * axis.y + s * axis.x;
  R[8] = c + omc * axis.z * axis.z;
  t[0] = -(R[0] * p1.x + R[1] * p1.y + R[2] * p1.z);
  t[1] = -(R[3] * p1.x + R[4] * p1.y + R[5] * p1.z);
  t[2] = -(R[6] * p1.x + R[7] * p1.y + R[8] * p1.z);
}

__global__ void ppf_frames_kernel(const float* __restrict__ pts6, int n, double* __restrict__ frames) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* p = pts6 + 6 * static_cast<size_t>(i);
  double R[9], t[3];
  ppf_transform_rt({p[0], p[1], p[2]}, {p[3], p[4], p[5]}, R, t);
  double* o = frames + 12 * static_cast<size_t>(i);
#pragma unroll
  for (int a = 0; a < 9; ++a) o[a] = R[a];
#pragma unroll
  for (int a = 0; a < 3; ++a) o[9 + a] = t[a];
}

// the planar angle of p2 in a frame ([CV] computeAlpha / the same lines of match())
__device__ __forceinline__ double ppf_alpha(const double* __restrict__ fr, const D3& p2) {
  const double my = fr[10] + (fr[3] * p2.x + fr[4] * p2.y + fr[5] * p2.z);
  const double mz = fr[11] + (fr[6] * p2.x + fr[7] * p2.y + fr[8] * p2.z);
  double alpha = atan2(-mz, my);
  if (alpha != alpha) return 0.0;
  if (sin(alpha) * mz < 0.0) alpha = -alpha;
  return -alpha;
}

struct KeySpace {
  double angle_step;
  double distance_step;  // (double)(float distance step), as upstream divides
  int na, nd;
};

// [CV] computePPFFeatures + the quantisation of hashPPF; -1: no bucket (NaN component or outside the model's table)
__device__ __forceinline__ int ppf_bucket(const float* __restrict__ a6, const float* __restrict__ b6, const KeySpace& ks) {
  const D3 p1 = {a6[0], a6[1], a6[2]}, n1 = {a6[3], a6[4], a6[5]};
  const D3 p2 = {b6[0], b6[1], b6[2]}, n2 = {b6[3], b6[4], b6[5]};
  double f0 = 0.0, f1 = 0.0, f2 = 0.0;
  D3 d = {p2.x - p1.x, p2.y - p1.y, p2.z - p1.z};
  const double f3 = sqrt(dot3(d, d));
  if (!(f3 <= kPpfEps)) {
    const double inv = 1.0 / f3;
    d.x *= inv;
    d.y *= inv;
    d.z *= inv;
    f0 = acos(dot3(n1, d));
    f1 = acos(dot3(n2, d));
    f2 = acos(dot3(n1, n2));
  }
  const double q0 = f0 / ks.angle_step, q1 = f1 / ks.angle_step, q2 = f2 / ks.angle_step, q3 = f3 / ks.distance_step;
  if (!(q0 == q0 && q1 == q1 && q2 == q2 && q3 == q3)) return -1;
  if (!(q0 < ks.na && q1 < ks.na && q2 < ks.na && q3 < ks.nd)) return -1;
  const int k0 = static_cast<int>(q0), k1 = static_cast<int>(q1), k2 = static_cast<int>(q2), k3 = static_cast<int>(q3);
  return ((k0 * ks.na + k1) * ks.na + k2) * ks.nd + k3;
}

// ---- training -----------------------------------------------------------------------------------------------------
// FILL = false: counts[bucket]++ ; FILL = true: nodes[cursor[bucket]++] = (i, alpha)
template <bool FILL>
__global__ void __launch_bounds__(256) ppf_train_pairs_kernel(const float* __restrict__ pts6, const double* __restrict__ frames,
                                                              int n, KeySpace ks, int chunk, int ranges,
                                                              uint32_t* __restrict__ counts_or_cursor, uint2* __restrict__ nodes) {
  const long long total = static_cast<long long>(n) * n;
  for (long long p = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; p < total;
       p += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int i = static_cast<int>(p / n), j = static_cast<int>(p - static_cast<long long>(i) * n);
    if (i == j) continue;
    const float* a6 = pts6 + 6 * static_cast<size_t>(i);
    const float* b6 = pts6 + 6 * static_cast<size_t>(j);
    int b = ppf_bucket(a6, b6, ks);
    if (b < 0) continue;
    b = b * ranges + i / chunk;
    if (!FILL) {
      atomicAdd(counts_or_cursor + b, 1u);
    } else {
      const float alpha = static_cast<float>(ppf_alpha(frames + 12 * static_cast<size_t>(i), {b6[0], b6[1], b6[2]}));
      const uint32_t pos = atomicAdd(counts_or_cursor + b, 1u);
      nodes[pos] = make_uint2(static_cast<uint32_t>(i), __float_as_uint(alpha));
    }
  }
}

// ---- voting -------------------------------------------------------------------------------------------------------
struct RefResult {
  uint32_t max_votes, ref_max, alpha_max, pad;
};

// (int)(num_angles * (alpha + 2 pi) / (4 pi)) like upstream.  The quotient by multiplication with 1 / (4 pi) is within
// 2 ulp of the division's: it decides the bin unless it lies that close to an integer, and only then is the division
// itself evaluated (out of line, so that its Newton sequence stays out of the voting loop).
__device__ __noinline__ double ppf_exact_quotient(double y) { return y / (4 * kPi); }
__device__ __forceinline__ int ppf_alpha_bin(double alpha, int num_angles) {
  const double y = num_angles * (alpha + 2 * kPi);
  double q = y * (1.0 / (4 * kPi));
  if (fabs(q - rint(q)) < 1e-9) q = ppf_exact_quotient(y);
  return static_cast<int>(q);
}

struct ScenePair {
  double alpha;  // alpha_scene
  int bucket;    // feature bin, -1: none
  int pad;
};

// dynamic shared memory: chunk * num_angles uint32 counters
__global__ void __launch_bounds__(256, 4) ppf_vote_kernel(const float* __restrict__ scene6, const double* __restrict__ scene_frames,
                                                       int m, int step, int n_ref, KeySpace ks,
                                                       const uint32_t* __restrict__ bucket_start, const uint2* __restrict__ nodes,
                                                       int n_model, int num_angles, int chunk, int ranges,
                                                       ScenePair* __restrict__ pair_scratch, RefResult* __restrict__ out) {
  extern __shared__ uint32_t s_acc[];
  __shared__ double s_fr[12];
  __shared__ float s_a6[6];
  __shared__ unsigned long long s_best[256 / 32];
  __shared__ uint32_t s_start[256], s_prefix[257];
  __shared__ double s_alpha[256];
  const int t = threadIdx.x;
  ScenePair* pairs = pair_scratch + static_cast<size_t>(blockIdx.x) * m;
  for (int ri = blockIdx.x; ri < n_ref; ri += gridDim.x) {
    const int i = ri * step;
    if (t < 12) s_fr[t] = scene_frames[12 * static_cast<size_t>(i) + t];
    if (t < 6) s_a6[t] = scene6[6 * static_cast<size_t>(i) + t];
    __syncthreads();
    // the feature bin and the planar angle of every scene pair (i, j), once
    for (int j = t; j < m; j += 256) {
      ScenePair sp;
      sp.bucket = -1;
      sp.alpha = 0.0;
      sp.pad = 0;
      if (j != i) {
        const float* b6 = scene6 + 6 * static_cast<size_t>(j);
        sp.bucket = ppf_bucket(s_a6, b6, ks);
        if (sp.bucket >= 0) sp.alpha = ppf_alpha(s_fr, {b6[0], b6[1], b6[2]});
      }
      pairs[j] = sp;
    }
    __syncthreads();
    unsigned long long best = 0xFFFFFFFFull;  // 0 votes at index 0
    for (int r = 0; r < ranges; ++r) {
      const int rows = min(chunk, n_model - r * chunk);
      const int bins = rows * num_angles;
      for (int a = t; a < bins; a += 256) s_acc[a] = 0u;
      __syncthreads();
      for (int j0 = 0; j0 < m; j0 += 256) {
        const int j = j0 + t;
        uint32_t start = 0, len = 0;
        double alpha_scene = 0.0;
        if (j < m) {
          const ScenePair sp = pairs[j];
          if (sp.bucket >= 0) {
            const size_t e = static_cast<size_t>(sp.bucket) * ranges + r;
            start = bucket_start[e];
            len = bucket_start[e + 1] - start;
            alpha_scene = sp.alpha;
          }
        }
        uint32_t total;
        const uint32_t before = block_exclusive_scan(len, &total);
        s_start[t] = start;
        s_prefix[t] = before;
        s_alpha[t] = alpha_scene;
        if (t == 255) s_prefix[256] = total;
        __syncthreads();
        // items [0, total): item `it` belongs to the scene pair p with prefix[p] <= it < prefix[p + 1].  A warp takes 32
        // consecutive items at a time, 256 items further every trip: the pair of its first item only moves forward
        // (one step per trip on average — buckets hold hundreds of pairs), every lane then steps on to its own pair
        int p0 = 0;
        for (uint32_t c0 = static_cast<uint32_t>(t & ~31); c0 < total; c0 += 256) {
          while (s_prefix[p0 + 1] <= c0) ++p0;  // (warp-uniform: broadcast reads)
          const uint32_t it = c0 + static_cast<uint32_t>(t & 31);
          if (it >= total) continue;
          int lo = p0;
          while (s_prefix[lo + 1] <= it) ++lo;
          const uint2 nd = nodes[s_start[lo] + (it - s_prefix[lo])];
          const double alpha = static_cast<double>(__uint_as_float(nd.y)) - s_alpha[lo];
          // (alpha == 2 pi exactly would index one past the row upstream: it goes to the last bin)
          const int alpha_index = min(ppf_alpha_bin(alpha, num_angles), num_angles - 1);
          atomicAdd(&s_acc[(static_cast<int>(nd.x) - r * chunk) * num_angles + alpha_index], 1u);
        }
        __syncthreads();
      }
      // [CV] "maximize the accumulator": strict >, scanning (k, j) upwards = the lowest index among the maxima; the
      // key (votes << 32 | ~index) makes that one 64-bit maximum
      const uint32_t base = static_cast<uint32_t>(r * chunk) * static_cast<uint32_t>(num_angles);
      for (int a = t; a < bins; a += 256) {
        const uint32_t v = s_acc[a];
        if (v) best = max(best, (static_cast<unsigned long long>(v) << 32) | (0xFFFFFFFFu - (base + static_cast<uint32_t>(a))));
      }
      __syncthreads();
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(0xFFFFFFFFu, best, o));
    if ((t & 31) == 0) s_best[t >> 5] = best;
    __syncthreads();
    if (t == 0) {
      for (int w = 1; w < 256 / 32; ++w) best = max(best, s_best[w]);
      const uint32_t idx = 0xFFFFFFFFu - static_cast<uint32_t>(best & 0xFFFFFFFFull);
      RefResult res;
      res.max_votes = static_cast<uint32_t>(best >> 32);
      res.ref_max = idx / static_cast<uint32_t>(num_angles);
      res.alpha_max = idx % static_cast<uint32_t>(num_angles);
      res.pad = 0;
      out[ri] = res;
    }
    __syncthreads();
  }
}

// ---- poses --------------------------------------------------------------------------------------------------------
__device__ void mat44_mul(const double* A, const double* B, double* C) {
  for (int r = 0; r < 4; ++r)
    for (int c = 0; c < 4; ++c) {
      double s = 0.0;
      for (int k = 0; k < 4; ++k) s += A[4 * r + k] * B[4 * k + c];
      C[4 * r + c] = s;
    }
}
__host__ __device__ inline void rt_to_pose(const double* R, const double* t, double* P) {
  for (int r = 0; r < 3; ++r) {
    for (int c = 0; c < 3; ++c) P[4 * r + c] = R[3 * r + c];
    P[4 * r + 3] = t[r];
  }
  P[12] = P[13] = P[14] = 0.0;
  P[15] = 1.0;
}
// [CV] dcmToQuat (w x y z), normalised
__host__ __device__ inline void dcm_to_quat(const double* R, double* q) {
  const double tr = R[0] + R[4] + R[8];
  if (tr > 0) {
    q[0] = tr + 1.0;
    q[1] = R[5] - R[7];
    q[2] = R[6] - R[2];
    q[3] = R[1] - R[3];
  } else {
    int i = 0;
    if (R[4] > R[0]) i = 1;
    if (R[8] > R[3 * i + i]) i = 2;
    const int j = (i + 1) % 3, k = (j + 1) % 3;
    q[i + 1] = R[3 * i + i] - R[3 * j + j] - R[3 * k + k] + 1.0;
    q[j + 1] = R[3 * i + j] + R[3 * j + i];
    q[k + 1] = R[3 * i + k] + R[3 * k + i];
    q[0] = R[3 * j + k] - R[3 * k + j];
  }
  const double nn = sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  const double s = 1.0 / nn;
  for (int a = 0; a < 4; ++a) q[a] *= s;
}
// [CV] Pose3D::updatePose: the rotation angle from the trace
__host__ __device__ inline double pose_angle(const double* R) {
  const double trace = R[0] + R[4] + R[8];
  if (fabs(trace - 3) <= kPpfEps) return 0.0;
  if (fabs(trace + 1) <= kPpfEps) return kPi;
  return acos((trace - 1) / 2);
}

__global__ void ppf_pose_kernel(const RefResult* __restrict__ refs, int n_ref, int step, const double* __restrict__ scene_frames,
                                const double* __restrict__ model_frames, int num_angles, peb_ppf_pose* __restrict__ out) {
  const int ri = blockIdx.x * blockDim.x + threadIdx.x;
  if (ri >= n_ref) return;
  const RefResult r = refs[ri];
  const double* sg = scene_frames + 12 * static_cast<size_t>(ri) * step;
  double RInv[9], tInv[3];
  for (int a = 0; a < 3; ++a)
    for (int b = 0; b < 3; ++b) RInv[3 * a + b] = sg[3 * b + a];
  for (int a = 0; a < 3; ++a) tInv[a] = -(RInv[3 * a] * sg[9] + RInv[3 * a + 1] * sg[10] + RInv[3 * a + 2] * sg[11]);
  double TsgInv[16], Tmg[16], Talpha[16], tmp[16], raw[16];
  rt_to_pose(RInv, tInv, TsgInv);
  const double* mg = model_frames + 12 * static_cast<size_t>(r.ref_max);
  rt_to_pose(mg, mg + 9, Tmg);
  const double alpha = (static_cast<int>(r.alpha_max) * (4 * kPi)) / num_angles - 2 * kPi;
  const double sa = sin(alpha), ca = cos(alpha);
  const double Rx[9] = {1, 0, 0, 0, ca, -sa, 0, sa, ca};  // [CV] getUnitXRotation
  const double tz[3] = {0, 0, 0};
  rt_to_pose(Rx, tz, Talpha);
  mat44_mul(Talpha, Tmg, tmp);
  mat44_mul(TsgInv, tmp, raw);
  peb_ppf_pose p;
  for (int a = 0; a < 16; ++a) p.pose[a] = raw[a];
  double R[9];
  for (int a = 0; a < 3; ++a)
    for (int b = 0; b < 3; ++b) R[3 * a + b] = raw[4 * a + b];
  p.t[0] = raw[3];
  p.t[1] = raw[7];
  p.t[2] = raw[11];
  p.angle = pose_angle(R);
  dcm_to_quat(R, p.q);
  p.alpha = alpha;
  p.residual = 0.0;
  p.num_votes = r.max_votes;
  p.model_index = r.ref_max;
  out[ri] = p;
}

// ---- host side ------------------------------------------------------------------------------------------------------
struct Sampled {
  int n = 0;
  float lo[3] = {0, 0, 0}, hi[3] = {0, 0, 0};
};

// the argument checks of ppf_sample, before anything is uploaded
int ppf_sample_check(peb_ctx* ctx, size_t n_in, float sample_step) {
  if (n_in == 0) return PEB_OK;
  if (n_in > static_cast<size_t>(INT32_MAX) / 8) return fail(ctx, PEB_E_INVALID_ARG, "ppf: too many points");
  if (!(sample_step > 0.0f) || !(sample_step <= 1.0f)) return fail(ctx, PEB_E_INVALID_ARG, "ppf: sampling step must be in (0, 1] (got %g)", sample_step);
  const int nsd = static_cast<int>(1.0 / sample_step);
  const long long cells = static_cast<long long>(nsd + 1) * (nsd + 1) * (nsd + 1);
  if (cells >= (1ll << 31)) return fail(ctx, PEB_E_UNSUPPORTED, "ppf: sampling step %g gives %lld lattice cells", sample_step, cells);
  return PEB_OK;
}

// samplePCByQuantization of a DEVICE cloud (n x 6 floats, read only): the sampled rows land in `out` (device), lattice
// order.  `out` must not alias d_in.
int ppf_sample_device(peb_ctx* ctx, const float* d_in, size_t n_in, float sample_step, DevBuf* out, Sampled* info) {
  info->n = 0;
  PEB_TRY(ppf_sample_check(ctx, n_in, sample_step));
  if (n_in == 0) return PEB_OK;
  const int n = static_cast<int>(n_in);
  const int nsd = static_cast<int>(1.0 / sample_step);
  const long long cells = static_cast<long long>(nsd + 1) * (nsd + 1) * (nsd + 1);
  PEB_CUDA(ctx, ctx->d_small.ensure(256));
  PEB_CUDA(ctx, ctx->h_small.ensure(256));
  unsigned* d_box = ctx->d_small.as<unsigned>();
  unsigned* h_box = ctx->h_small.as<unsigned>();
  PEB_CUDA(ctx, cudaMemsetAsync(d_box, 0xFF, 12, ctx->stream));
  PEB_CUDA(ctx, cudaMemsetAsync(d_box + 3, 0x00, 12, ctx->stream));
  PEB_LAUNCH(ctx, ppf_bbox_kernel, std::min(ceil_div(n, 256), kSmCount * 4), 256, 0, d_in, n, d_box);
  PEB_CUDA(ctx, cudaMemcpyAsync(h_box, d_box, 24, cudaMemcpyDeviceToHost, ctx->stream));
  PEB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (h_box[0] == 0xFFFFFFFFu) return PEB_OK;  // no finite point
  SampleParams sp;
  for (int a = 0; a < 3; ++a) {
    info->lo[a] = f32_from_ordered(h_box[a]);
    info->hi[a] = f32_from_ordered(h_box[3 + a]);
    sp.lo[a] = info->lo[a];
    sp.range[a] = info->hi[a] - info->lo[a];
  }
  sp.nsd = nsd;
  sp.sentinel = static_cast<uint32_t>(cells);
  int key_bits = 1;
  while ((1ll << key_bits) <= cells) ++key_bits;
  Grid& g = ctx->aux_grid;  // its sort buffers
  PEB_CUDA(ctx, g.keys.ensure(static_cast<size_t>(n) * 4));
  PEB_CUDA(ctx, g.vals.ensure(static_cast<size_t>(n) * 4));
  PEB_CUDA(ctx, g.keys_tmp.ensure(static_cast<size_t>(n) * 4));
  PEB_CUDA(ctx, g.vals_tmp.ensure(static_cast<size_t>(n) * 4));
  PEB_LAUNCH(ctx, ppf_cell_key_kernel, ceil_div(n, 256), 256, 0, d_in, n, sp, g.keys.as<uint32_t>(), g.vals.as<uint32_t>());
  uint32_t *sk = nullptr, *sv = nullptr;
  PEB_TRY(sort_pairs(ctx, g.keys.as<uint32_t>(), g.vals.as<uint32_t>(), g.keys_tmp.as<uint32_t>(), g.vals_tmp.as<uint32_t>(), n,
                     key_bits, &sk, &sv));
  // run heads -> their compacted order
  PEB_CUDA(ctx, ctx->vg_flags.ensure(static_cast<size_t>(n) * 4));
  PEB_CUDA(ctx, ctx->vg_scan.ensure(static_cast<size_t>(n) * 4 + 4));
  PEB_CUDA(ctx, ctx->vg_starts.ensure(static_cast<size_t>(n) * 4));
  uint32_t* flags = ctx->vg_flags.as<uint32_t>();
  uint32_t* slots = ctx->vg_scan.as<uint32_t>();
  uint32_t* d_total = slots + n;
  PEB_LAUNCH(ctx, ppf_run_flag_kernel, ceil_div(n, 256), 256, 0, sk, n, sp.sentinel, flags);
  PEB_TRY(exclusive_scan_u32(ctx, flags, slots, n, d_total));
  PEB_LAUNCH(ctx, ppf_run_start_kernel, ceil_div(n, 256), 256, 0, flags, slots, n, ctx->vg_starts.as<uint32_t>());
  uint32_t* h_total = ctx->h_small.as<uint32_t>() + 16;
  PEB_CUDA(ctx, cudaMemcpyAsync(h_total, d_total, 4, cudaMemcpyDeviceToHost, ctx->stream));
  PEB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  const int n_runs = static_cast<int>(*h_total);
  info->n = n_runs;
  if (n_runs == 0) return PEB_OK;
  PEB_CUDA(ctx, out->ensure(static_cast<size_t>(n_runs) * 24));
  PEB_LAUNCH(ctx, ppf_cell_mean_kernel, ceil_div(static_cast<long long>(n_runs) * 32, 128), 128, 0, d_in, sk, sv, n,
             ctx->vg_starts.as<uint32_t>(), n_runs, out->as<float>());
  return PEB_OK;
}

// the same for a host cloud: uploaded to `staging` (ctx->d_stage for a scene, the model's own rows for training) first
int ppf_sample(peb_ctx* ctx, const float* h_pc6, size_t n_in, float sample_step, DevBuf* staging, DevBuf* out, Sampled* info) {
  info->n = 0;
  PEB_TRY(ppf_sample_check(ctx, n_in, sample_step));
  if (n_in == 0) return PEB_OK;
  PEB_CUDA(ctx, staging->ensure(n_in * 24));
  PEB_CUDA(ctx, cudaMemcpyAsync(staging->p, h_pc6, n_in * 24, cudaMemcpyHostToDevice, ctx->stream));
  return ppf_sample_device(ctx, staging->as<float>(), n_in, sample_step, out, info);
}

// [CV] Pose3D::updatePoseQuat
void update_pose_quat(peb_ppf_pose& p, const double q[4], const double t[3]) {
  const double sqw = q[0] * q[0], sqx = q[1] * q[1], sqy = q[2] * q[2], sqz = q[3] * q[3];
  double R[9];
  R[0] = sqx - sqy - sqz + sqw;
  R[4] = -sqx + sqy - sqz + sqw;
  R[8] = -sqx - sqy + sqz + sqw;
  double t1 = q[1] * q[2], t2 = q[3] * q[0];
  R[3] = 2.0 * (t1 + t2);
  R[1] = 2.0 * (t1 - t2);
  t1 = q[1] * q[3];
  t2 = q[2] * q[0];
  R[6] = 2.0 * (t1 - t2);
  R[2] = 2.0 * (t1 + t2);
  t1 = q[2] * q[3];
  t2 = q[1] * q[0];
  R[7] = 2.0 * (t1 + t2);
  R[5] = 2.0 * (t1 - t2);
  for (int a = 0; a < 4; ++a) p.q[a] = q[a];
  for (int a = 0; a < 3; ++a) p.t[a] = t[a];
  rt_to_pose(R, t, p.pose);
  p.angle = pose_angle(R);
}

// [CV] PPF3DDetector::clusterPoses (+ matchPose).  Ties of the two sorts keep their input order (std::sort upstream
// leaves them unspecified).
void cluster_poses(const peb_ppf_model& m, std::vector<peb_ppf_pose> poses, std::vector<peb_ppf_pose>& out) {
  std::stable_sort(poses.begin(), poses.end(), [](const peb_ppf_pose& a, const peb_ppf_pose& b) { return a.num_votes > b.num_votes; });
  struct Cluster {
    std::vector<int> members;
    uint64_t votes = 0;
  };
  std::vector<Cluster> clusters;
  for (size_t i = 0; i < poses.size(); ++i) {
    bool assigned = false;
    for (size_t c = 0; c < clusters.size() && !assigned; ++c) {
      const peb_ppf_pose& centre = poses[static_cast<size_t>(clusters[c].members[0])];
      const double dx = centre.t[0] - poses[i].t[0], dy = centre.t[1] - poses[i].t[1], dz = centre.t[2] - poses[i].t[2];
      const double dn = std::sqrt(dx * dx + dy * dy + dz * dz);
      const double phi = std::fabs(poses[i].angle - centre.angle);
      if (phi < m.rotation_threshold && dn < m.position_threshold) {
        clusters[c].members.push_back(static_cast<int>(i));
        clusters[c].votes += poses[i].num_votes;
        assigned = true;
      }
    }
    if (!assigned) {
      Cluster c;
      c.members.push_back(static_cast<int>(i));
      c.votes = poses[i].num_votes;
      clusters.push_back(c);
    }
  }
  std::stable_sort(clusters.begin(), clusters.end(), [](const Cluster& a, const Cluster& b) { return a.votes > b.votes; });
  out.clear();
  for (const Cluster& c : clusters) {
    double q[4] = {0, 0, 0, 0}, t[3] = {0, 0, 0};
    const int sz = static_cast<int>(c.members.size());
    double wsum = 0;
    for (int mi : c.members) {
      const peb_ppf_pose& p = poses[static_cast<size_t>(mi)];
      const double w = m.prm.use_weighted_avg ? static_cast<double>(p.num_votes) : 1.0;
      if (m.prm.use_weighted_avg) {
        for (int a = 0; a < 4; ++a) q[a] += w * p.q[a];
        for (int a = 0; a < 3; ++a) t[a] += w * p.t[a];
      } else {
        for (int a = 0; a < 4; ++a) q[a] += p.q[a];
        for (int a = 0; a < 3; ++a) t[a] += p.t[a];
      }
      wsum += w;
    }
    const double inv = m.prm.use_weighted_avg ? 1.0 / wsum : 1.0 / sz;
    for (int a = 0; a < 3; ++a) t[a] *= inv;
    for (int a = 0; a < 4; ++a) q[a] *= inv;
    peb_ppf_pose r = poses[static_cast<size_t>(c.members[0])];
    update_pose_quat(r, q, t);
    r.num_votes = c.votes;
    out.push_back(r);
  }
}

struct DeviceScope {
  int prev = -1;
  explicit DeviceScope(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceScope() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

int train_impl(peb_ctx* ctx, const float* model6, size_t n_model, const peb_ppf_params* prm, peb_ppf_model** out) {
  if (!ctx || !out) return PEB_E_INVALID_ARG;
  *out = nullptr;
  if (!prm || !model6) return fail(ctx, PEB_E_INVALID_ARG, "ppf_train: null model / params");
  if (!(prm->num_angles >= 1.0) || !(prm->relative_sampling_step > 0.0))
    return fail(ctx, PEB_E_INVALID_ARG, "ppf_train: num_angles %g / sampling step %g", prm->num_angles, prm->relative_sampling_step);
  DeviceScope scope(ctx->device);
  peb_ppf_model* m = new peb_ppf_model();
  struct Drop {
    peb_ppf_model* m;
    ~Drop() {
      if (m) peb_ppf_model_destroy(m);
    }
  } drop{m};
  m->ctx = ctx;
  m->device = ctx->device;
  m->prm = *prm;
  // [CV] PPF3DDetector::PPF3DDetector / setSearchParams
  m->angle_step = (360.0 / prm->num_angles) * kPi / 180.0;
  m->position_threshold = prm->position_threshold < 0 ? prm->relative_sampling_step : prm->position_threshold;
  m->rotation_threshold = prm->rotation_threshold < 0 ? ((360 / m->angle_step) / 180.0 * kPi) : prm->rotation_threshold;
  m->num_angles = static_cast<int>(std::floor(2 * kPi / m->angle_step));
  Sampled info;
  // the rows stay on the device with the model: peb_surface_match refines against them without another upload
  PEB_TRY(ppf_sample(ctx, model6, n_model, static_cast<float>(prm->relative_sampling_step), &m->rows, &m->sampled, &info));
  m->n_rows = n_model;
  if (info.n < 2) return fail(ctx, PEB_E_INVALID_ARG, "ppf_train: the model samples to %d points", info.n);
  // (a voting tile flattens the buckets of 256 scene pairs into one 32-bit item range: 256 n^2 must stay below 2^32)
  if (info.n > 4095) return fail(ctx, PEB_E_UNSUPPORTED, "ppf_train: %d sampled model points (at most 4095)", info.n);
  m->n = info.n;
  const float dx = info.hi[0] - info.lo[0], dy = info.hi[1] - info.lo[1], dz = info.hi[2] - info.lo[2];
  const float diameter = std::sqrt(dx * dx + dy * dy + dz * dz);
  m->distance_step = static_cast<float>(diameter * prm->relative_sampling_step);
  if (!(m->distance_step > 0.0f)) return fail(ctx, PEB_E_INVALID_ARG, "ppf_train: degenerate model (diameter %g)", diameter);
  // the key space: angles in [0, pi], distances up to the diameter (+ 1 bin of slack each)
  m->na = static_cast<int>(kPi / m->angle_step) + 2;
  m->nd = static_cast<int>(static_cast<double>(diameter) / static_cast<double>(m->distance_step)) + 2;
  const long long entries = static_cast<long long>(m->na) * m->na * m->na * m->nd;
  if (entries > (64ll << 20)) return fail(ctx, PEB_E_UNSUPPORTED, "ppf_train: %lld feature bins (num_angles %g) exceed the direct table", entries, prm->num_angles);
  const KeySpace ks = {m->angle_step, static_cast<double>(m->distance_step), m->na, m->nd};
  // voting keeps the accumulator rows of `chunk` model reference points in shared memory (kVoteSmemBytes)
  m->chunk = std::max(1, static_cast<int>(kVoteSmemBytes / (static_cast<size_t>(m->num_angles) * 4)));
  m->ranges = ceil_div(m->n, m->chunk);
  if (entries * m->ranges > (256ll << 20)) return fail(ctx, PEB_E_UNSUPPORTED, "ppf_train: feature table of %lld x %d entries", entries, m->ranges);
  PEB_CUDA(ctx, m->frames.ensure(static_cast<size_t>(m->n) * 12 * sizeof(double)));
  PEB_LAUNCH(ctx, ppf_frames_kernel, ceil_div(m->n, 128), 128, 0, m->sampled.as<float>(), m->n, m->frames.as<double>());
  const int E = static_cast<int>(entries * m->ranges);
  PEB_CUDA(ctx, m->bucket_start.ensure((static_cast<size_t>(E) + 1) * 4));
  DevBuf cursor;
  struct Free {
    DevBuf* b;
    ~Free() { b->release(); }
  } free_cursor{&cursor};
  PEB_CUDA(ctx, cursor.ensure((static_cast<size_t>(E) + 1) * 4));
  PEB_CUDA(ctx, cudaMemsetAsync(cursor.p, 0, (static_cast<size_t>(E) + 1) * 4, ctx->stream));
  const long long pairs = static_cast<long long>(m->n) * m->n;
  const int blocks = static_cast<int>(std::min<long long>((pairs + 255) / 256, kSmCount * 16));
  PEB_LAUNCH(ctx, ppf_train_pairs_kernel<false>, blocks, 256, 0, m->sampled.as<float>(), m->frames.as<double>(), m->n, ks,
             m->chunk, m->ranges, cursor.as<uint32_t>(), static_cast<uint2*>(nullptr));
  PEB_TRY(exclusive_scan_u32(ctx, cursor.as<uint32_t>(), m->bucket_start.as<uint32_t>(), E + 1, nullptr));
  PEB_CUDA(ctx, cudaMemcpyAsync(cursor.p, m->bucket_start.p, (static_cast<size_t>(E) + 1) * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  PEB_CUDA(ctx, m->nodes.ensure(static_cast<size_t>(pairs) * sizeof(uint2)));
  PEB_LAUNCH(ctx, ppf_train_pairs_kernel<true>, blocks, 256, 0, m->sampled.as<float>(), m->frames.as<double>(), m->n, ks,
             m->chunk, m->ranges, cursor.as<uint32_t>(), m->nodes.as<uint2>());
  m->h_sampled.resize(static_cast<size_t>(m->n) * 6);
  PEB_CUDA(ctx, cudaMemcpyAsync(m->h_sampled.data(), m->sampled.p, m->h_sampled.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
  PEB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  drop.m = nullptr;
  *out = m;
  return PEB_OK;
}

// the checks of peb_ppf_match that do not depend on where the scene is
int match_check(peb_ctx* ctx, const peb_ppf_model* m, double rel_sample_step) {
  if (m->ctx != ctx) return fail(ctx, PEB_E_INVALID_ARG, "ppf_match: the model was trained on another context");
  if (!(rel_sample_step > 0.0) || !(rel_sample_step <= 1.0))
    return fail(ctx, PEB_E_INVALID_ARG, "ppf_match: relative scene sample step must be in (0, 1] (got %g)", rel_sample_step);
  return PEB_OK;
}

// match over a scene that is already sampled into ctx->nrm_in (info from ppf_sample*): raw poses in reference order, then
// clustered.  Uses nrm_out (scene frames) and cv_arena.
int match_sampled(peb_ctx* ctx, const peb_ppf_model* m, const Sampled& info, double rel_sample_step,
                  std::vector<peb_ppf_pose>& h_raw, std::vector<peb_ppf_pose>& clustered) {
  h_raw.clear();
  clustered.clear();
  const int step = static_cast<int>(1.0 / rel_sample_step);
  DevBuf& scene = ctx->nrm_in;       // sampled scene rows
  DevBuf& frames = ctx->nrm_out;     // their frames
  const int ms = info.n;
  if (ms == 0) return PEB_OK;
  const int n_ref = (ms + step - 1) / step;
  PEB_CUDA(ctx, frames.ensure(static_cast<size_t>(ms) * 12 * sizeof(double)));
  PEB_LAUNCH(ctx, ppf_frames_kernel, ceil_div(ms, 128), 128, 0, scene.as<float>(), ms, frames.as<double>());
  const KeySpace ks = {m->angle_step, static_cast<double>(m->distance_step), m->na, m->nd};
  const int blocks = std::min(n_ref, kSmCount * 4);
  const size_t pair_bytes = static_cast<size_t>(blocks) * ms * sizeof(ScenePair);
  const size_t ref_bytes = static_cast<size_t>(n_ref) * sizeof(RefResult);
  const size_t pose_bytes = static_cast<size_t>(n_ref) * sizeof(peb_ppf_pose);
  PEB_CUDA(ctx, ctx->cv_arena.ensure(pair_bytes + ref_bytes + pose_bytes + 512));
  unsigned char* base = ctx->cv_arena.as<unsigned char>();
  ScenePair* pair_scratch = reinterpret_cast<ScenePair*>(base);
  RefResult* refs = reinterpret_cast<RefResult*>(base + ((pair_bytes + 255) / 256) * 256);
  peb_ppf_pose* d_poses = reinterpret_cast<peb_ppf_pose*>(reinterpret_cast<unsigned char*>(refs) + ((ref_bytes + 255) / 256) * 256);
  const size_t smem = static_cast<size_t>(std::min(m->chunk, m->n)) * m->num_angles * 4;
  PEB_CUDA(ctx, cudaFuncSetAttribute(ppf_vote_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(kVoteSmemBytes)));
  PEB_LAUNCH(ctx, ppf_vote_kernel, blocks, 256, smem, scene.as<float>(), frames.as<double>(), ms, step, n_ref, ks,
             m->bucket_start.as<uint32_t>(), m->nodes.as<uint2>(), m->n, m->num_angles, m->chunk, m->ranges, pair_scratch, refs);
  PEB_LAUNCH(ctx, ppf_pose_kernel, ceil_div(n_ref, 128), 128, 0, refs, n_ref, step, frames.as<double>(), m->frames.as<double>(),
             m->num_angles, d_poses);
  h_raw.resize(static_cast<size_t>(n_ref));
  PEB_CUDA(ctx, cudaMemcpyAsync(h_raw.data(), d_poses, pose_bytes, cudaMemcpyDeviceToHost, ctx->stream));
  PEB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  cluster_poses(*m, h_raw, clustered);
  return PEB_OK;
}

int match_impl(peb_ctx* ctx, const peb_ppf_model* m, const float* scene6, size_t n_scene, double rel_sample_step,
               double rel_distance, peb_ppf_pose* results, size_t cap, size_t* out_n, peb_ppf_pose* raw, size_t cap_raw,
               size_t* out_n_raw) {
  if (!ctx) return PEB_E_INVALID_ARG;
  if (out_n) *out_n = 0;
  if (out_n_raw) *out_n_raw = 0;
  if (!m || !scene6) return fail(ctx, PEB_E_INVALID_ARG, "ppf_match: null model / scene");
  PEB_TRY(match_check(ctx, m, rel_sample_step));
  DeviceScope scope(ctx->device);
  Sampled info;
  PEB_TRY(ppf_sample(ctx, scene6, n_scene, static_cast<float>(rel_distance), &ctx->d_stage, &ctx->nrm_in, &info));
  std::vector<peb_ppf_pose> h_raw, clustered;
  PEB_TRY(match_sampled(ctx, m, info, rel_sample_step, h_raw, clustered));
  if (out_n_raw) *out_n_raw = h_raw.size();
  if (raw) std::memcpy(raw, h_raw.data(), std::min(cap_raw, h_raw.size()) * sizeof(peb_ppf_pose));
  if (out_n) *out_n = clustered.size();
  if (results) std::memcpy(results, clustered.data(), std::min(cap, clustered.size()) * sizeof(peb_ppf_pose));
  return PEB_OK;
}

template <typename Fn>
int guarded(peb_ctx* ctx, const char* what, Fn fn) noexcept {
  int code = PEB_E_CUDA;
  const char* why = "unexpected C++ exception";
  try {
    return fn();
  } catch (const std::bad_alloc&) {
    code = PEB_E_OOM;
    why = "out of host memory";
  } catch (...) {
  }
  try {
    if (ctx) ctx->err = std::string(what) + ": " + why;
  } catch (...) {
  }
  return code;
}

}  // namespace

// peb_ppf_match over a DEVICE scene (n x 6 floats, not written; must not be ctx->nrm_in / nrm_out / cv_arena / d_stage):
// the clustered poses, most votes first.  Same checks (after the null ones) and bytes as the host entry point.
int ppf_match_device(peb_ctx* ctx, const peb_ppf_model* m, const float* d_scene6, size_t n_scene, double rel_sample_step,
                     double rel_distance, std::vector<peb_ppf_pose>& clustered) {
  clustered.clear();
  PEB_TRY(match_check(ctx, m, rel_sample_step));
  DeviceScope scope(ctx->device);
  Sampled info;
  PEB_TRY(ppf_sample_device(ctx, d_scene6, n_scene, static_cast<float>(rel_distance), &ctx->nrm_in, &info));
  std::vector<peb_ppf_pose> h_raw;
  return match_sampled(ctx, m, info, rel_sample_step, h_raw, clustered);
}

peb_ctx* ppf_model_ctx(const peb_ppf_model* m) { return m->ctx; }

const float* ppf_model_rows(const peb_ppf_model* m, size_t* n_rows) {
  *n_rows = m->n_rows;
  return m->rows.as<float>();
}

// [CV] Pose3D::appendPose, given the appended pose (icp_pose * pose): pose, then q, angle and t recomputed from it
void ppf_set_appended_pose(peb_ppf_pose& p, const double* pose16) {
  for (int a = 0; a < 16; ++a) p.pose[a] = pose16[a];
  double R[9];
  for (int a = 0; a < 3; ++a)
    for (int b = 0; b < 3; ++b) R[3 * a + b] = pose16[4 * a + b];
  dcm_to_quat(R, p.q);
  p.angle = pose_angle(R);
  p.t[0] = pose16[3];
  p.t[1] = pose16[7];
  p.t[2] = pose16[11];
}

}  // namespace peb

extern "C" {

PEB_API void peb_ppf_params_default(peb_ppf_params* p) {
  if (!p) return;
  p->relative_sampling_step = 0.03;
  p->relative_distance_step = 0.03;
  p->num_angles = 40.0;
  p->position_threshold = -1.0;
  p->rotation_threshold = -1.0;
  p->use_weighted_avg = 0;
  p->reserved = 0;
}

PEB_API int peb_ppf_train(peb_ctx* ctx, const float* model_xyzn, size_t n_model, const peb_ppf_params* params, peb_ppf_model** out) {
  return peb::guarded(ctx, "peb_ppf_train", [&]() { return peb::train_impl(ctx, model_xyzn, n_model, params, out); });
}

PEB_API void peb_ppf_model_destroy(peb_ppf_model* m) {
  if (!m) return;
  {
    peb::DeviceScope scope(m->device);
    m->sampled.release();
    m->frames.release();
    m->bucket_start.release();
    m->nodes.release();
    m->rows.release();
  }
  delete m;
}

PEB_API int peb_ppf_model_sampled(const peb_ppf_model* m, float* out6, size_t cap, size_t* out_n) {
  if (!m) return PEB_E_INVALID_ARG;
  if (out_n) *out_n = static_cast<size_t>(m->n);
  if (out6) std::memcpy(out6, m->h_sampled.data(), std::min(cap, static_cast<size_t>(m->n)) * 24);
  return PEB_OK;
}

PEB_API int peb_ppf_match(peb_ctx* ctx, const peb_ppf_model* m, const float* scene_xyzn, size_t n_scene,
                          double relative_scene_sample_step, double relative_scene_distance, peb_ppf_pose* results, size_t cap,
                          size_t* out_n, peb_ppf_pose* raw, size_t cap_raw, size_t* out_n_raw) {
  return peb::guarded(ctx, "peb_ppf_match", [&]() {
    return peb::match_impl(ctx, m, scene_xyzn, n_scene, relative_scene_sample_step, relative_scene_distance, results, cap, out_n,
                           raw, cap_raw, out_n_raw);
  });
}

}  // extern "C"
