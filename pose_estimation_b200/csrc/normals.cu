// normals.cu — pcl::NormalEstimation<PointXYZ, Normal>::computeFeature with setKSearch(k)
// ([PCL] features/impl/normal_3d.hpp, features/normal_3d.h, features/impl/feature.hpp;
//  SURVEY.md 8a-8) on the device.
//
// The k nearest neighbours (the point itself included, ascending squared distance, exactly
// what KdTreeFLANN::nearestKSearch returns) come from a uniform grid over the cloud whose cell
// edge is chosen so that the 3x3x3 block around a point usually already holds them.
//
// k <= 32 (normals_warp_kernel): a WARP per query, 32 consecutive queries of the cell-sorted cloud per warp.  The
// candidates of the 3 x 3 x 3 block are read 32 at a time (one per lane, consecutive lanes = consecutive points of a grid
// row), a chunk that holds anything better than the current k-th neighbour is sorted with a warp bitonic network
// (64-bit (distance, position) keys in registers, shuffles) and merged into the sorted list the warp keeps one entry
// per lane.  The covariance is then accumulated over the neighbours IN LIST ORDER, sequentially, in float, without
// FMA — PCL 1.10's single-pass computeMeanAndCovarianceMatrix: its nine sums are nine independent chains, one per
// lane, fed by broadcasting neighbour after neighbour.  The closed-form eigen33 (core_math.cuh) of the warp's 32
// queries finally runs one query per lane.  A query whose k-th neighbour is not proven by the 3 x 3 x 3 block (sparse
// borders) goes to a list that the general kernel below finishes.
// k > 32, or leftovers (normals_knn_kernel): one thread per query; its candidate list lives in shared memory, column
// per thread, kept sorted by insertion, rings until the bound proves the list.
// Algorithmic HBM bytes: N * (16 read + 16 k gather + 32 write).
//
// cv::ppf_match_3d::computeNormalsPC3d (cv_normals_*; DESIGN.md §13) runs the same grid and the same two searches and
// only swaps the tail: float products summed in double in list order, OpenCV's Jacobi eigen solver in double
// (core_math.cuh : cv_eigen_sym3), the last eigenvector rounded to float and the float viewpoint flip.
#include <algorithm>

#include "nn_graph.cuh"
#include "nn_search.cuh"

namespace peb {

namespace {

// The candidate list of one thread: k entries, ascending.  An entry is the 64-bit key
// (squared distance bits << 32) | sorted position: squared distances are non-negative floats, so the integer order of
// the keys is the list's order (smaller distance first, then smaller position) and one 64-bit compare / load / store
// does the work of two.
struct KnnList {
  unsigned long long* e;  // [k][T], this thread's column
  int stride;             // T
  int k;
  int count;
  unsigned long long worst;  // key of the last entry once the list is full
};

__device__ __forceinline__ unsigned long long knn_key(float d2, int j) {
  return (static_cast<unsigned long long>(__float_as_uint(d2)) << 32) | static_cast<unsigned>(j);
}
__device__ __forceinline__ int knn_key_pos(unsigned long long key) { return static_cast<int>(key & 0xFFFFFFFFull); }

__device__ __forceinline__ void knn_insert(KnnList& l, float d2, int j) {
  const unsigned long long key = knn_key(d2, j);
  if (l.count == l.k && !(key < l.worst)) return;
  int pos = (l.count < l.k) ? l.count : l.k - 1;
  while (pos > 0) {
    const unsigned long long prev = l.e[(pos - 1) * l.stride];
    if (prev > key) {
      l.e[pos * l.stride] = prev;
      --pos;
    } else {
      break;
    }
  }
  l.e[pos * l.stride] = key;
  if (l.count < l.k) ++l.count;
  if (l.count == l.k) l.worst = l.e[(l.k - 1) * l.stride];
}

__device__ __forceinline__ void knn_scan_range(const GridView& g, uint32_t s, uint32_t e, float qx, float qy, float qz,
                                               KnnList& l) {
  for (uint32_t j = s; j < e; ++j) {
    const float4 p = g.pts[j];
    const float d2 = l2_simple(qx, qy, qz, p.x, p.y, p.z);
    knn_insert(l, d2, static_cast<int>(j));
  }
}

__device__ __forceinline__ void knn_scan_ring(const GridView& g, float qx, float qy, float qz, int cx, int cy, int cz,
                                              int r, bool full, KnnList& l) {
  const int w = 2 * r + 1;
  const int x0 = max(cx - r, 0), x1 = min(cx + r, g.dx - 1);
  for (int row = 0; row < w * w; ++row) {
    const int oy = row % w - r, oz = row / w - r;
    const int y = cy + oy, z = cz + oz;
    if (y < 0 || y >= g.dy || z < 0 || z >= g.dz) continue;
    const long long base = (static_cast<long long>(z) * g.dy + y) * g.dx;
    const bool outer = full || oy == -r || oy == r || oz == -r || oz == r;
    if (outer) {
      knn_scan_range(g, g.cell_start[base + x0], g.cell_start[base + x1 + 1], qx, qy, qz, l);
    } else {
      if (cx - r >= 0) knn_scan_range(g, g.cell_start[base + cx - r], g.cell_start[base + cx - r + 1], qx, qy, qz, l);
      if (cx + r < g.dx) knn_scan_range(g, g.cell_start[base + cx + r], g.cell_start[base + cx + r + 1], qx, qy, qz, l);
    }
  }
}

__global__ void normals_fill_nan_kernel(float* __restrict__ out8, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float qnan = __int_as_float(0x7fc00000);
  float4* o = reinterpret_cast<float4*>(out8 + 8 * static_cast<size_t>(i));
  o[0] = make_float4(qnan, qnan, qnan, 0.0f);
  o[1] = make_float4(qnan, 0.0f, 0.0f, 0.0f);
}

// the min(k, g.n) nearest points of p into this thread's column of the shared-memory list, ascending (distance, position)
__device__ __forceinline__ void knn_list_search(const GridView& g, const float4& p, int k, unsigned long long* se, KnnList& l) {
  l.e = se + threadIdx.x;
  l.stride = blockDim.x;
  l.k = min(k, g.n);
  l.count = 0;
  l.worst = ~0ull;
  const int cx = grid_coord(p.x, g.ox, g.inv_h, g.dx);
  const int cy = grid_coord(p.y, g.oy, g.inv_h, g.dy);
  const int cz = grid_coord(p.z, g.oz, g.inv_h, g.dz);
  int r = 1;
  bool full = true;
  for (;;) {
    knn_scan_ring(g, p.x, p.y, p.z, cx, cy, cz, r, full, l);
    bool covers_all;
    const float b2 = grid_ring_bound2(g, p.x, p.y, p.z, cx, cy, cz, r, covers_all);
    if (covers_all || (l.count == l.k && __uint_as_float(static_cast<unsigned>(l.worst >> 32)) <= b2)) break;
    ++r;
    full = false;
  }
}

// list == nullptr: every sorted point is a query; else the queries are list[0 .. *list_n)
__global__ void normals_knn_kernel(const GridView g, int k, float vx, float vy, float vz, float* __restrict__ out8,
                                   int32_t* __restrict__ out_nn, const int* __restrict__ list,
                                   const int* __restrict__ list_n) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int T = blockDim.x;
  unsigned long long* se = reinterpret_cast<unsigned long long*>(smem_raw);
  int q = blockIdx.x * T + threadIdx.x;
  if (list) {
    if (q >= *list_n) return;
    q = list[q];
  }
  if (q >= g.n) return;
  const float4 p = g.pts[q];
  const int orig = __float_as_int(p.w);
  KnnList l;
  knn_list_search(g, p, k, se, l);
  float* o = out8 + 8 * static_cast<size_t>(orig);
  if (out_nn) {
    for (int i = 0; i < k; ++i)
      out_nn[static_cast<size_t>(orig) * k + i] = i < l.count ? __float_as_int(g.pts[knn_key_pos(l.e[i * T])].w) : -1;
  }
  if (l.count < 3) return;  // stays NaN ([PCL] normal_3d.h: computePointNormal fails below 3 points)
  float accu[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int i = 0; i < l.count; ++i) {
    const float4 c = g.pts[knn_key_pos(l.e[i * T])];
    accu[0] += c.x * c.x;
    accu[1] += c.x * c.y;
    accu[2] += c.x * c.z;
    accu[3] += c.y * c.y;
    accu[4] += c.y * c.z;
    accu[5] += c.z * c.z;
    accu[6] += c.x;
    accu[7] += c.y;
    accu[8] += c.z;
  }
  float res[8];
  normal_from_accu(accu, l.count, p.x, p.y, p.z, vx, vy, vz, res);
  reinterpret_cast<float4*>(o)[0] = make_float4(res[0], res[1], res[2], res[3]);
  reinterpret_cast<float4*>(o)[1] = make_float4(res[4], res[5], res[6], res[7]);
}

// ---- k <= 32: one thread per query, the candidate list in REGISTERS ----------------------------------------------
// K slots (d2, position), ascending.  An insertion is branch-free — every slot takes its left neighbour, the new
// candidate or itself (one compare + four selects per slot, all slots independent) — so the 32 queries of a warp, which
// are neighbours in the cell-sorted cloud and walk the same grid rows, stay in lock-step where the shared-memory
// insertion sort of the general kernel serialises their different shift lengths.  A list for k < K neighbours keeps
// K - k sentinels (d2 = -1, never displaced) in front, so that the k-th neighbour is always slot K - 1.
template <int K>
struct RegList {
  float d[K];
  int j[K];
};

// candidates arrive in ascending position (ring 1: rows in ascending (z, y), cells in ascending x), so a candidate that
// ties with a listed one has the larger position and goes behind it: strict < on the distance is the (d2, position) order
template <int K>
__device__ __forceinline__ void reglist_insert_ascending(RegList<K>& l, float x, int xj) {
  if (!(x < l.d[K - 1])) return;
#pragma unroll
  for (int i = K - 1; i >= 1; --i) {
    const bool shift = x < l.d[i - 1];
    const bool here = x < l.d[i];
    l.j[i] = shift ? l.j[i - 1] : (here ? xj : l.j[i]);
    l.d[i] = shift ? l.d[i - 1] : (here ? x : l.d[i]);
  }
  const bool here = x < l.d[0];
  l.j[0] = here ? xj : l.j[0];
  l.d[0] = here ? x : l.d[0];
}

// any arrival order (shells of ring >= 2): the full (d2, position) comparison
template <int K>
__device__ __forceinline__ void reglist_insert_any(RegList<K>& l, float x, int xj) {
  auto less = [](float a, int aj, float b, int bj) { return a < b || (a == b && static_cast<unsigned>(aj) < static_cast<unsigned>(bj)); };
  if (!less(x, xj, l.d[K - 1], l.j[K - 1])) return;
#pragma unroll
  for (int i = K - 1; i >= 1; --i) {
    const bool shift = less(x, xj, l.d[i - 1], l.j[i - 1]);
    const bool here = less(x, xj, l.d[i], l.j[i]);
    l.j[i] = shift ? l.j[i - 1] : (here ? xj : l.j[i]);
    l.d[i] = shift ? l.d[i - 1] : (here ? x : l.d[i]);
  }
  const bool here = less(x, xj, l.d[0], l.j[0]);
  l.j[0] = here ? xj : l.j[0];
  l.d[0] = here ? x : l.d[0];
}

template <int K, bool ASC>
__device__ __forceinline__ void reglist_scan_range(const GridView& g, uint32_t s, uint32_t e, float qx, float qy, float qz,
                                                   RegList<K>& l) {
  for (uint32_t j = s; j < e; ++j) {
    const float4 p = g.pts[j];
    const float d2 = l2_simple(qx, qy, qz, p.x, p.y, p.z);
    if (ASC) reglist_insert_ascending<K>(l, d2, static_cast<int>(j));
    else reglist_insert_any<K>(l, d2, static_cast<int>(j));
  }
}

// the kk nearest points of p (grid g, the point itself included if it is in g) in slots K - kk .. K - 1, ascending
// (distance, position); slots in front hold sentinels (j = -1)
template <int K>
__device__ __forceinline__ void reglist_knn(const GridView& g, const float4& p, int kk, RegList<K>& l) {
#pragma unroll
  for (int i = 0; i < K; ++i) {
    const bool sentinel = i < K - kk;
    l.d[i] = sentinel ? -1.0f : pos_inf();
    l.j[i] = -1;
  }
  const int cx = grid_coord(p.x, g.ox, g.inv_h, g.dx);
  const int cy = grid_coord(p.y, g.oy, g.inv_h, g.dy);
  const int cz = grid_coord(p.z, g.oz, g.inv_h, g.dz);
  {  // ring 1: the 3 x 3 x 3 block, rows in ascending position
    const int x0 = max(cx - 1, 0), x1 = min(cx + 1, g.dx - 1);
    for (int z = max(cz - 1, 0); z <= min(cz + 1, g.dz - 1); ++z)
      for (int y = max(cy - 1, 0); y <= min(cy + 1, g.dy - 1); ++y) {
        const long long base = (static_cast<long long>(z) * g.dy + y) * g.dx;
        reglist_scan_range<K, true>(g, g.cell_start[base + x0], g.cell_start[base + x1 + 1], p.x, p.y, p.z, l);
      }
  }
  for (int r = 1;; ++r) {
    bool covers_all;
    const float b2 = grid_ring_bound2(g, p.x, p.y, p.z, cx, cy, cz, r, covers_all);
    if (covers_all || (l.j[K - 1] >= 0 && l.d[K - 1] <= b2)) break;
    // the shell of ring r + 1 (sparse borders only)
    const int rr = r + 1, w = 2 * rr + 1;
    const int x0 = max(cx - rr, 0), x1 = min(cx + rr, g.dx - 1);
    for (int row = 0; row < w * w; ++row) {
      const int oy = row % w - rr, oz = row / w - rr;
      const int y = cy + oy, z = cz + oz;
      if (y < 0 || y >= g.dy || z < 0 || z >= g.dz) continue;
      const long long base = (static_cast<long long>(z) * g.dy + y) * g.dx;
      if (oy == -rr || oy == rr || oz == -rr || oz == rr) {
        reglist_scan_range<K, false>(g, g.cell_start[base + x0], g.cell_start[base + x1 + 1], p.x, p.y, p.z, l);
      } else {
        if (cx - rr >= 0) reglist_scan_range<K, false>(g, g.cell_start[base + cx - rr], g.cell_start[base + cx - rr + 1], p.x, p.y, p.z, l);
        if (cx + rr < g.dx) reglist_scan_range<K, false>(g, g.cell_start[base + cx + rr], g.cell_start[base + cx + rr + 1], p.x, p.y, p.z, l);
      }
    }
  }
}

template <int K>
__global__ void __launch_bounds__(128, 4) normals_reglist_kernel(const GridView g, int k, float vx, float vy, float vz,
                                                                 float* __restrict__ out8, int32_t* __restrict__ out_nn) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= g.n) return;
  const float4 p = g.pts[q];
  const int orig = __float_as_int(p.w);
  const int kk = min(k, g.n);  // neighbours wanted
  RegList<K> l;
  reglist_knn<K>(g, p, kk, l);
  // the neighbours in list order: slots K - kk .. K - 1 ([PCL] normal_3d.hpp: computePointNormal over nn_indices)
  int count = 0;
  float accu[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int s = 0; s < K; ++s) {
    if (l.j[s] >= 0) {
      const float4 c = g.pts[l.j[s]];
      if (out_nn) out_nn[static_cast<size_t>(orig) * k + (s - (K - kk))] = __float_as_int(c.w);
      accu[0] += c.x * c.x;
      accu[1] += c.x * c.y;
      accu[2] += c.x * c.z;
      accu[3] += c.y * c.y;
      accu[4] += c.y * c.z;
      accu[5] += c.z * c.z;
      accu[6] += c.x;
      accu[7] += c.y;
      accu[8] += c.z;
      ++count;
    }
  }
  if (count < 3) return;  // stays NaN ([PCL] normal_3d.h: computePointNormal fails below 3 points)
  float res[8];
  normal_from_accu(accu, count, p.x, p.y, p.z, vx, vy, vz, res);
  float4* o = reinterpret_cast<float4*>(out8 + 8 * static_cast<size_t>(orig));
  o[0] = make_float4(res[0], res[1], res[2], res[3]);
  o[1] = make_float4(res[4], res[5], res[6], res[7]);
}

template <int K>
int launch_reglist(peb_ctx* ctx, const GridView& g, int k, const float vp[3], float* d_out8, int32_t* d_out_nn) {
  PEB_LAUNCH(ctx, normals_reglist_kernel<K>, ceil_div(g.n, 128), 128, 0, g, k, vp[0], vp[1], vp[2], d_out8, d_out_nn);
  return PEB_OK;
}

// ---- cv::ppf_match_3d::computeNormalsPC3d (DESIGN.md §13): the same k-NN, OpenCV's tail -----------------------------
// Every row gets the input's xyz; a non-finite point (not in the grid) also gets a NaN normal.  The normal kernels
// below then write the normals of the finite points.
__global__ void __launch_bounds__(256) cv_normals_fill_kernel(const float4* __restrict__ in, int n, float* __restrict__ out6) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = in[i];
  float* o = out6 + 6 * static_cast<size_t>(i);
  o[0] = p.x;
  o[1] = p.y;
  o[2] = p.z;
  if (!finite3(p.x, p.y, p.z)) {
    const float qnan = __int_as_float(0x7fc00000);
    o[3] = o[4] = o[5] = qnan;
  }
}

struct CvNormalArgs {
  int k;      // neighbours; the launcher guarantees 1 <= k <= g.n
  int flip;   // flipNormalViewpoint
  float vx, vy, vz;
  float* out6;      // rows of x y z nx ny nz, by original index
  int32_t* out_nn;  // nullable, n x k original indices
};

__device__ __forceinline__ void cv_normal_store(const CvNormalArgs& a, const float4& p, int orig, const double (&acc)[9]) {
  float nrm[3];
  cv_normal_from_moments(acc, a.k, p.x, p.y, p.z, a.flip != 0, a.vx, a.vy, a.vz, nrm);
  float* o = a.out6 + 6 * static_cast<size_t>(orig);
  o[3] = nrm[0];
  o[4] = nrm[1];
  o[5] = nrm[2];
}

// k <= K <= 32: the register list of normals_reglist_kernel; the k neighbours are slots K - k .. K - 1, in list order
template <int K>
__global__ void __launch_bounds__(128, 4) cv_normals_reglist_kernel(const GridView g, const CvNormalArgs a) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= g.n) return;
  const float4 p = g.pts[q];
  const int orig = __float_as_int(p.w);
  RegList<K> l;
  reglist_knn<K>(g, p, a.k, l);
  double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
  for (int s = 0; s < K; ++s) {
    if (l.j[s] >= 0) {
      const float4 c = g.pts[l.j[s]];
      if (a.out_nn) a.out_nn[static_cast<size_t>(orig) * a.k + (s - (K - a.k))] = __float_as_int(c.w);
      cv_moments_add(acc, c.x, c.y, c.z);
    }
  }
  cv_normal_store(a, p, orig, acc);
}

// k > 32: the shared-memory list of normals_knn_kernel
__global__ void cv_normals_knn_kernel(const GridView g, const CvNormalArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int T = blockDim.x;
  const int q = blockIdx.x * T + threadIdx.x;
  if (q >= g.n) return;
  const float4 p = g.pts[q];
  const int orig = __float_as_int(p.w);
  KnnList l;
  knn_list_search(g, p, a.k, reinterpret_cast<unsigned long long*>(smem_raw), l);
  double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int i = 0; i < l.count; ++i) {
    const float4 c = g.pts[knn_key_pos(l.e[i * T])];
    if (a.out_nn) a.out_nn[static_cast<size_t>(orig) * a.k + i] = __float_as_int(c.w);
    cv_moments_add(acc, c.x, c.y, c.z);
  }
  cv_normal_store(a, p, orig, acc);
}

template <int K>
int launch_cv_reglist(peb_ctx* ctx, const GridView& g, const CvNormalArgs& a) {
  PEB_LAUNCH(ctx, cv_normals_reglist_kernel<K>, ceil_div(g.n, 128), 128, 0, g, a);
  return PEB_OK;
}

// The k-nearest-neighbour graph of a grid's own points (nn_graph.cuh): row(q) = the kGraphK nearest OTHER points of
// sorted position q, ascending (distance, position), in half rows of 12 with the distances from q to the neighbour
// behind every chunk of four.
constexpr int kGraphSlots = kGraphK + 2;  // the point itself + the row + the point behind the row
// writes row q; returns the row's outer bound (squared distance from q to neighbour kGraphK + 1; +inf: none)
__device__ __forceinline__ float knn_graph_row(const GridView& g, KnnRow* __restrict__ rows, int q) {
  const float4 p = g.pts[q];
  RegList<kGraphSlots> l;
  reglist_knn<kGraphSlots>(g, p, min(kGraphSlots, g.n), l);
  // the other points in list order: entry m of the row comes from the m-th slot that is filled and not q itself
  uint32_t pos[kGraphK + 1];
  float d2[kGraphK + 1];
#pragma unroll
  for (int t = 0; t <= kGraphK; ++t) {
    pos[t] = static_cast<uint32_t>(q);  // (a missing neighbour: the point itself, see nn_graph.cuh)
    d2[t] = pos_inf();
  }
  int m = 0;
#pragma unroll
  for (int s = 0; s < kGraphSlots; ++s) {
    if (l.j[s] >= 0 && l.j[s] != q) {
#pragma unroll
      for (int t = 0; t <= kGraphK; ++t)
        if (t == m) {
          pos[t] = static_cast<uint32_t>(l.j[s]);
          d2[t] = l.d[s];
        }
      ++m;
    }
  }
  uint4* u = reinterpret_cast<uint4*>(rows + q);
#pragma unroll
  for (int h = 0; h < kGraphHalves; ++h) {
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const int t = 12 * h + 4 * c;
      u[4 * h + c] = make_uint4(pos[t], pos[t + 1], pos[t + 2], pos[t + 3]);
    }
    reinterpret_cast<float4*>(u)[4 * h + 3] = make_float4(d2[12 * h + 4], d2[12 * h + 8], d2[12 * h + 12], 0.0f);
  }
  return d2[kGraphK];
}

__global__ void __launch_bounds__(128, 4) knn_graph_kernel(const GridView g, KnnRow* __restrict__ rows,
                                                           double* __restrict__ stat) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  // (no early return: the block sums its rows' outer bounds at the end)
  float outer = 0.0f;
  if (q < g.n) outer = knn_graph_row(g, rows, q);
  // sum and count of the finite outer bounds (icp.cu decides per hypothesis from their mean when the graph pays)
  float v = (outer > 0.0f && outer < pos_inf()) ? outer : 0.0f;
  float c = (outer > 0.0f && outer < pos_inf()) ? 1.0f : 0.0f;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    c += __shfl_xor_sync(0xFFFFFFFFu, c, o);
  }
  if ((threadIdx.x & 31) == 0 && c > 0.0f) {
    atomicAdd(stat, static_cast<double>(v));
    atomicAdd(stat + 1, static_cast<double>(c));
  }
}

// the flatness certificate's per-point record (nn_graph.cuh : knn_aux_of), one thread per target point
__global__ void __launch_bounds__(128) knn_aux_kernel(const GridView g, const KnnRow* __restrict__ rows, float4* __restrict__ aux) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < g.n) aux[j] = knn_aux_of(g, rows, j);
}

}  // namespace

// the graph of the target grid, built once per target and kept until the target changes (icp.cu asks for it)
int target_graph_ensure(peb_ctx* ctx) {
  if (ctx->tgt_knn_valid) return PEB_OK;
  const GridView& g = ctx->tgt_grid.view;
  PEB_CUDA(ctx, ctx->tgt_knn.ensure(std::max<size_t>(g.n, 1) * sizeof(KnnRow)));
  PEB_CUDA(ctx, ctx->tgt_knn_stat.ensure(2 * sizeof(double)));
  PEB_CUDA(ctx, cudaMemsetAsync(ctx->tgt_knn_stat.p, 0, 2 * sizeof(double), ctx->stream));
  if (g.n > 0)
    PEB_LAUNCH(ctx, knn_graph_kernel, ceil_div(g.n, 128), 128, 0, g, ctx->tgt_knn.as<KnnRow>(), ctx->tgt_knn_stat.as<double>());
  PEB_CUDA(ctx, ctx->tgt_knn_aux.ensure(std::max<size_t>(g.n, 1) * sizeof(float4)));
  if (g.n > 0)
    PEB_LAUNCH(ctx, knn_aux_kernel, ceil_div(g.n, 128), 128, 0, g, ctx->tgt_knn.as<KnnRow>(), ctx->tgt_knn_aux.as<float4>());
  ctx->tgt_knn_valid = true;
  return PEB_OK;
}

int normals_knn_device(peb_ctx* ctx, const float4* d_in, int n, int k, const float vp[3], float* d_out8,
                       int32_t* d_out_nn) {
  if (k < 1) return fail(ctx, PEB_E_INVALID_ARG, "normals_knn: k must be >= 1 (got %d)", k);
  if (k > 192) return fail(ctx, PEB_E_UNSUPPORTED, "normals_knn: k = %d > 192 has no CUDA path (no CPU fallback)", k);
  if (n == 0) return PEB_OK;
  PEB_LAUNCH(ctx, normals_fill_nan_kernel, ceil_div(n, 256), 256, 0, d_out8, n);
  if (d_out_nn) PEB_CUDA(ctx, cudaMemsetAsync(d_out_nn, 0xFF, static_cast<size_t>(n) * k * sizeof(int32_t), ctx->stream));
  // cell edge: the k-th neighbour of a surface point lies sqrt(k / (pi * occupancy)) cells away and the 3 x 3 x 3 block
  // proves everything within one cell of the query's own cell, so k / 2.4 points per occupied cell (0.87 cells) lets
  // ring 1 settle all but the border queries at ~9 * k / 2.4 candidates each
  const float occupancy = fmaxf(2.0f, static_cast<float>(k) / 2.4f);
  PEB_TRY(grid_build(ctx, &ctx->aux_grid, d_in, nullptr, n, occupancy));
  const GridView& g = ctx->aux_grid.view;
  if (g.n == 0) return PEB_OK;
  if (k <= 8) return launch_reglist<8>(ctx, g, k, vp, d_out8, d_out_nn);
  if (k <= 16) return launch_reglist<16>(ctx, g, k, vp, d_out8, d_out_nn);
  if (k <= 24) return launch_reglist<24>(ctx, g, k, vp, d_out8, d_out_nn);
  if (k <= 32) return launch_reglist<32>(ctx, g, k, vp, d_out8, d_out_nn);
  const int T = k <= 48 ? 128 : (k <= 96 ? 64 : 32);
  const size_t smem = static_cast<size_t>(k) * T * 8;
  PEB_LAUNCH(ctx, normals_knn_kernel, ceil_div(g.n, T), T, smem, g, k, vp[0], vp[1], vp[2], d_out8, d_out_nn,
             static_cast<const int*>(nullptr), static_cast<const int*>(nullptr));
  return PEB_OK;
}

int cv_normals_device(peb_ctx* ctx, const float4* d_in, int n, int k, bool flip, const float vp[3], float* d_out6,
                      int32_t* d_out_nn) {
  if (k < 1) return fail(ctx, PEB_E_INVALID_ARG, "cv_normals: k must be >= 1 (got %d)", k);
  if (k > 192) return fail(ctx, PEB_E_UNSUPPORTED, "cv_normals: k = %d > 192 has no CUDA path (no CPU fallback)", k);
  if (n == 0) return PEB_OK;
  // the grid and the cell edge of normals_knn_device: the search is the same
  const float occupancy = fmaxf(2.0f, static_cast<float>(k) / 2.4f);
  PEB_TRY(grid_build(ctx, &ctx->aux_grid, d_in, nullptr, n, occupancy));
  const GridView& g = ctx->aux_grid.view;
  if (k > g.n)
    return fail(ctx, PEB_E_INVALID_ARG, "cv_normals: k = %d exceeds the %d finite points of the cloud", k, g.n);
  PEB_LAUNCH(ctx, cv_normals_fill_kernel, ceil_div(n, 256), 256, 0, d_in, n, d_out6);
  if (d_out_nn) PEB_CUDA(ctx, cudaMemsetAsync(d_out_nn, 0xFF, static_cast<size_t>(n) * k * sizeof(int32_t), ctx->stream));
  const CvNormalArgs a{k, flip ? 1 : 0, vp[0], vp[1], vp[2], d_out6, d_out_nn};
  if (k <= 8) return launch_cv_reglist<8>(ctx, g, a);
  if (k <= 16) return launch_cv_reglist<16>(ctx, g, a);
  if (k <= 24) return launch_cv_reglist<24>(ctx, g, a);
  if (k <= 32) return launch_cv_reglist<32>(ctx, g, a);
  const int T = k <= 48 ? 128 : (k <= 96 ? 64 : 32);
  const size_t smem = static_cast<size_t>(k) * T * 8;
  PEB_LAUNCH(ctx, cv_normals_knn_kernel, ceil_div(g.n, T), T, smem, g, a);
  return PEB_OK;
}

}  // namespace peb
