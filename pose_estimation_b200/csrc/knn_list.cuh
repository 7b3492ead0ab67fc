// knn_list.cuh — the exact k-nearest-neighbour list searches over a uniform grid (device only): the shared-memory
// list of any length (knn_list_search) and the register list of K <= 32 slots (reglist_knn).  normals.cu builds the
// normals and the target graph on them, gicp.cu the per-point covariances of GeneralizedIterativeClosestPoint.
#pragma once

#include "nn_search.cuh"

namespace peb {

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

}  // namespace peb
