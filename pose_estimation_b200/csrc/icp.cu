// icp.cu — pcl::IterativeClosestPoint / IterativeClosestPointWithNormals on the device.
//
// One launch per ICP iteration, no host round trip inside an align (SURVEY.md H4):
//
//   icp_iteration_kernel   grid = (blocks_per_hypothesis, H)
//     every query:  working point <- increment of the previous iteration * working point
//                   ([PCL] registration/impl/icp.hpp : transformCloud, in place, float)
//                   exact 1-NN over the uniform grid (nn_search.cuh)
//                   [PCL] registration/impl/correspondence_estimation.hpp : determineCorrespondences
//                   (d2 > max_dist^2 rejected) and correspondence_rejection_distance.cpp (keep iff <)
//                   moments of the estimator accumulated in double
//     every block:  warp shuffle -> shared memory -> one partial record in global memory
//     last block :  (atomic ticket) sums the partial records in block order — deterministic —
//                   and runs the solve + convergence criteria in double (core_math.cuh),
//                   leaving the increment and the state for the next launch.
//   icp_fitness_kernel     [PCL] registration/impl/registration.hpp : getFitnessScore, then packs
//                   the peb_icp_result record.
//
// Launch 0 of an align searches cold: ring search, G lanes per query (far queries touch hundreds
// of grid rows, the lanes of a group split them).  Every later launch is warm: one thread per
// query, seeded with the previous iteration's match, which travels in the .w slot of the working
// point (nn grid_nn_warm: only the cells inside the ball of that candidate's distance).
// Later launches of an align that has already converged return at once (state.active == 0).
// The batched mode is the same code with H > 1: one working cloud per hypothesis so that PCL's
// incremental float update is reproduced exactly for every hypothesis.
#include <algorithm>

#include "block_select.cuh"
#include "nn_cache.cuh"
#include "nn_graph.cuh"
#include "nn_search.cuh"
#include "nn_upfront.cuh"

namespace peb {

namespace {

constexpr int kIcpThreads = 128;
// Register caps (measured on B200, bench C4 / C2): a single align is latency-bound per launch and
// wants no spills (5 blocks/SM = 96 registers); the batched mode is throughput-bound and gains 17 %
// from 8 blocks/SM (64 registers, a few spills to L1) through the extra warps that hide L2 latency.
constexpr int kMinBlocksSingle = 5;
#ifndef PEB_MIN_BLOCKS_BATCH
#define PEB_MIN_BLOCKS_BATCH 8
#endif
constexpr int kMinBlocksBatch = PEB_MIN_BLOCKS_BATCH;  // (development: -DPEB_MIN_BLOCKS_BATCH=n builds a variant library, PEB_LIB_VARIANT)
// The search launch of a split iteration (icp_search_kernel) holds no moments and no solve: without a cap it needs 82
// registers, so its cap is chosen on its own (measured, profiles/README.md).
#ifndef PEB_MIN_BLOCKS_SEARCH
#define PEB_MIN_BLOCKS_SEARCH 10
#endif
constexpr int kMinBlocksSearch = PEB_MIN_BLOCKS_SEARCH;

struct IcpLaunch {
  GridView grid;
  const float4* src;     // n_src FINITE source points in patch order, .w = original index
  float4* work;          // H x n_src working clouds (same order); .w = sorted position of the last match
  float* slack;          // H x n_src: how far the point may still move before its match must be searched again
  const int* anchors;    // nullable, H x n_anchor: match (sorted position) of the first point of every 32-point patch
  int n_anchor;
  float seed_guard2;     // (cells)^2: an anchor farther than this from the query is not used as a seed
  int coop_max_rows;     // first iteration: patches verify their candidates together while the common region has at most this many grid rows (0: never)
  unsigned long long* dbg;  // nullable: 8 timestamps (ns, %globaltimer) per launch, written by the last block
  int launch_idx;
  IcpState* states;      // H
  double* partials;      // H x part_stride x kAccMax
  int part_stride;       // block records per hypothesis: the same for every launch of an align (the cold and the warm
                         // launches may use different blocks_per_hyp, and chains / launch dependencies let them overlap)
  int32_t* corr_idx;     // nullable, indexed by ORIGINAL source index (single align only)
  float* corr_d2;        // nullable
  Mat4* trace;           // nullable, trace_cap increments (single align only)
  peb_icp_result* results;  // H (fitness kernel)
  IcpCriteria crit;
  double max_dist_sqr;
  double fitness_max_range;
  float stop_d2;         // NN search may stop once every unexamined point is farther than this
  float fitness_stop_d2;
  float rej_max2;
  int use_rejector;
  int n_src;
  int blocks_per_hyp;
  int trace_cap;
  int fitness_only;      // peb_fitness_score: the record's n_correspondences carries the inlier count
  int warm;              // seed every search with the match stored in the working point's .w
  int* epochs;           // nullable, H: solved iterations per hypothesis, published after the state is complete
  int* err_flag;         // raised if a dependency wait runs into its bound
  float margin;          // extra search radius that buys the skip-the-search certificate (0: none)
  NnCache* cache;        // nullable, H x n_src candidate caches (nn_cache.cuh) of the cached warm launches
  float cache_r_cells;   // radius (cells) a cache entry's collecting search covers
  int cache_init;        // this launch is the first cached one: every entry is still garbage
  const KnnRow* knn;     // nullable: the target's k-NN graph (nn_graph.cuh) for the warm searches
  const double* knn_stat;  // [0] sum, [1] count of the finite outer bounds (next2[2]) of the graph's rows
  float knn_kappa;       // a hypothesis searches over the graph once 4 * (its last MSE) * kappa < the mean outer bound
  int cold_graph;        // launch 0: candidates by greedy descent on the graph instead of the 3 x 3 x 3 probe
  int knn_peek_until;    // graph launches up to this one look at the four nearest neighbours of the previous match before a walk
  const float4* knn_aux; // nullable: the flatness certificate's per-point records (nn_graph.cuh : knn_aux_of)
};

__global__ void icp_init_kernel(IcpState* __restrict__ states, const float* __restrict__ guesses, int H,
                                int* __restrict__ epochs) {
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  if (epochs && h <= H) epochs[h] = 0;  // (entry H is the error flag)
  if (h >= H) return;
  IcpState st;
  st.inc = mat4_identity();
  if (guesses) {
#pragma unroll
    for (int i = 0; i < 16; ++i) st.final_t.m[i] = guesses[16 * h + i];
  } else {
    st.final_t = mat4_identity();
  }
  st.prev_mse = DBL_MAX;
  st.cur_mse = DBL_MAX;
  st.fit_sum = 0.0;
  st.iterations = 0;
  st.state = PEB_NOT_CONVERGED;
  st.converged = 0;
  st.similar = 0;
  st.ncorr = 0;
  st.active = 1;
  st.fit_n = 0;
  st.pad0 = 0;
  st.ticket = 0;
  st.ticket_fit = 0;
  st.ticket_search = 0;
  st.searched = 0;
  states[h] = st;
}

// sums NACC doubles over the block; the result is valid in threads [0, NACC) of warp 0
template <int NACC>
__device__ __forceinline__ double block_reduce_acc(double (&acc)[NACC], double (*sm)[kAccMax]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < NACC; ++i) {
    double v = acc[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
    if (lane == 0) sm[warp][i] = v;
  }
  __syncthreads();
  double r = 0.0;
  if (threadIdx.x < NACC) {
#pragma unroll
    for (int w = 0; w < kIcpThreads / 32; ++w) r += sm[w][threadIdx.x];
  }
  return r;
}

// the last block of a hypothesis sums the per-block records in block order (fixed order => the
// double sums do not depend on scheduling); result in sm_out[0..NACC)
template <int NACC>
__device__ __forceinline__ void reduce_partials(const double* __restrict__ part, int n_blocks, double (*sm)[kAccMax],
                                                double* sm_out) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  constexpr int kW = kIcpThreads / 32;
  double v = 0.0;
  if (lane < NACC) {
    // warp w owns the contiguous block range [b0, b1); sixteen independent loads in flight per lane
    // (the L2 round trip, not the adds, is what this loop waits for); the order of the adds is fixed
    const int per = (n_blocks + kW - 1) / kW;
    const int b0 = warp * per, b1 = min(b0 + per, n_blocks);
    const double* p = part + lane;
    int b = b0;
    for (; b + 16 <= b1; b += 16) {
      double t[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) t[k] = __ldcg(p + static_cast<size_t>(b + k) * kAccMax);
#pragma unroll
      for (int k = 0; k < 16; ++k) v += t[k];
    }
    for (; b < b1; ++b) v += __ldcg(p + static_cast<size_t>(b) * kAccMax);
    sm[warp][lane] = v;
  }
  __syncthreads();
  if (threadIdx.x < NACC) {
    double r = 0.0;
#pragma unroll
    for (int w = 0; w < kW; ++w) r += sm[w][threadIdx.x];
    sm_out[threadIdx.x] = r;
  }
  __syncthreads();
}

// Iteration 0 has no previous match to start from.  The source is stored in compact 32-point
// patches (common.cuh), so one cold ring search per patch — this kernel, one thread per patch and
// hypothesis, all lanes busy — gives every point of the patch a nearby seed; the iteration kernel
// then runs grid_nn_seeded for all points instead of 32 divergent ring searches per warp.
__global__ void __launch_bounds__(128) icp_anchor_kernel(const IcpLaunch L, int* __restrict__ anchors) {
  const int a = blockIdx.x * blockDim.x + threadIdx.x;
  const int h = blockIdx.y;
  if (a >= L.n_anchor) return;
  const IcpState* st = L.states + h;
  float T[16];
  bool apply = false;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    T[i] = __ldcg(&st->final_t.m[i]);
    if (T[i] != ((i % 5 == 0) ? 1.0f : 0.0f)) apply = true;
  }
  float4 p = L.src[32 * a];
  if (apply) {
    float ox, oy, oz;
    transform_icp(T, p.x, p.y, p.z, ox, oy, oz);
    p.x = ox;
    p.y = oy;
    p.z = oz;
  }
  // a seed only (every candidate derived from it is verified later): the first ring that holds a point is enough
  const NnBest best = grid_nn<1, true>(L.grid, p.x, p.y, p.z, L.stop_d2);
  anchors[static_cast<size_t>(h) * L.n_anchor + a] = best.j;
}

__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// The solve runs once per launch in one thread; keeping it out of line keeps its registers and
// local arrays out of the per-query loop's allocation.
// (templated on the register cap of the calling kernel so that the single-align copy is not
//  squeezed into the batched kernels' 64 registers)
template <int MB>
__device__ __noinline__ void finish_iteration(IcpState* st, const IcpCriteria* cr, const double* acc, Mat4* trace,
                                              int trace_cap, unsigned long long* dbg) {
  if (dbg) dbg[5] = global_ns();
  IcpState s = *st;
  if (dbg) dbg[6] = global_ns() + (s.iterations < -5 ? 1 : 0);
  icp_finish_iteration(s, *cr, acc);
  if (dbg) dbg[7] = global_ns() + (s.iterations < -5 ? 1 : 0);
  s.ticket = 0;
  if (trace && s.state != PEB_NO_CORRESPONDENCES && s.iterations >= 1 && s.iterations <= trace_cap)
    trace[s.iterations - 1] = s.inc;
  *st = s;
}

// PDL (common.cuh : PEB_LAUNCH_PDL): let the next launch of the stream be scheduled now, then wait
// until everything the previous launch wrote is complete and visible.
__device__ __forceinline__ void pdl_trigger_and_wait() {
  asm volatile("griddepcontrol.launch_dependents;");
  asm volatile("griddepcontrol.wait;" ::: "memory");
}

__device__ __forceinline__ int ld_acquire_gpu(const int* p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}


// A hypothesis that has stopped iterating (converged, iteration cap, too few correspondences) publishes this instead
// of + 1, so that everything that may still wait for it is released by the SAME release / acquire pair that makes
// its final state visible (looking at IcpState::active instead would race with the state's other fields).
constexpr int kEpochStopped = 1 << 20;
constexpr unsigned long long kFlagWaitLimitNs = 20ull * 1000ull * 1000ull * 1000ull;  // a dependency that never comes is a bug: give up after 20 s
// Waits (thread 0, then the block) until `need` iterations of the hypothesis have been solved and published, or the
// hypothesis has stopped.  See icp_iteration_kernel for why this cannot deadlock.
__device__ __forceinline__ void wait_for_hypothesis(const int* __restrict__ solved, int need, int* err_flag) {
  if (threadIdx.x == 0 && ld_acquire_gpu(solved) < need) {
    const unsigned long long t0 = global_ns();
    unsigned spins = 0;
    while (ld_acquire_gpu(solved) < need) {
      __nanosleep(40);
      if ((++spins & 0xFFFu) == 0u && global_ns() - t0 > kFlagWaitLimitNs) {
        atomicExch(err_flag, 1);
        break;
      }
    }
  }
  __syncthreads();
}

// Waits (thread 0, then the block) until `need` search launches of the hypothesis have completed (a split iteration's
// moment launch, icp_moment_kernel) or the hypothesis has stopped (its epoch carries kEpochStopped; its later search launches
// count nothing).  Bounded like wait_for_hypothesis.
__device__ __forceinline__ void wait_for_search(const int* __restrict__ searched, int need, const int* __restrict__ solved,
                                                int* err_flag) {
  if (threadIdx.x == 0 && ld_acquire_gpu(searched) < need && ld_acquire_gpu(solved) < kEpochStopped) {
    const unsigned long long t0 = global_ns();
    unsigned spins = 0;
    while (ld_acquire_gpu(searched) < need && ld_acquire_gpu(solved) < kEpochStopped) {
      __nanosleep(40);
      if ((++spins & 0xFFFu) == 0u && global_ns() - t0 > kFlagWaitLimitNs) {
        atomicExch(err_flag, 1);
        break;
      }
    }
  }
  __syncthreads();
}

// Does hypothesis `st` search over the target's k-NN graph in this launch?  The graph pays once the matches are close
// enough for its certificate (4 d^2 < the row's outer bound): while the hypothesis is still millimetres off, every query
// would scan its row in vain and walk the grid afterwards.  The mean squared distance of the last iteration's
// correspondences predicts this iteration's d^2; the choice only moves time (both searches are exact), so a coarse
// predictor is enough.  kappa = 0: always.
__device__ __forceinline__ bool graph_pays(const IcpLaunch& L, const IcpState* st) {
  if (!L.knn) return false;
  if (L.knn_kappa <= 0.0f) return true;
  const double mse = __ldcg(&st->cur_mse);
  const double cnt = __ldcg(L.knn_stat + 1);
  return cnt > 0.0 && 4.0 * mse * static_cast<double>(L.knn_kappa) * cnt < __ldcg(L.knn_stat);
}

// adds one accepted correspondence (working point p, match t = the target's point j, squared distance d2) to the
// estimator's moment sums
template <int EST, int NACC>
__device__ __forceinline__ void add_moments(const GridView& g, const float4& p, const float4& t, int j, float d2,
                                            double (&acc)[NACC]) {
  if (EST == PEB_ESTIMATOR_SVD) {
    const double sx = p.x, sy = p.y, sz = p.z, tx = t.x, ty = t.y, tz = t.z;
    acc[0] += 1.0;
    acc[1] += sx;
    acc[2] += sy;
    acc[3] += sz;
    acc[4] += tx;
    acc[5] += ty;
    acc[6] += tz;
    // (the product of two widened floats is exact in double, so the fused form rounds exactly like multiply-then-add:
    //  one DFMA instead of DMUL + DADD under -fmad=false, bit-identical sums)
    acc[7] = fma(tx, sx, acc[7]);
    acc[8] = fma(tx, sy, acc[8]);
    acc[9] = fma(tx, sz, acc[9]);
    acc[10] = fma(ty, sx, acc[10]);
    acc[11] = fma(ty, sy, acc[11]);
    acc[12] = fma(ty, sz, acc[12]);
    acc[13] = fma(tz, sx, acc[13]);
    acc[14] = fma(tz, sy, acc[14]);
    acc[15] = fma(tz, sz, acc[15]);
    acc[16] += static_cast<double>(d2);
  } else {
    acc[0] += 1.0;
    acc[NACC - 1] += static_cast<double>(d2);
    const float4 nr = g.normals[j];
    // [PCL] transformation_estimation_point_to_plane_lls.hpp: pairs with a non-finite
    // member are left out of the normal equations (they still count as correspondences)
    if (finite3(t.x, t.y, t.z) && finite3(nr.x, nr.y, nr.z)) {
      const float sx = p.x, sy = p.y, sz = p.z, dx = t.x, dy = t.y, dz = t.z;
      const float nx = nr.x, ny = nr.y, nz = nr.z;
      const double a = nz * sy - ny * sz;  // float expressions, widened afterwards
      const double b = nx * sz - nz * sx;
      const double c = ny * sx - nx * sy;
      acc[1] += a * a;
      acc[2] += a * b;
      acc[3] += a * c;
      acc[4] += a * nx;
      acc[5] += a * ny;
      acc[6] += a * nz;
      acc[7] += b * b;
      acc[8] += b * c;
      acc[9] += b * nx;
      acc[10] += b * ny;
      acc[11] += b * nz;
      acc[12] += c * c;
      acc[13] += c * nx;
      acc[14] += c * ny;
      acc[15] += c * nz;
      acc[16] += nx * nx;  // float products
      acc[17] += nx * ny;
      acc[18] += nx * nz;
      acc[19] += ny * ny;
      acc[20] += ny * nz;
      acc[21] += nz * nz;
      const double d = nx * dx + ny * dy + nz * dz - nx * sx - ny * sy - nz * sz;
      acc[22] += a * d;
      acc[23] += b * d;
      acc[24] += c * d;
      acc[25] += nx * d;
      acc[26] += ny * d;
      acc[27] += nz * d;
    }
  }
}
// adds one accepted correspondence (working point p, match best) to the estimator's moment sums
template <int EST, int NACC>
__device__ __forceinline__ void accumulate_pair(const GridView& g, const float4& p, const NnBest& best,
                                                double (&acc)[NACC]) {
  static_assert((EST == PEB_ESTIMATOR_SVD && NACC == kAccSvd) || (EST != PEB_ESTIMATOR_SVD && NACC == kAccLls), "layout");
  const float4 t = g.pts[best.j];
  add_moments<EST, NACC>(g, p, t, best.j, best.d2, acc);
}

// First-iteration search of the 32 queries of a warp (one source patch), all lanes together.  A query
// gets its candidate from its patch's anchor (icp_anchor_kernel); the candidates are then verified by
// the warp as a whole (nn_search.cuh : grid_nn_coop_verify) or, for spread-out patches, one by one.
// Queries without a usable seed search cold.
__device__ __forceinline__ NnBest first_iteration_search(const IcpLaunch& L, int h, int i, bool valid, const float4& p,
                                                         const float* T, bool apply, CoopTile* tile) {
  NnBest best;
  best.d2 = pos_inf();
  best.idx = -1;
  best.j = -1;
  bool need = false;  // holds a candidate that is not verified yet
  int group = 0;      // 0: seeded by the own anchor, 1: by the next patch's (the two places are verified separately)
  if (valid) {
    // Seed: the match of this patch's anchor (its first point).  A patch is 32 consecutive points of
    // the cell-sorted source, so it may hold points from two places (the end of one run of cells and
    // the start of the next); the tail of such a patch continues into the NEXT patch, whose anchor is
    // then the nearby one.  A seed farther than seed_guard cells would only blow the ball up.
    int j_seed = -1;
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    group = 0;
    const int patch = i >> 5;
#pragma unroll 1
    for (int k = 0; k < 2 && j_seed < 0; ++k) {
      const int pa = patch + k;
      if (pa >= L.n_anchor) break;
      const int js = __ldcg(L.anchors + static_cast<size_t>(h) * L.n_anchor + pa);
      if (js < 0) continue;
      // the anchor query, recomputed (same arithmetic as the caller's): where the seed was found from
      a = L.src[32 * pa];
      if (apply) {
        float ox, oy, oz;
        transform_icp(T, a.x, a.y, a.z, ox, oy, oz);
        a.x = ox;
        a.y = oy;
        a.z = oz;
      }
      const float ax = p.x - a.x, ay = p.y - a.y, az = p.z - a.z;
      if (ax * ax + ay * ay + az * az <= L.seed_guard2 * L.grid.h * L.grid.h) {
        j_seed = js;
        group = k;
      }
    }
    if (j_seed >= 0) {
      // the candidate: greedy descent on the target's k-NN graph from the anchor's match ("cold_graph"), or the best of
      // the 3 x 3 x 3 block around the anchor's match shifted by (q - q_anchor)
      best = (L.knn && L.cold_graph) ? grid_nn_graph_descend(L.grid, L.knn, p.x, p.y, p.z, j_seed)
                                     : grid_nn_seed_probe(L.grid, p.x, p.y, p.z, j_seed, a.x, a.y, a.z);
      need = true;
    } else {
      best = grid_nn<1>(L.grid, p.x, p.y, p.z, L.stop_d2);
      PEB_COOP_COUNT_LANE(6);
    }
  }
  PEB_COOP_COUNT(7, __any_sync(0xFFFFFFFFu, valid && !need) ? 1 : 0);
#pragma unroll 1
  for (int k = 0; k < 2; ++k) {
    const bool mine = need && group == k;
    bool done = false;
    if (L.coop_max_rows > 0) done = grid_nn_coop_verify(L.grid, tile, mine, p.x, p.y, p.z, L.stop_d2, L.coop_max_rows, best);
    if (!done && mine) grid_ball_search(L.grid, p.x, p.y, p.z, L.stop_d2, best);
  }
  return best;
}

// One query of one ICP iteration: working point i of hypothesis h is moved by T (the previous
// increment, or the guess in the first iteration), its exact nearest neighbour is searched (seeded
// by its previous match when there is one), the correspondence is thresholded and added to the
// estimator's moment sums.  Shared by the per-iteration kernel and the work-queue kernel.
// UPF: the warm search fetches all row bounds of its ball up front (nn_upfront.cuh; experimental, off by default):
// 0 = off, 2 / 3 = balls whose box spans up to 2 x 2 / 3 x 3 grid rows take that path; 4 = the search over the target's
// k-NN graph (nn_graph.cuh; L.knn)
template <int G, int EST, bool CERT, int UPF, int NACC>
__device__ __forceinline__ void icp_query(const IcpLaunch& L, const int h, float4* __restrict__ work, const int i,
                                          const bool first, const bool apply, const bool graph, const float* T,
                                          CoopTile* tile, double (&acc)[NACC]) {
  const int lane_in_group = threadIdx.x & (G - 1);
  const bool in = i < L.n_src;
  float4 p = make_float4(0.f, 0.f, 0.f, 1.f);
  if (in) p = first ? L.src[i] : work[i];
  const int j_prev = first ? -1 : __float_as_int(p.w);  // last iteration's match (sorted position)
  const bool valid = in && finite3(p.x, p.y, p.z);
  float moved = 0.0f;
  if (valid && apply) {
    float ox, oy, oz;
    transform_icp(T, p.x, p.y, p.z, ox, oy, oz);
    if (CERT) {
      const float mx = ox - p.x, my = oy - p.y, mz = oz - p.z;
      moved = sqrtf(mx * mx + my * my + mz * mz);
    }
    p.x = ox;
    p.y = oy;
    p.z = oz;
  }
  // queries of a group run the search together; invalid ones idle through it
  NnBest best;
  best.d2 = pos_inf();
  best.idx = -1;
  best.j = -1;
  float slack = -1.0f;
  if (G == 1 && first && L.anchors) {
    // (uniform branch: every lane of the warp takes part, valid or not)
    best = first_iteration_search(L, h, i, valid, p, T, apply, tile);
    if (CERT && valid) L.slack[static_cast<size_t>(h) * L.n_src + i] = -1.0f;
  } else if (valid) {
    float* sl = L.slack + static_cast<size_t>(h) * L.n_src + i;
    if (G == 1 && L.warm && j_prev >= 0 && j_prev < L.grid.n) {
      if (CERT) {
        // certificate of the previous search (core_math.cuh : grid_nn_warm_cert): every other
        // target point was at least `slack` farther than the match; the point has moved by `moved`
        slack = *sl - 2.000002f * moved - 1e-5f * L.grid.h;
        if (slack > 0.0f) {
          const float4 t = L.grid.pts[j_prev];
          best.d2 = l2_simple(p.x, p.y, p.z, t.x, t.y, t.z);
          best.idx = __float_as_int(t.w);
          best.j = j_prev;
        } else {
          best = grid_nn_warm_cert(L.grid, p.x, p.y, p.z, j_prev, L.stop_d2, L.margin, &slack);
        }
        *sl = slack;
      } else {
        // (UPF 6: the graph search with the flatness certificate — a kernel of its own, so that the launches that do not
        //  use it carry none of its registers)
        if (UPF == 4 || UPF == 6) best = graph ? grid_nn_warm_graph(L.grid, L.knn, p.x, p.y, p.z, j_prev, L.stop_d2, kGraphSkipHopeless, L.launch_idx <= L.knn_peek_until, UPF == 6 ? L.knn_aux : nullptr)
                                   : grid_nn_warm(L.grid, p.x, p.y, p.z, j_prev, L.stop_d2);
        else best = UPF ? grid_nn_warm_upfront<(UPF == 3 ? 3 : 2)>(L.grid, p.x, p.y, p.z, j_prev, L.stop_d2)
                        : grid_nn_warm(L.grid, p.x, p.y, p.z, j_prev, L.stop_d2);
      }
    } else {
      best = grid_nn<G>(L.grid, p.x, p.y, p.z, L.stop_d2);
      if (CERT && lane_in_group == 0) *sl = -1.0f;
    }
  }
  if (in && lane_in_group == 0 && (first || valid)) {
    p.w = __int_as_float(best.j);
    work[i] = p;
  }
  bool keep = valid && best.idx >= 0;
  if (keep && static_cast<double>(best.d2) > L.max_dist_sqr) keep = false;
  if (keep && L.use_rejector && !(best.d2 < L.rej_max2)) keep = false;
  if (in && lane_in_group == 0 && L.corr_idx) {
    const int orig = __float_as_int(L.src[i].w);
    L.corr_idx[orig] = keep ? best.idx : -1;
    L.corr_d2[orig] = keep ? best.d2 : 0.0f;
  }
  if (keep && lane_in_group == 0) accumulate_pair<EST>(L.grid, p, best, acc);
}

// The search half of icp_query (move, search, store the working point) for one lane per query, no certificate and no
// graph: a split iteration's search launch (icp_search_kernel) except where it searches over the graph.  A copy rather
// than a helper shared with icp_query, so that the fused kernels keep their code generation.  p: the moved point; valid:
// the query's point was finite before.
__device__ __forceinline__ NnBest icp_search_query(const IcpLaunch& L, const int h, float4* __restrict__ work, const int i,
                                                   const bool first, const bool apply, const float* T, CoopTile* tile,
                                                   float4& p, bool& valid) {
  const bool in = i < L.n_src;
  p = make_float4(0.f, 0.f, 0.f, 1.f);
  if (in) p = first ? L.src[i] : work[i];
  const int j_prev = first ? -1 : __float_as_int(p.w);  // last iteration's match (sorted position)
  valid = in && finite3(p.x, p.y, p.z);
  if (valid && apply) {
    float ox, oy, oz;
    transform_icp(T, p.x, p.y, p.z, ox, oy, oz);
    p.x = ox;
    p.y = oy;
    p.z = oz;
  }
  NnBest best;
  best.d2 = pos_inf();
  best.idx = -1;
  best.j = -1;
  if (first && L.anchors) {
    // (uniform branch: every lane of the warp takes part, valid or not)
    best = first_iteration_search(L, h, i, valid, p, T, apply, tile);
  } else if (valid) {
    if (L.warm && j_prev >= 0 && j_prev < L.grid.n) best = grid_nn_warm(L.grid, p.x, p.y, p.z, j_prev, L.stop_d2);
    else best = grid_nn<1>(L.grid, p.x, p.y, p.z, L.stop_d2);
  }
  if (in && (first || valid)) {
    p.w = __int_as_float(best.j);
    work[i] = p;
  }
  return best;
}

// [PCL] determineCorrespondences (d2 > max_dist^2 rejected) and the distance rejector (kept iff d2 < max)
__device__ __forceinline__ bool keep_pair(const IcpLaunch& L, const bool valid, const NnBest& best) {
  bool keep = valid && best.idx >= 0;
  if (keep && static_cast<double>(best.d2) > L.max_dist_sqr) keep = false;
  if (keep && L.use_rejector && !(best.d2 < L.rej_max2)) keep = false;
  return keep;
}

// s_inc <- the transform every query of this launch is moved by; s_flags <- active, first iteration, apply transform,
// warm searches over the k-NN graph.  (Followed by a barrier in the caller.)
template <bool FIRST, int UPF>
__device__ __forceinline__ void load_launch_flags(const IcpLaunch& L, const IcpState* st, float* s_inc, int* s_flags) {
  // the guess in launch 0, else the last increment
  if (threadIdx.x < 16) s_inc[threadIdx.x] = FIRST ? __ldcg(&st->final_t.m[threadIdx.x]) : __ldcg(&st->inc.m[threadIdx.x]);
  if (threadIdx.x == 32) {
    const int active = __ldcg(&st->active);
    const int first = FIRST ? 1 : 0;
    int apply = 1;
    if (first) {
      // [PCL] icp.hpp: the guess is applied only if it differs from the identity
      apply = 0;
      for (int i = 0; i < 16; ++i) {
        const float g = __ldcg(&st->final_t.m[i]);
        if (g != ((i % 5 == 0) ? 1.0f : 0.0f)) apply = 1;
      }
    }
    s_flags[0] = active;
    s_flags[1] = first;
    s_flags[2] = apply;
    const int graph = ((UPF == 4 || UPF == 6) && graph_pays(L, st)) ? 1 : 0;
    s_flags[3] = graph;
  }
}

// One block's share of one ICP iteration of hypothesis h: chunk `blk` of L.blocks_per_hyp.  Shared by
// the per-iteration kernel (blk = blockIdx.x, h = blockIdx.y) and the work-queue kernel below.
template <int G, int EST, int MB, bool CERT, bool FIRST, int UPF>
__device__ __forceinline__ void icp_iteration_body(const IcpLaunch& L, const int h, const int blk) {
  unsigned long long t_dbg[5];
  if (L.dbg) t_dbg[0] = global_ns();
  constexpr int NACC = (EST == PEB_ESTIMATOR_SVD) ? kAccSvd : kAccLls;
  __shared__ double sm[kIcpThreads / 32][kAccMax];
  __shared__ double sm_tot[kAccMax];
  __shared__ float s_inc[16];
  __shared__ int s_flags[4];  // active, first iteration, apply transform, warm searches over the k-NN graph
  __shared__ CoopTile s_tile[kIcpThreads / 32];  // first iteration of a batch: one staging tile per warp
  IcpState* st = L.states + h;
  // the transform every query of this launch is moved by: the guess in launch 0, else the last increment
  if (threadIdx.x < 16) s_inc[threadIdx.x] = FIRST ? __ldcg(&st->final_t.m[threadIdx.x]) : __ldcg(&st->inc.m[threadIdx.x]);
  if (threadIdx.x == 32) {
    const int active = __ldcg(&st->active);
    const int first = FIRST ? 1 : 0;
    int apply = 1;
    if (first) {
      // [PCL] icp.hpp: the guess is applied only if it differs from the identity
      apply = 0;
      for (int i = 0; i < 16; ++i) {
        const float g = __ldcg(&st->final_t.m[i]);
        if (g != ((i % 5 == 0) ? 1.0f : 0.0f)) apply = 1;
      }
    }
    s_flags[0] = active;
    s_flags[1] = first;
    s_flags[2] = apply;
    const int graph = ((UPF == 4 || UPF == 6) && graph_pays(L, st)) ? 1 : 0;
    s_flags[3] = graph;
  }
  __syncthreads();
  if (!s_flags[0]) return;
  constexpr bool first = FIRST;
  const bool apply = s_flags[2] != 0;
  // (read from shared memory where it is used: 16 registers less in the search loop)
  const float* T = s_inc;

  double acc[NACC];
#pragma unroll
  for (int i = 0; i < NACC; ++i) acc[i] = 0.0;

  float4* work = L.work + static_cast<size_t>(h) * L.n_src;
  constexpr int kQ = kIcpThreads / G;  // queries per block per pass
  const int q_local = threadIdx.x / G;
  const bool graph = (UPF == 4 || UPF == 6) && s_flags[3] != 0;
  // (Measured and dropped: fetching the working point of the NEXT pass while this pass searches — cp.async into one or
  //  two shared-memory slots per thread, or prefetch.global.L2.  work[i] is the one load of a warm launch that comes
  //  from HBM, the first of three dependent levels, but with 25 warps per SM in flight it is already hidden:
  //  15 020-15 050 against 15 170 hypotheses/s without, profiles/r2_al_prefetch_modes.txt.)
  for (int base = blk * kQ; base < L.n_src; base += L.blocks_per_hyp * kQ)
    icp_query<G, EST, CERT, UPF>(L, h, work, base + q_local, first, apply, graph, T, &s_tile[threadIdx.x >> 5], acc);

  if (L.dbg) t_dbg[1] = global_ns();
  const double r = block_reduce_acc<NACC>(acc, sm);
  double* part = L.partials + (static_cast<size_t>(h) * L.part_stride) * kAccMax;
  if (threadIdx.x < NACC) __stcg(part + static_cast<size_t>(blk) * kAccMax + threadIdx.x, r);
  __threadfence();
  __syncthreads();
  __shared__ int s_last;
  if (threadIdx.x == 0) {
    const unsigned t = atomicAdd(&st->ticket, 1u);
    s_last = (t == static_cast<unsigned>(L.blocks_per_hyp) - 1u);
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  if (L.dbg) t_dbg[2] = global_ns();
  reduce_partials<NACC>(part, L.blocks_per_hyp, sm, sm_tot);
  if (L.dbg) t_dbg[3] = global_ns();
  if (threadIdx.x == 0) {
    finish_iteration<MB>(st, &L.crit, sm_tot, L.trace, L.trace_cap, (L.dbg && h == 0) ? L.dbg + 8 * L.launch_idx : nullptr);
    if (L.dbg && h == 0) {
      t_dbg[4] = global_ns();
      for (int k = 0; k < 5; ++k) L.dbg[8 * L.launch_idx + k] = t_dbg[k];
    }
    if (L.epochs) {  // the state of h is complete: blocks of the next launch that wait for h may go on
      const int still_active = st->active;  // (this thread wrote it)
      __threadfence();
      atomicAdd(L.epochs + h, still_active ? 1 : kEpochStopped);
    }
  }
}

// FIRST: launch 0 of an align (the state's iteration counter is 0 exactly then) — a compile-time
// property so that the first iteration's search code stays out of the warm kernels' register budget.
// Dependencies between the launches of an align.  A launch is issued with programmatic dependent launch and
// triggers its successor at once, so the successor's blocks take SM slots as soon as ALL blocks of this launch
// are resident or done.  Launch 0 then waits for everything before it (griddepcontrol.wait: init, anchors).
// A warm launch does not wait for the whole previous grid: a block of hypothesis h only needs iteration
// launch_idx - 1 OF h — its last block publishes epochs[h] after writing the state (release / acquire) —
// so hypotheses whose solve is done move on while the previous launch still drains its tail.  No deadlock: a
// waiting block only waits for blocks of earlier launches, and those were all resident before it was dispatched.
// The wait is bounded (a dependency that never comes would be a bug): it then raises the error flag, which the
// fitness kernel reports in every record.
template <int G, int EST, int MB, bool CERT, bool FIRST, int UPF = 0>
__global__ void __launch_bounds__(kIcpThreads, MB) icp_iteration_kernel(const IcpLaunch L) {
  if (FIRST || L.epochs == nullptr) {
    pdl_trigger_and_wait();
  } else {
    asm volatile("griddepcontrol.launch_dependents;");
    wait_for_hypothesis(L.epochs + blockIdx.y, L.launch_idx, L.err_flag);
  }
  icp_iteration_body<G, EST, MB, CERT, FIRST, UPF>(L, blockIdx.y, blockIdx.x);
}

// ---- one iteration of a batch as two launches: the searches, then the moments and the solve ----------------------
// In icp_iteration_kernel the double moment sums (17 for SVD, 28 for LLS), the block reduction and the out-of-line
// solve share the allocation of the search loop: the batched kernels spill at their 64-register cap, and their late
// launches, bound by the L2 latency of the searches, run with about 25 resident warps per SM.  Split:
//   icp_search_kernel  grid = (search blocks per hypothesis, H): the fused kernel's search half (icp_search_query;
//                      over the k-NN graph icp_search_graph_queued, which walks the grid in dense warps) and nothing
//                      else — no double state, no reduction, no solve — under its own register cap (kMinBlocksSearch): more
//                      resident warps to hide the search's latency.  Its block count is free: it writes no records.
//   icp_moment_kernel  grid = (blocks_per_hyp, H): per query the working point and its match are read back and d2 is
//                      recomputed as every search path computes it (l2_simple of the query and the match); threshold,
//                      moments, block record, ticket, reduction and solve follow as in icp_iteration_body.  Its blocks
//                      and its query-to-thread mapping (G = 1) are the fused kernel's, so every double is added in the
//                      same order: byte-identical records.  It reads the working clouds once more.
// A point that this launch's transform makes non-finite (a non-finite guess or increment) is still a valid query of the
// fused kernel, which searches it; its match is stored as -2 - j in .w so that the moment launch can tell, and the next
// search launch, for which the point is invalid, resets it to -1 (the fitness search is exact whether it starts warm or
// cold, so nothing else reads the difference).
// Dependencies with flags: a search block of (h, k) waits for epochs[h] >= k as a fused block does; if h is active, every
// search block then takes a ticket of the state (ticket_search), and the last one resets it and publishes searched = k + 1
// (fence + atomic); a moment block of (h, k) waits for searched >= k + 1 or for h to have stopped (wait_for_search).  The
// split launches of an align are a prefix of its launches (the host keeps it so), hence the count.  The launches of an
// active hypothesis never overlap (search k + 1 waits for the solve of k), so the ticket's reset races with nothing; those
// of a stopped one do (its epoch releases them all), and they take no ticket.  Every block still waits only for blocks of
// earlier launches (see icp_iteration_kernel).  Without flags both launches wait for the whole previous grid.
// The search stride is gridDim.x: its blocks per hypothesis are free (it writes no records).

// .w of a searched valid query: its match, or -2 - match for a point this launch's transform made non-finite
__device__ __forceinline__ int search_slot(float x, float y, float z, int j) {
  return (j >= 0 && !finite3(x, y, z)) ? -2 - j : j;
}

// A query the graph could not prove, waiting in its warp's queue: the moved point, the sorted position of the best point
// the graph met (-1: no previous match, a cold search) and the query's index.  20 bytes: lanes reading consecutive
// entries hit 32 different banks.
struct SearchQueued {
  float x, y, z;
  int cand;
  int i;
};
constexpr int kSearchQueue = 64;  // per warp: at most 31 waiting + one pass of 32

// The search launch of a hypothesis that searches over the graph (graph_pays).  In a late launch the row of the previous
// match proves nearly every query, but the ~6 % it cannot prove walk the grid (grid_ball_search: per-lane loops, 8
// dependent load levels) while the rest of their warp idles.  Here every lane moves its query and tries the graph
// (grid_nn_graph_try); a proven query stores its working point at once, an unproven one goes to the warp's queue with
// everything its walk needs, and whenever 32 are waiting (and once at the end) the warp walks them one per lane.  No block
// barrier: the warps of a block queue and drain on their own.  The walk is exact for any candidate, and the candidate is
// rebuilt from its position with the expression the graph computed it with, so every match is the per-lane search's and
// every working point is written once, with the same bytes.
template <int UPF>
__device__ __forceinline__ void icp_search_graph_queued(const IcpLaunch& L, float4* __restrict__ work, const bool apply,
                                                        const float* T) {
  __shared__ SearchQueued s_queue[kIcpThreads / 32][kSearchQueue];
  SearchQueued* queue = s_queue[threadIdx.x >> 5];
  const int lane = threadIdx.x & 31;
  const bool peek = L.launch_idx <= L.knn_peek_until;
  int n_queue = 0;  // (warp-uniform)
  // lanes [0, count) walk the grid for the LAST count entries of the queue
  auto drain = [&](int count) {
    if (lane < count) {
      const SearchQueued e = queue[n_queue - count + lane];
      NnBest best;
      if (e.cand >= 0) {
        const float4 t = L.grid.pts[e.cand];
        best.d2 = l2_simple(e.x, e.y, e.z, t.x, t.y, t.z);
        best.idx = point_index(t);
        best.j = e.cand;
        grid_ball_search(L.grid, e.x, e.y, e.z, L.stop_d2, best);
      } else {
        best = grid_nn<1>(L.grid, e.x, e.y, e.z, L.stop_d2);
      }
      work[e.i] = make_float4(e.x, e.y, e.z, __int_as_float(search_slot(e.x, e.y, e.z, best.j)));
    }
    n_queue -= count;
    __syncwarp();
  };
  for (int base = blockIdx.x * kIcpThreads; base < L.n_src; base += gridDim.x * kIcpThreads) {
    const int i = base + threadIdx.x;
    const bool in = i < L.n_src;
    float4 p = make_float4(0.f, 0.f, 0.f, 1.f);
    if (in) p = work[i];
    const int j_prev = __float_as_int(p.w);  // last iteration's match (sorted position)
    bool need = false;
    int cand = -1;
    if (in && finite3(p.x, p.y, p.z)) {
      if (apply) {
        float ox, oy, oz;
        transform_icp(T, p.x, p.y, p.z, ox, oy, oz);
        p.x = ox;
        p.y = oy;
        p.z = oz;
      }
      need = true;
      if (L.warm && j_prev >= 0 && j_prev < L.grid.n) {
        NnBest best;
        need = !grid_nn_graph_try(L.grid, L.knn, p.x, p.y, p.z, j_prev, best, kGraphSkipHopeless, peek,
                                  UPF == 6 ? L.knn_aux : nullptr);
        if (need) cand = best.j;
        else work[i] = make_float4(p.x, p.y, p.z, __int_as_float(search_slot(p.x, p.y, p.z, best.j)));
      }
    } else if (in && j_prev <= -2) {
      reinterpret_cast<int*>(work + i)[3] = -1;  // invalid before this launch: no match to carry (see above)
    }
    const unsigned m = __ballot_sync(0xFFFFFFFFu, need);
    if (m) {
      if (need) queue[n_queue + __popc(m & ((1u << lane) - 1u))] = SearchQueued{p.x, p.y, p.z, cand, i};
      n_queue += __popc(m);
      __syncwarp();
      if (n_queue >= 32) drain(32);
    }
  }
  if (n_queue) drain(n_queue);
}

template <int MB, bool FIRST, int UPF>
__global__ void __launch_bounds__(kIcpThreads, MB) icp_search_kernel(const IcpLaunch L) {
  if (FIRST || L.epochs == nullptr) {
    pdl_trigger_and_wait();
  } else {
    asm volatile("griddepcontrol.launch_dependents;");
    wait_for_hypothesis(L.epochs + blockIdx.y, L.launch_idx, L.err_flag);
  }
  const int h = blockIdx.y, blk = blockIdx.x;
  __shared__ float s_inc[16];
  __shared__ int s_flags[4];
  __shared__ CoopTile s_tile[kIcpThreads / 32];
  IcpState* st = L.states + h;
  load_launch_flags<FIRST, UPF>(L, st, s_inc, s_flags);
  __syncthreads();
  if (s_flags[0]) {
    const bool apply = s_flags[2] != 0;
    const bool graph = (UPF == 4 || UPF == 6) && s_flags[3] != 0;
    float4* work = L.work + static_cast<size_t>(h) * L.n_src;
    if (!FIRST && graph) icp_search_graph_queued<UPF>(L, work, apply, s_inc);
    else for (int base = blk * kIcpThreads; base < L.n_src; base += gridDim.x * kIcpThreads) {
      const int i = base + threadIdx.x;
      float4 p;
      bool valid;
      const NnBest best = icp_search_query(L, h, work, i, FIRST, apply, s_inc, &s_tile[threadIdx.x >> 5], p, valid);
      int* w = reinterpret_cast<int*>(work + i) + 3;
      if (valid && best.j >= 0 && !finite3(p.x, p.y, p.z)) *w = -2 - best.j;
      else if (!FIRST && !valid && i < L.n_src && __float_as_int(p.w) <= -2) *w = -1;
    }
  }
  if (L.epochs && s_flags[0]) {
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      if (atomicAdd(&st->ticket_search, 1u) == gridDim.x - 1u) {
        st->ticket_search = 0u;
        __threadfence();
        atomicAdd(&st->searched, 1);
      }
    }
  }
}

// ---- the moment launch's copy pipeline ----
// In pass k, block blk of a hypothesis reads queries blk * 128 + t + k * blocks_per_hyp * 128: one contiguous 2 KB chunk of
// the working cloud per pass.  A per-thread load loop keeps one 512-byte load per warp in flight and then waits for the
// dependent gather of the match, about 16 KB per SM: the launch was bound by that, at a third of HBM bandwidth.  Instead
// thread 0 streams the chunks into a ring of kMomentRing slots in shared memory with 1-D bulk copies (one mbarrier per slot):
// a slot is refilled once every thread has added its pass, kMomentRing - 2 passes before the threads read it.  The
// accumulators keep their registers and every thread still adds its queries in increasing pass order, so every double is
// summed as before.
#ifndef PEB_MOMENT_RING
#define PEB_MOMENT_RING 4
#endif
constexpr int kMomentRing = PEB_MOMENT_RING;  // (development: -DPEB_MOMENT_RING=n builds a variant library, PEB_LIB_VARIANT)
static_assert(kMomentRing >= 2 && (kMomentRing & (kMomentRing - 1)) == 0, "ring depth: a power of two >= 2");
#ifndef PEB_MOMENT_EVICT_FIRST
#define PEB_MOMENT_EVICT_FIRST 0
#endif

__device__ __forceinline__ uint32_t smem_addr(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

// thread 0: `bytes` (a multiple of 16) from global src into shared dst; completion is counted on the mbarrier bar
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
#if PEB_MOMENT_EVICT_FIRST
  // the working clouds are read once per iteration: let them leave L2 before the target's structures do
  uint64_t policy;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(policy) : "memory");
#else
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
#endif
}

__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred done;\n"
      "WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 done, [%0], %1;\n"
      "@!done bra WAIT;\n"
      "}\n" ::"r"(bar), "r"(parity) : "memory");
}

// one query of a moment pass: its match j (-1: no pair) and the match t, read one pass before the query is added.  (The
// working point is read from the ring again when it is added: 3 registers less in flight.  The point-to-plane sums hold
// 58 of the 64 registers in doubles: there the match and its normal are read when added, as before, so as not to spill.)
template <int EST>
struct MomentGather {
  static constexpr bool kAhead = EST == PEB_ESTIMATOR_SVD;
  float4 t;
  int j;
};

// CHAIN: the align has a rejector chain (icp_reject_kernel ran between the two launches): a pair is summed iff
// kept[i] of its hypothesis is set, and the single align's correspondence outputs are written here.
template <int EST, int MB, bool CHAIN>
__global__ void __launch_bounds__(kIcpThreads, MB) icp_moment_kernel(const IcpLaunch L, const unsigned char* __restrict__ kept) {
  if (L.epochs == nullptr) {
    pdl_trigger_and_wait();
  } else {
    asm volatile("griddepcontrol.launch_dependents;");
    wait_for_search(&L.states[blockIdx.y].searched, L.launch_idx + 1, L.epochs + blockIdx.y, L.err_flag);
  }
  const int h = blockIdx.y, blk = blockIdx.x;
  constexpr int NACC = (EST == PEB_ESTIMATOR_SVD) ? kAccSvd : kAccLls;
  __shared__ double sm[kIcpThreads / 32][kAccMax];
  __shared__ double sm_tot[kAccMax];
  __shared__ int s_active;
  __shared__ alignas(16) float4 s_ring[kMomentRing][kIcpThreads];
  __shared__ alignas(8) unsigned long long s_full[kMomentRing];
  IcpState* st = L.states + h;
  if (threadIdx.x == 0) s_active = __ldcg(&st->active);
  __syncthreads();
  if (!s_active) return;  // (before any copy: a block never leaves with one outstanding)

  double acc[NACC];
#pragma unroll
  for (int i = 0; i < NACC; ++i) acc[i] = 0.0;
  const float4* work = L.work + static_cast<size_t>(h) * L.n_src;
  const int i0 = blk * kIcpThreads, stride = L.blocks_per_hyp * kIcpThreads;
  const int n_pass = i0 < L.n_src ? (L.n_src - i0 + stride - 1) / stride : 0;  // (block-uniform)
  // pass k into slot k % kMomentRing; the last chunk is clipped to n_src
  auto issue = [&](int k) {
    const int i = i0 + k * stride;
    const int slot = k & (kMomentRing - 1);
    bulk_copy_g2s(smem_addr(s_ring[slot]), work + i, static_cast<uint32_t>(min(kIcpThreads, L.n_src - i)) * sizeof(float4),
                  smem_addr(&s_full[slot]));
  };
  if (threadIdx.x == 0) {
#pragma unroll
    for (int s = 0; s < kMomentRing; ++s) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_addr(&s_full[s])) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    // The working points were written by the search grid through the generic proxy and acquired above (wait_for_search or
    // griddepcontrol.wait); the bulk copies read them through the async proxy, which that acquire does not order.
    asm volatile("fence.proxy.async.global;" ::: "memory");
    for (int k = 0; k < min(kMomentRing, n_pass); ++k) issue(k);
  }
  __syncthreads();

  // waits for pass k's chunk, reads this thread's query and starts the gathers of its match
  using Gather = MomentGather<EST>;
  auto fetch = [&](int k, Gather& q) {
    const int slot = k & (kMomentRing - 1);
    mbar_wait(smem_addr(&s_full[slot]), (k / kMomentRing) & 1);
    const int i = i0 + k * stride + threadIdx.x;
    q.j = -1;
    if (i >= L.n_src) return;  // (past the clipped end: the slot holds an older chunk's bytes)
    const float4 p = s_ring[slot][threadIdx.x];
    int j = __float_as_int(p.w);
    if (j <= -2) j = -2 - j;  // made non-finite by this launch's transform: searched all the same (see above)
    else if (!finite3(p.x, p.y, p.z)) j = -1;
    q.j = j;
    if (Gather::kAhead && j >= 0) q.t = L.grid.pts[j];
  };
  auto add = [&](int k, const Gather& q) {
    const float4 p = s_ring[k & (kMomentRing - 1)][threadIdx.x];
    const int i = i0 + k * stride + threadIdx.x;
    if (CHAIN) {
      NnBest best;
      const bool keep = q.j >= 0 && kept[static_cast<size_t>(h) * L.n_src + i];
      if (keep) {
        const float4 t = Gather::kAhead ? q.t : L.grid.pts[q.j];
        best.d2 = l2_simple(p.x, p.y, p.z, t.x, t.y, t.z);
        best.idx = point_index(t);
        add_moments<EST, NACC>(L.grid, p, t, q.j, best.d2, acc);
      }
      if (L.corr_idx && i < L.n_src) {
        const int orig = __float_as_int(L.src[i].w);
        L.corr_idx[orig] = keep ? best.idx : -1;
        L.corr_d2[orig] = keep ? best.d2 : 0.0f;
      }
      return;
    }
    if (q.j < 0) return;
    const float4 t = Gather::kAhead ? q.t : L.grid.pts[q.j];
    NnBest best;
    best.d2 = l2_simple(p.x, p.y, p.z, t.x, t.y, t.z);
    best.idx = point_index(t);
    best.j = q.j;
    if (keep_pair(L, true, best)) add_moments<EST, NACC>(L.grid, p, t, q.j, best.d2, acc);
  };
  // at pass k: every thread has added pass k - 1, whose slot takes pass k - 1 + kMomentRing
  auto refill = [&](int k) {
    __syncthreads();
    if (threadIdx.x == 0 && k >= 1 && k - 1 + kMomentRing < n_pass) issue(k - 1 + kMomentRing);
  };
  // pass k: refill, start pass k + 1's gathers into `next`, add pass k (`cur`)
  auto step = [&](int k, const Gather& cur, Gather& next) {
    refill(k);
    if (k + 1 < n_pass) fetch(k + 1, next);
    add(k, cur);
  };

  if constexpr (Gather::kAhead) {
    // (two records that swap roles: a copy from one to the other would wait for the gathers in flight)
    Gather qa, qb;
    if (n_pass > 0) fetch(0, qa);
#pragma unroll 1
    for (int k = 0; k < n_pass; k += 2) {
      step(k, qa, qb);
      if (k + 1 < n_pass) step(k + 1, qb, qa);
    }
  } else {
#pragma unroll 1
    for (int k = 0; k < n_pass; ++k) {
      refill(k);
      Gather q;
      fetch(k, q);
      add(k, q);
    }
  }

  // ---- the block's record, the last block's solve: as in icp_iteration_body ----
  const double r = block_reduce_acc<NACC>(acc, sm);
  double* part = L.partials + (static_cast<size_t>(h) * L.part_stride) * kAccMax;
  if (threadIdx.x < NACC) __stcg(part + static_cast<size_t>(blk) * kAccMax + threadIdx.x, r);
  __threadfence();
  __syncthreads();
  __shared__ int s_last;
  if (threadIdx.x == 0) {
    const unsigned t = atomicAdd(&st->ticket, 1u);
    s_last = (t == static_cast<unsigned>(L.blocks_per_hyp) - 1u);
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  reduce_partials<NACC>(part, L.blocks_per_hyp, sm, sm_tot);
  if (threadIdx.x == 0) {
    finish_iteration<MB>(st, &L.crit, sm_tot, L.trace, L.trace_cap, nullptr);
    if (L.epochs) {
      const int still_active = st->active;
      __threadfence();
      atomicAdd(L.epochs + h, still_active ? 1 : kEpochStopped);
    }
  }
}

// ---- correspondence rejectors (peb_icp_align_ex) --------------------------------------------------------------------
// An align with a rejector chain runs every iteration as three launches: icp_search_kernel, icp_reject_kernel and
// icp_moment_kernel<CHAIN = true>.  Between the search and the moments every pair of the iteration is known and no moment
// has been summed: the reject launch gives every hypothesis one block of kRejThreads threads, which applies the threshold,
// rejector_max_dist and then the chain in order to all pairs of its hypothesis (a __syncthreads between stages) and leaves
// one kept byte per working point.  One block sees the whole pair set, so the order statistics and the one-to-one table
// need no cross-block protocol; the launches wait for the whole previous grid (griddepcontrol.wait, no epoch flags).
//   MEDIAN_DISTANCE  score (rej_score), exact (m / 2)-th order statistic over the kept pairs (block_select_nth), keep iff
//                    (double) score <= median * factor.
//   TRIMMED          the (n_keep - 1)-th smallest d2 v over the kept pairs; all pairs below v stay, and of the pairs AT v the
//                    ones of the smallest original source indices (a second select over those indices) fill n_keep.
//   ONE_TO_ONE       atomicMin of (d2 bits << 32 | original source index) into the hypothesis's row of the table (indexed by
//                    the match's sorted position), then every pair reads its entry back: the one that finds its own key
//                    wins and resets the entry to all ones.  A loser reads the winner's key or all ones, never its own, so
//                    the table is all ones again after every stage without a pass over it (it is set once, when allocated).
// Sign bits are cleared before a select (a NaN distance from a non-finite working point sorts last instead of being lost).
constexpr int kRejThreads = 1024;

struct RejChain {
  int kind[PEB_MAX_REJECTORS];
  int min_corr[PEB_MAX_REJECTORS];
  double value[PEB_MAX_REJECTORS];
  int n;
  unsigned char* kept;         // H x n_src: the pair of working point i survives the chain
  unsigned long long* o2o;     // H x grid.n one-to-one keys, all ones between stages (nullptr without ONE_TO_ONE)
};

// the pair of working point i as the moment launch reads it (best.idx = -1: no pair)
__device__ __forceinline__ NnBest rej_pair(const IcpLaunch& L, const float4* __restrict__ work, int i, float4& p, bool& valid) {
  p = __ldcg(work + i);
  valid = finite3(p.x, p.y, p.z);
  int j = __float_as_int(p.w);
  if (j <= -2) {
    valid = true;
    j = -2 - j;
  }
  NnBest best;
  best.d2 = pos_inf();
  best.idx = -1;
  best.j = -1;
  if (valid && j >= 0) {
    const float4 t = L.grid.pts[j];
    best.d2 = l2_simple(p.x, p.y, p.z, t.x, t.y, t.z);
    best.idx = point_index(t);
    best.j = j;
  }
  return best;
}

__device__ __forceinline__ unsigned abs_bits(float v) { return __float_as_uint(v) & 0x7FFFFFFFu; }

// [PCL] CorrespondenceRejectorMedianDistance's score: DataContainer::getCorrespondenceScore, (src.getVector4fMap() -
// tgt.getVector4fMap()).squaredNorm() in float, w = 1 on both sides; Eigen's 4-lane reduction (v0 + v2) + (v1 + v3),
// the last term 0.  Written without contraction (the library is built with -fmad=false).
__device__ __forceinline__ float rej_score(const IcpLaunch& L, const float4& p, int j) {
  const float4 t = L.grid.pts[j];
  const float dx = p.x - t.x, dy = p.y - t.y, dz = p.z - t.z;
  return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dz, dz)), __fmul_rn(dy, dy));
}

// number of kept pairs of the block's hypothesis (every thread gets it)
__device__ __forceinline__ int rej_count(const unsigned char* kept, int n) {
  int m = 0;
  for (int base = 0; base < n; base += kRejThreads) {
    const int i = base + threadIdx.x;
    m += __syncthreads_count(i < n && kept[i]);
  }
  return m;
}

__global__ void __launch_bounds__(kRejThreads, 1) icp_reject_kernel(const IcpLaunch L, const RejChain R) {
  pdl_trigger_and_wait();
  __shared__ unsigned hist[2048];
  __shared__ unsigned s_state[2];
  __shared__ unsigned s_wsum[32];
  __shared__ int s_active;
  const int h = blockIdx.x;
  if (threadIdx.x == 0) s_active = __ldcg(&L.states[h].active);
  __syncthreads();
  if (!s_active) return;
  const int n = L.n_src;
  const float4* work = L.work + static_cast<size_t>(h) * n;
  unsigned char* kept = R.kept + static_cast<size_t>(h) * n;
  unsigned long long* tab = R.o2o ? R.o2o + static_cast<size_t>(h) * L.grid.n : nullptr;
  for (int i = threadIdx.x; i < n; i += kRejThreads) {
    float4 p;
    bool valid;
    const NnBest b = rej_pair(L, work, i, p, valid);
    kept[i] = keep_pair(L, valid, b) ? 1 : 0;
  }
  __syncthreads();
  for (int s = 0; s < R.n; ++s) {
    const int kind = R.kind[s];
    if (kind == PEB_REJECTOR_DISTANCE) {
      const float lim = static_cast<float>(R.value[s] * R.value[s]);
      for (int i = threadIdx.x; i < n; i += kRejThreads) {
        if (!kept[i]) continue;
        float4 p;
        bool valid;
        const NnBest b = rej_pair(L, work, i, p, valid);
        if (!(b.d2 < lim)) kept[i] = 0;
      }
    } else if (kind == PEB_REJECTOR_MEDIAN_DISTANCE) {
      const int m = rej_count(kept, n);
      if (m == 0) continue;
      auto score = [&](int i) {
        if (!kept[i]) return -1.0f;
        float4 p;
        bool valid;
        const NnBest b = rej_pair(L, work, i, p, valid);
        return __uint_as_float(abs_bits(rej_score(L, p, b.j)));
      };
      const float med = block_select_nth<decltype(score), true>(score, n, m / 2, hist, s_state, s_wsum);
      const double lim = static_cast<double>(med) * R.value[s];
      for (int i = threadIdx.x; i < n; i += kRejThreads) {
        if (!kept[i]) continue;
        float4 p;
        bool valid;
        const NnBest b = rej_pair(L, work, i, p, valid);
        if (!(static_cast<double>(rej_score(L, p, b.j)) <= lim)) kept[i] = 0;
      }
    } else if (kind == PEB_REJECTOR_ONE_TO_ONE) {
      for (int i = threadIdx.x; i < n; i += kRejThreads) {
        if (!kept[i]) continue;
        float4 p;
        bool valid;
        const NnBest b = rej_pair(L, work, i, p, valid);
        const unsigned long long key = (static_cast<unsigned long long>(abs_bits(b.d2)) << 32) |
                                       static_cast<unsigned>(__float_as_int(L.src[i].w));
        atomicMin(tab + b.j, key);
      }
      __syncthreads();
      for (int i = threadIdx.x; i < n; i += kRejThreads) {
        if (!kept[i]) continue;
        float4 p;
        bool valid;
        const NnBest b = rej_pair(L, work, i, p, valid);
        const unsigned long long key = (static_cast<unsigned long long>(abs_bits(b.d2)) << 32) |
                                       static_cast<unsigned>(__float_as_int(L.src[i].w));
        if (__ldcg(tab + b.j) == key) __stcg(tab + b.j, ~0ull);
        else kept[i] = 0;
      }
    } else {  // PEB_REJECTOR_TRIMMED
      const int m = rej_count(kept, n);
      const float ratio = fminf(1.0f, fmaxf(0.0f, static_cast<float>(R.value[s])));
      const int n_keep = max(static_cast<int>(floorf(ratio * static_cast<float>(m))), R.min_corr[s]);
      if (n_keep >= m) continue;
      unsigned vb = 0u;  // the d2 bits of the cut
      int o_cut = -1;    // pairs at the cut with source index <= o_cut stay
      if (n_keep > 0) {
        auto d2_of = [&](int i) {
          if (!kept[i]) return -1.0f;
          float4 p;
          bool valid;
          return __uint_as_float(abs_bits(rej_pair(L, work, i, p, valid).d2));
        };
        vb = __float_as_uint(block_select_nth<decltype(d2_of), true>(d2_of, n, n_keep - 1, hist, s_state, s_wsum));
        int below = 0;
        for (int base = 0; base < n; base += kRejThreads) {
          const int i = base + threadIdx.x;
          bool lt = false;
          if (i < n && kept[i]) {
            float4 p;
            bool valid;
            lt = abs_bits(rej_pair(L, work, i, p, valid).d2) < vb;
          }
          below += __syncthreads_count(lt);
        }
        auto src_at_cut = [&](int i) {
          if (!kept[i]) return -1.0f;
          float4 p;
          bool valid;
          if (abs_bits(rej_pair(L, work, i, p, valid).d2) != vb) return -1.0f;
          return __int_as_float(__float_as_int(L.src[i].w));
        };
        o_cut = __float_as_int(block_select_nth<decltype(src_at_cut), true>(src_at_cut, n, n_keep - below - 1, hist, s_state, s_wsum));
      }
      for (int i = threadIdx.x; i < n; i += kRejThreads) {
        if (!kept[i]) continue;
        bool stay = false;
        if (n_keep > 0) {
          float4 p;
          bool valid;
          const unsigned db = abs_bits(rej_pair(L, work, i, p, valid).d2);
          stay = db < vb || (db == vb && __float_as_int(L.src[i].w) <= o_cut);
        }
        if (!stay) kept[i] = 0;
      }
    }
    __syncthreads();
  }
}

// ---- warm iterations with the queries of a block binned by the size of their search ------------------------------
// The ball walk of a warm query visits the rows of the ball's bounding box (core_math.cuh : grid_ball_search); a
// lane with a 1 x 1 box next to a lane with a 3 x 4 box idles through eleven row steps, and almost every warp of 32
// consecutive queries holds such a lane (box rows per query on C4: 1: 19 %, 2: 35 %, 3-4: 38 %, more: 8 %; the plain
// kernel runs at ~15 of 32 active lanes).  Here a block takes a TILE of kBinQ passes of the plain kernel's loop:
//   1. every thread moves its kBinQ queries, gathers their previous matches and parks query + candidate in shared
//      memory, classed by the number of rows the walk will visit (queries without a previous match search cold:
//      heaviest class);
//   2. the tile is counting-sorted by class, heaviest first;
//   3. warps draw 32 sorted queries at a time from a shared counter and search them — the lanes of a warp now walk
//      (nearly) the same number of rows;
//   4. every thread takes ITS queries back in the plain kernel's order: working point written, threshold, moments.
// The queries, the searches and the order of every thread's double sums are those of icp_iteration_kernel: results
// are bit-identical by construction (tests/test_gpu_bin_option.py).
constexpr int kBinQ = 4;                         // plain-loop passes per tile
constexpr int kBinTile = kBinQ * kIcpThreads;    // queries per tile
constexpr int kBinClasses = 5;                   // searching classes, heaviest first; class kBinClasses = nothing to search

__device__ __forceinline__ int bin_class_of_rows(int rows) {
  return rows >= 7 ? 0 : rows >= 5 ? 1 : rows >= 3 ? 2 : rows == 2 ? 3 : 4;
}

template <int EST, int MB>
__global__ void __launch_bounds__(kIcpThreads, MB) icp_iteration_binned_kernel(const IcpLaunch L) {
  if (L.epochs == nullptr) {
    pdl_trigger_and_wait();
  } else {
    asm volatile("griddepcontrol.launch_dependents;");
    wait_for_hypothesis(L.epochs + blockIdx.y, L.launch_idx, L.err_flag);
  }
  const int h = blockIdx.y, blk = blockIdx.x;
  constexpr int NACC = (EST == PEB_ESTIMATOR_SVD) ? kAccSvd : kAccLls;
  __shared__ double sm[kIcpThreads / 32][kAccMax];
  __shared__ double sm_tot[kAccMax];
  __shared__ float s_inc[16];
  __shared__ int s_active;
  __shared__ float s_qx[kBinTile], s_qy[kBinTile], s_qz[kBinTile], s_d2[kBinTile];
  __shared__ int s_idx[kBinTile], s_j[kBinTile];
  __shared__ unsigned short s_key[kBinTile], s_perm[kBinTile];
  __shared__ int s_cnt[2][kBinClasses + 1];  // per class; [kBinClasses] = the chunk counter of phase 3 (double-buffered by tile parity)
  IcpState* st = L.states + h;
  if (threadIdx.x < 16) s_inc[threadIdx.x] = __ldcg(&st->inc.m[threadIdx.x]);
  if (threadIdx.x == 32) s_active = __ldcg(&st->active);
  if (threadIdx.x >= 64 && threadIdx.x < 64 + 2 * (kBinClasses + 1)) (&s_cnt[0][0])[threadIdx.x - 64] = 0;
  __syncthreads();
  if (!s_active) return;
  const float* T = s_inc;
  float4* work = L.work + static_cast<size_t>(h) * L.n_src;
  const int stride = L.blocks_per_hyp * kIcpThreads;
  const int lane = threadIdx.x & 31;
  const unsigned lt = (1u << lane) - 1u;

  double acc[NACC];
#pragma unroll
  for (int i = 0; i < NACC; ++i) acc[i] = 0.0;

  int buf = 0;
  for (int base0 = blk * kIcpThreads; base0 < L.n_src; base0 += kBinQ * stride, buf ^= 1) {
    // ---- 1: move, gather the previous match, class ----
#pragma unroll 1
    for (int kk = 0; kk < kBinQ; ++kk) {
      const int i = base0 + kk * stride + threadIdx.x;
      const int slot = kk * kIcpThreads + threadIdx.x;
      int cls = kBinClasses;
      float qx = 0.0f, qy = 0.0f, qz = 0.0f, d2 = pos_inf();
      int idx = -1, j = -2;  // -2: nothing here (out of range or a non-finite working point), -1: no previous match
      if (i < L.n_src) {
        const float4 p = work[i];
        if (finite3(p.x, p.y, p.z)) {
          transform_icp(T, p.x, p.y, p.z, qx, qy, qz);
          const int j_prev = __float_as_int(p.w);
          cls = 0;  // no usable previous match: cold search
          j = -1;
          if (L.warm && j_prev >= 0 && j_prev < L.grid.n) {
            const float4 t = L.grid.pts[j_prev];
            d2 = l2_simple(qx, qy, qz, t.x, t.y, t.z);
            idx = __float_as_int(t.w);
            j = j_prev;
            cls = bin_class_of_rows(grid_ball_rows(L.grid, qy, qz, d2, L.stop_d2));
          }
        }
      }
      s_qx[slot] = qx;
      s_qy[slot] = qy;
      s_qz[slot] = qz;
      s_d2[slot] = d2;
      s_idx[slot] = idx;
      s_j[slot] = j;
      // position inside the class: one shared-memory atomic per class present in the warp
      const unsigned same = __match_any_sync(0xFFFFFFFFu, cls);
      const int leader = __ffs(same) - 1;
      int at = 0;
      if (lane == leader && cls < kBinClasses) at = atomicAdd(&s_cnt[buf][cls], __popc(same));
      at = __shfl_sync(0xFFFFFFFFu, at, leader);
      s_key[slot] = static_cast<unsigned short>((cls << 12) | (at + __popc(same & lt)));
    }
    __syncthreads();
    // ---- 2: counting sort by class ----
    int off[kBinClasses + 1];
    off[0] = 0;
#pragma unroll
    for (int c = 0; c < kBinClasses; ++c) off[c + 1] = off[c] + s_cnt[buf][c];
    const int n_search = off[kBinClasses];
#pragma unroll
    for (int kk = 0; kk < kBinQ; ++kk) {
      const int slot = kk * kIcpThreads + threadIdx.x;
      const int key = s_key[slot];
      const int cls = key >> 12;
      if (cls < kBinClasses) {
        int o = 0;
#pragma unroll
        for (int c = 1; c < kBinClasses; ++c) o = cls == c ? off[c] : o;
        s_perm[o + (key & 0xFFF)] = static_cast<unsigned short>(slot);
      }
    }
    // (the other buffer's counters were last read before this tile's first barrier: reset them for the next tile)
    if (threadIdx.x < kBinClasses + 1) s_cnt[buf ^ 1][threadIdx.x] = 0;
    __syncthreads();
    // ---- 3: searches, 32 sorted queries per draw ----
    for (;;) {
      int c = 0;
      if (lane == 0) c = atomicAdd(&s_cnt[buf][kBinClasses], 1);
      c = __shfl_sync(0xFFFFFFFFu, c, 0);
      if (c * 32 >= n_search) break;
      const int k = c * 32 + lane;
      if (k < n_search) {
        const int slot = s_perm[k];
        NnBest best;
        best.d2 = s_d2[slot];
        best.idx = s_idx[slot];
        best.j = s_j[slot];
        const float qx = s_qx[slot], qy = s_qy[slot], qz = s_qz[slot];
        if (best.j >= 0) grid_ball_search(L.grid, qx, qy, qz, L.stop_d2, best);
        else best = grid_nn<1>(L.grid, qx, qy, qz, L.stop_d2);
        s_d2[slot] = best.d2;
        s_idx[slot] = best.idx;
        s_j[slot] = best.j;
      }
    }
    __syncthreads();
    // ---- 4: every thread its own queries, in the plain kernel's order ----
#pragma unroll 1
    for (int kk = 0; kk < kBinQ; ++kk) {
      const int i = base0 + kk * stride + threadIdx.x;
      const int slot = kk * kIcpThreads + threadIdx.x;
      if (i >= L.n_src) break;
      NnBest best;
      best.j = s_j[slot];
      if (best.j == -2) continue;  // non-finite working point: untouched, no correspondence
      best.d2 = s_d2[slot];
      best.idx = s_idx[slot];
      float4 p;
      p.x = s_qx[slot];
      p.y = s_qy[slot];
      p.z = s_qz[slot];
      p.w = __int_as_float(best.j);
      work[i] = p;
      bool keep = best.idx >= 0;
      if (keep && static_cast<double>(best.d2) > L.max_dist_sqr) keep = false;
      if (keep && L.use_rejector && !(best.d2 < L.rej_max2)) keep = false;
      if (L.corr_idx) {
        const int orig = __float_as_int(L.src[i].w);
        L.corr_idx[orig] = keep ? best.idx : -1;
        L.corr_d2[orig] = keep ? best.d2 : 0.0f;
      }
      if (keep) accumulate_pair<EST>(L.grid, p, best, acc);
    }
    // (phase 1 of the next tile writes only this thread's own slots, and the sort keys / permutation are rewritten
    //  behind its first barrier: no barrier needed here)
  }

  // ---- the block's record, the last block's solve: as in icp_iteration_body ----
  const double r = block_reduce_acc<NACC>(acc, sm);
  double* part = L.partials + (static_cast<size_t>(h) * L.part_stride) * kAccMax;
  if (threadIdx.x < NACC) __stcg(part + static_cast<size_t>(blk) * kAccMax + threadIdx.x, r);
  __threadfence();
  __syncthreads();
  __shared__ int s_last;
  if (threadIdx.x == 0) {
    const unsigned t = atomicAdd(&st->ticket, 1u);
    s_last = (t == static_cast<unsigned>(L.blocks_per_hyp) - 1u);
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  reduce_partials<NACC>(part, L.blocks_per_hyp, sm, sm_tot);
  if (threadIdx.x == 0) {
    finish_iteration<MB>(st, &L.crit, sm_tot, L.trace, L.trace_cap, nullptr);
    if (L.epochs) {
      const int still_active = st->active;
      __threadfence();
      atomicAdd(L.epochs + h, still_active ? 1 : kEpochStopped);
    }
  }
}

// ---- warm iterations over the k-NN graph with the unproven queries of a tile walked by dense warps -----------------
// In a graph launch (nn_graph.cuh) most queries are settled by the row of their previous match; the few that are not
// — points of the model that lie millimetres off the scene: 6 % of the queries of a late C4 iteration — walk the grid
// for a ball of several rows.  Inside icp_iteration_kernel such a lane keeps its whole warp waiting: ncu attributes half
// of the warp instructions AND half of the stall samples of a late launch to the walk, at 8 of 32 active lanes
// (profiles/r2_af_*).  Here every WARP takes a tile of TQ passes of the plain kernel's loop on its own (no block
// barrier: a first version that staged the tile of the whole block in shared memory behind __syncthreads lost 8 % —
// three warps idle while one walks):
//   1. every lane moves its TQ queries and tries the graph (grid_nn_graph_try); the moved point goes to the working
//      cloud at once with the best point met so far in .w (the match if proven); unproven queries (and those without
//      a previous match) are queued in the warp's shared-memory queue, and whenever 32 are waiting
//   2. the warp drains them, one per lane — a full warp that walks the grid (query and candidate are read back from
//      the working cloud; only the position in .w is rewritten);
//   3. a lane adds proven queries to its moment sums at once; a query that waits for a walk, and every later query of
//      the same lane and tile (the ORDER of a thread's sums is the plain kernel's), is taken up after the drain: point
//      and match re-read from the working cloud (L2), the squared distance recomputed with the same expression.
// MEASURED SLOWER, off by default ("warm_graph_queue"): 13 450 (tiles of 8 passes) and 13 310 (16) against 14 440
// hypotheses/s for the plain graph kernel on C4; putting off ALL queries of a tile instead: 14 130; the block-wide
// version: 13 280 (profiles/r2_ai_graph_queue.txt).  The walks it saves (a quarter of the warp-level walks are left)
// cost less than what it adds: the L2 round trips of the re-reads in phases 2 and 3, which nothing overlaps in a
// latency-bound kernel, and 330 more bytes of spills at the 64-register cap.
// Queries, exact searches (same tie rule) and the order of every thread's double sums are those of
// icp_iteration_kernel: byte-identical records (tests/test_gpu_warm_options.py).  Hypotheses that do not search over
// the graph in this launch (graph_pays) run the plain body.
template <int EST, int MB, int TQ>
__global__ void __launch_bounds__(kIcpThreads, MB) icp_iteration_graphq_kernel(const IcpLaunch L) {
  static_assert(TQ >= 1 && TQ <= 32, "one validity bit per pass of a tile");
  if (L.epochs == nullptr) {
    pdl_trigger_and_wait();
  } else {
    asm volatile("griddepcontrol.launch_dependents;");
    wait_for_hypothesis(L.epochs + blockIdx.y, L.launch_idx, L.err_flag);
  }
  const int h = blockIdx.y, blk = blockIdx.x;
  IcpState* st = L.states + h;
  __shared__ int s_mode[2];  // active, graph
  if (threadIdx.x == 0) {
    s_mode[0] = __ldcg(&st->active);
    s_mode[1] = graph_pays(L, st) ? 1 : 0;
  }
  __syncthreads();
  if (!s_mode[0]) return;
  if (!s_mode[1]) {  // (block-uniform)
    icp_iteration_body<1, EST, MB, false, false, 0>(L, h, blk);
    return;
  }
  constexpr int NACC = (EST == PEB_ESTIMATOR_SVD) ? kAccSvd : kAccLls;
  __shared__ double sm[kIcpThreads / 32][kAccMax];
  __shared__ double sm_tot[kAccMax];
  __shared__ float s_inc[16];
  __shared__ int s_queue[kIcpThreads / 32][64];  // per warp: query indices waiting for a grid walk (at most 31 + 32)
  if (threadIdx.x < 16) s_inc[threadIdx.x] = __ldcg(&st->inc.m[threadIdx.x]);
  __syncthreads();
  const float* T = s_inc;
  float4* work = L.work + static_cast<size_t>(h) * L.n_src;
  const int stride = L.blocks_per_hyp * kIcpThreads;
  const int lane = threadIdx.x & 31;
  const unsigned lt = (1u << lane) - 1u;
  int* queue = s_queue[threadIdx.x >> 5];

  // lanes [0, count) walk the grid for the LAST count entries of the queue
  auto drain = [&](int n_queue, int count) {
    if (lane < count) {
      const int i = queue[n_queue - count + lane];
      const float4 q = __ldcg(work + i);
      NnBest best;
      best.j = __float_as_int(q.w);
      if (best.j >= 0) {
        const float4 t = L.grid.pts[best.j];
        best.d2 = l2_simple(q.x, q.y, q.z, t.x, t.y, t.z);
        best.idx = point_index(t);
        grid_ball_search(L.grid, q.x, q.y, q.z, L.stop_d2, best);
      } else {
        best = grid_nn<1>(L.grid, q.x, q.y, q.z, L.stop_d2);
      }
      __stcg(reinterpret_cast<int*>(work + i) + 3, best.j);
    }
    __syncwarp();
  };

  double acc[NACC];
#pragma unroll
  for (int i = 0; i < NACC; ++i) acc[i] = 0.0;

  for (int base0 = blk * kIcpThreads; base0 < L.n_src; base0 += TQ * stride) {
    // ---- 1 (+ 2 whenever a warp's worth of walks is waiting): move, try the graph ----
    // A lane adds a proven query to its sums at once — unless one of its earlier queries of this tile is still
    // waiting for its walk: the order of a thread's sums is the plain kernel's, so everything behind a waiting
    // query waits with it (defer_mask) and is taken up again in phase 3.
    unsigned defer_mask = 0u;
    int n_queue = 0;  // (warp-uniform)
#pragma unroll 1
    for (int kk = 0; kk < TQ; ++kk) {
      const int i = base0 + kk * stride + threadIdx.x;
      if (i - lane >= L.n_src) break;  // (warp-uniform: the warp's first query of this pass)
      bool need = false;
      if (i < L.n_src) {
        float4 p = work[i];
        if (finite3(p.x, p.y, p.z)) {
          const int j_prev = __float_as_int(p.w);
          float qx, qy, qz;
          transform_icp(T, p.x, p.y, p.z, qx, qy, qz);
          p.x = qx;
          p.y = qy;
          p.z = qz;
          NnBest best;
          best.d2 = pos_inf();
          best.idx = -1;
          best.j = -1;
          need = true;
          if (j_prev >= 0 && j_prev < L.grid.n) need = !grid_nn_graph_try(L.grid, L.knn, qx, qy, qz, j_prev, best, kGraphSkipHopeless);
          p.w = __int_as_float(best.j);
          __stcg(work + i, p);
          if (need || defer_mask) {
            defer_mask |= 1u << kk;
          } else {
            bool keep = best.idx >= 0;
            if (keep && static_cast<double>(best.d2) > L.max_dist_sqr) keep = false;
            if (keep && L.use_rejector && !(best.d2 < L.rej_max2)) keep = false;
            if (keep) accumulate_pair<EST>(L.grid, p, best, acc);
          }
        }
      }
      const unsigned m = __ballot_sync(0xFFFFFFFFu, need);
      if (m) {
        if (need) queue[n_queue + __popc(m & lt)] = i;
        n_queue += __popc(m);
        __syncwarp();
        if (n_queue >= 32) {
          drain(n_queue, 32);
          n_queue -= 32;
        }
      }
    }
    if (n_queue) drain(n_queue, n_queue);
    // ---- 3: every lane the queries it had to put off, in the plain kernel's order ----
#pragma unroll 1
    for (int kk = 0; kk < TQ; ++kk) {
      if (!((defer_mask >> kk) & 1u)) continue;
      const int i = base0 + kk * stride + threadIdx.x;
      const float4 p = __ldcg(work + i);
      NnBest best;
      best.j = __float_as_int(p.w);
      if (best.j < 0) continue;  // nothing found within the search limit
      const float4 t = L.grid.pts[best.j];
      best.d2 = l2_simple(p.x, p.y, p.z, t.x, t.y, t.z);
      best.idx = point_index(t);
      bool keep = best.idx >= 0;
      if (keep && static_cast<double>(best.d2) > L.max_dist_sqr) keep = false;
      if (keep && L.use_rejector && !(best.d2 < L.rej_max2)) keep = false;
      if (keep) accumulate_pair<EST>(L.grid, p, best, acc);
    }
  }

  // ---- the block's record, the last block's solve: as in icp_iteration_body ----
  const double r = block_reduce_acc<NACC>(acc, sm);
  double* part = L.partials + (static_cast<size_t>(h) * L.part_stride) * kAccMax;
  if (threadIdx.x < NACC) __stcg(part + static_cast<size_t>(blk) * kAccMax + threadIdx.x, r);
  __threadfence();
  __syncthreads();
  __shared__ int s_last;
  if (threadIdx.x == 0) {
    const unsigned t = atomicAdd(&st->ticket, 1u);
    s_last = (t == static_cast<unsigned>(L.blocks_per_hyp) - 1u);
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  reduce_partials<NACC>(part, L.blocks_per_hyp, sm, sm_tot);
  if (threadIdx.x == 0) {
    finish_iteration<MB>(st, &L.crit, sm_tot, L.trace, L.trace_cap, nullptr);
    if (L.epochs) {
      const int still_active = st->active;
      __threadfence();
      atomicAdd(L.epochs + h, still_active ? 1 : kEpochStopped);
    }
  }
}

// ---- warm iterations with the candidate cache (nn_cache.cuh) -----------------------------------------------------
// Phase A, queries in rounds of one per thread: move the working point, try the certificate of its cache entry
// (kCacheK gathers, no grid walk, uniform over the warp).  Queries whose certificate fails are queued in shared memory
// and, every third round, collected again by DENSE warps — one queued query per thread, every lane busy with the same
// kind of fixed-radius search.  A query the ball of radius R finds nothing for (far from the scene) takes the plain warm
// search, as before.  Phase B: every thread accumulates ITS queries in the order of the plain kernel — working point and
// match re-read from the working cloud — so that the double sums, and with them every result, are bit-identical to the
// plain warm kernel's.
constexpr int kCacheRoundsPerFlush = 3;
constexpr int kCacheQueue = kIcpThreads * kCacheRoundsPerFlush;

__device__ __forceinline__ void cache_rebuild(const IcpLaunch& L, NnCache* __restrict__ cache, float4* __restrict__ work, int i) {
  float4 p = work[i];  // already moved; .w = the previous match
  const int j_prev = __float_as_int(p.w);
  NnTop top;
  grid_ball_collect(L.grid, p.x, p.y, p.z, L.cache_r_cells, top);
  NnCache ce = nn_cache_from_top(L.grid, p.x, p.y, p.z, L.cache_r_cells, top);
  int j = top.j[0];
  // the collection ranks everything in the cells it touched, but only the ball of radius R is covered completely: its
  // best point is the nearest neighbour only if it lies inside that ball
  if (j >= 0 && !(sqrtf(top.d2[0]) * (1.0f + 4e-6f) < L.cache_r_cells * L.grid.h)) j = -1;
  if (j < 0) {  // nothing within R: the plain search (its ball is the previous match's distance), no certificate
    NnBest best;
    if (j_prev >= 0 && j_prev < L.grid.n) best = grid_nn_warm(L.grid, p.x, p.y, p.z, j_prev, L.stop_d2);
    else best = grid_nn<1>(L.grid, p.x, p.y, p.z, L.stop_d2);
    j = best.j;
    ce.bound = 0.0f;
  }
  cache[i] = ce;
  p.w = __int_as_float(j);
  work[i] = p;
}

template <int EST, int MB>
__global__ void __launch_bounds__(kIcpThreads, MB) icp_iteration_cached_kernel(const IcpLaunch L) {
  if (L.epochs == nullptr) {
    pdl_trigger_and_wait();
  } else {
    asm volatile("griddepcontrol.launch_dependents;");
    wait_for_hypothesis(L.epochs + blockIdx.y, L.launch_idx, L.err_flag);
  }
  const int h = blockIdx.y, blk = blockIdx.x;
  constexpr int NACC = (EST == PEB_ESTIMATOR_SVD) ? kAccSvd : kAccLls;
  __shared__ double sm[kIcpThreads / 32][kAccMax];
  __shared__ double sm_tot[kAccMax];
  __shared__ float s_inc[16];
  __shared__ int s_active;
  __shared__ int s_queue[kCacheQueue];
  __shared__ int s_qn;
  IcpState* st = L.states + h;
  if (threadIdx.x < 16) s_inc[threadIdx.x] = __ldcg(&st->inc.m[threadIdx.x]);
  if (threadIdx.x == 32) {
    s_active = __ldcg(&st->active);
    s_qn = 0;
  }
  __syncthreads();
  if (!s_active) return;
  const float* T = s_inc;
  float4* work = L.work + static_cast<size_t>(h) * L.n_src;
  NnCache* cache = L.cache + static_cast<size_t>(h) * L.n_src;
  const int stride = L.blocks_per_hyp * kIcpThreads;

  // ---- phase A: nearest neighbours ----
  int round = 0;
  for (int base = blk * kIcpThreads; base < L.n_src; base += stride, ++round) {
    const int i = base + threadIdx.x;
    bool pending = false;
    if (i < L.n_src) {
      float4 p = work[i];
      if (finite3(p.x, p.y, p.z)) {
        float ox, oy, oz;
        transform_icp(T, p.x, p.y, p.z, ox, oy, oz);
        p.x = ox;
        p.y = oy;
        p.z = oz;
        NnBest best;
        if (!L.cache_init && nn_cache_lookup(L.grid, cache[i], p.x, p.y, p.z, best)) p.w = __int_as_float(best.j);
        else pending = true;
        work[i] = p;  // (a pending query keeps its previous match in .w until it is collected again)
      }
    }
    const unsigned mask = __ballot_sync(0xFFFFFFFFu, pending);
    if (mask) {
      const int lane = threadIdx.x & 31;
      int at = 0;
      if (lane == 0) at = atomicAdd(&s_qn, __popc(mask));
      at = __shfl_sync(0xFFFFFFFFu, at, 0);
      if (pending) s_queue[at + __popc(mask & ((1u << lane) - 1u))] = i;
    }
    const bool last = base + stride >= L.n_src;
    if (round % kCacheRoundsPerFlush == kCacheRoundsPerFlush - 1 || last) {
      __syncthreads();
      const int qn = s_qn;
      for (int k = threadIdx.x; k < qn; k += kIcpThreads) cache_rebuild(L, cache, work, s_queue[k]);
      __syncthreads();
      if (threadIdx.x == 0) s_qn = 0;
      // (the next push is separated from this reset by the ballot of the next round only: make it visible first)
      __syncthreads();
    }
  }

  // ---- phase B: thresholds and moments, every thread its own queries in order ----
  double acc[NACC];
#pragma unroll
  for (int i = 0; i < NACC; ++i) acc[i] = 0.0;
  for (int base = blk * kIcpThreads; base < L.n_src; base += stride) {
    const int i = base + threadIdx.x;
    if (i >= L.n_src) continue;
    const float4 p = work[i];
    const bool valid = finite3(p.x, p.y, p.z);
    const int j = __float_as_int(p.w);
    NnBest best;
    best.d2 = pos_inf();
    best.idx = -1;
    best.j = -1;
    if (valid && j >= 0) {
      const float4 t = L.grid.pts[j];
      best.d2 = l2_simple(p.x, p.y, p.z, t.x, t.y, t.z);
      best.idx = __float_as_int(t.w);
      best.j = j;
    }
    bool keep = valid && best.idx >= 0;
    if (keep && static_cast<double>(best.d2) > L.max_dist_sqr) keep = false;
    if (keep && L.use_rejector && !(best.d2 < L.rej_max2)) keep = false;
    if (L.corr_idx) {
      const int orig = __float_as_int(L.src[i].w);
      L.corr_idx[orig] = keep ? best.idx : -1;
      L.corr_d2[orig] = keep ? best.d2 : 0.0f;
    }
    if (keep) accumulate_pair<EST>(L.grid, p, best, acc);
  }

  // ---- the block's record, the last block's solve: as in icp_iteration_body ----
  const double r = block_reduce_acc<NACC>(acc, sm);
  double* part = L.partials + (static_cast<size_t>(h) * L.part_stride) * kAccMax;
  if (threadIdx.x < NACC) __stcg(part + static_cast<size_t>(blk) * kAccMax + threadIdx.x, r);
  __threadfence();
  __syncthreads();
  __shared__ int s_last;
  if (threadIdx.x == 0) {
    const unsigned t = atomicAdd(&st->ticket, 1u);
    s_last = (t == static_cast<unsigned>(L.blocks_per_hyp) - 1u);
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  reduce_partials<NACC>(part, L.blocks_per_hyp, sm, sm_tot);
  if (threadIdx.x == 0) {
    finish_iteration<MB>(st, &L.crit, sm_tot, L.trace, L.trace_cap, nullptr);
    if (L.epochs) {
      const int still_active = st->active;
      __threadfence();
      atomicAdd(L.epochs + h, still_active ? 1 : kEpochStopped);
    }
  }
}

// [PCL] registration/impl/registration.hpp : getFitnessScore(max_range) with the final transform
// applied by pcl::transformPointCloud's association (transform_tpc), then the result record.
template <int G>
__global__ void __launch_bounds__(kIcpThreads) icp_fitness_kernel(const IcpLaunch L) {
  __shared__ double sm[kIcpThreads / 32][kAccMax];
  __shared__ double sm_tot[kAccMax];
  if (L.epochs == nullptr) {
    pdl_trigger_and_wait();
  } else {  // only the last iteration of THIS hypothesis is needed (L.launch_idx = number of iteration launches)
    asm volatile("griddepcontrol.launch_dependents;");
    wait_for_hypothesis(L.epochs + blockIdx.y, L.launch_idx, L.err_flag);
  }
  const int h = blockIdx.y;
  IcpState* st = L.states + h;
  float T[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) T[i] = __ldcg(&st->final_t.m[i]);
  const bool graph = G == 1 && graph_pays(L, st);  // (uniform over the block)
  double acc[2] = {0.0, 0.0};
  const int lane_in_group = threadIdx.x & (G - 1);
  constexpr int kQ = kIcpThreads / G;
  const int q_local = threadIdx.x / G;
  for (int base = blockIdx.x * kQ; base < L.n_src; base += L.blocks_per_hyp * kQ) {
    const int i = base + q_local;
    float4 p = make_float4(0.f, 0.f, 0.f, 1.f);
    if (i < L.n_src) p = L.src[i];
    const bool valid = i < L.n_src && finite3(p.x, p.y, p.z);
    NnBest best;
    best.d2 = pos_inf();
    best.idx = -1;
    best.j = -1;
    if (valid) {
      float qx, qy, qz;
      transform_tpc(T, p.x, p.y, p.z, qx, qy, qz);
      int j_prev = -1;
      float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
      if (G == 1 && L.warm) {
        w = L.work[static_cast<size_t>(h) * L.n_src + i];
        j_prev = __float_as_int(w.w);
      }
      if (G == 1 && j_prev >= 0 && j_prev < L.grid.n) {
        // the working point sits where the last search ran; the fitness query is that point after
        // the last increment (and pcl::transformPointCloud's rounding)
        float slack = -1.0f;
        if (L.margin > 0.0f) {
          const float mx = qx - w.x, my = qy - w.y, mz = qz - w.z;
          const float moved = sqrtf(mx * mx + my * my + mz * mz);
          slack = L.slack[static_cast<size_t>(h) * L.n_src + i] - 2.000002f * moved - 1e-5f * L.grid.h;
        }
        if (slack > 0.0f) {
          const float4 t = L.grid.pts[j_prev];
          best.d2 = l2_simple(qx, qy, qz, t.x, t.y, t.z);
          best.idx = __float_as_int(t.w);
          best.j = j_prev;
        } else {
          best = graph ? grid_nn_warm_graph(L.grid, L.knn, qx, qy, qz, j_prev, L.fitness_stop_d2, kGraphSkipHopeless)
                       : grid_nn_warm(L.grid, qx, qy, qz, j_prev, L.fitness_stop_d2);
        }
      } else {
        best = grid_nn<G>(L.grid, qx, qy, qz, L.fitness_stop_d2);
      }
    }
    if (valid && best.idx >= 0 && lane_in_group == 0 && static_cast<double>(best.d2) <= L.fitness_max_range) {
      acc[0] += static_cast<double>(best.d2);
      acc[1] += 1.0;
    }
  }
  const double r = block_reduce_acc<2>(acc, sm);
  double* part = L.partials + (static_cast<size_t>(h) * L.part_stride) * kAccMax;
  if (threadIdx.x < 2) __stcg(part + static_cast<size_t>(blockIdx.x) * kAccMax + threadIdx.x, r);
  __threadfence();
  __syncthreads();
  __shared__ int s_last;
  if (threadIdx.x == 0) {
    const unsigned t = atomicAdd(&st->ticket_fit, 1u);
    s_last = (t == static_cast<unsigned>(L.blocks_per_hyp) - 1u);
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  reduce_partials<2>(part, L.blocks_per_hyp, sm, sm_tot);
  if (threadIdx.x == 0) {
    IcpState s = *st;
    s.fit_sum = sm_tot[0];
    s.fit_n = static_cast<int>(sm_tot[1]);
    s.ticket_fit = 0;
    *st = s;
    peb_icp_result res;
#pragma unroll
    for (int i = 0; i < 16; ++i) res.T[i] = s.final_t.m[i];
    res.fitness = s.fit_n > 0 ? s.fit_sum / static_cast<double>(s.fit_n) : DBL_MAX;
    res.last_mse = s.cur_mse;
    res.iterations = s.iterations;
    res.converged = s.converged;
    res.state = s.state;
    res.n_correspondences = L.fitness_only ? s.fit_n : s.ncorr;
    if (L.err_flag && __ldcg(L.err_flag) != 0) res.state = PEB_STATE_INTERNAL_ERROR;  // a dependency wait hit its bound
    L.results[h] = res;
  }
}

// output = final * input ([PCL] icp.hpp: transformCloud(*input_, output, final_transformation_))
__global__ void __launch_bounds__(256) icp_output_kernel(const float4* __restrict__ src, int n,
                                                         const IcpState* __restrict__ st, float4* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float T[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) T[k] = __ldg(&st->final_t.m[k]);
  float4 p = src[i];
  if (finite3(p.x, p.y, p.z)) {
    float ox, oy, oz;
    transform_icp(T, p.x, p.y, p.z, ox, oy, oz);
    p.x = ox;
    p.y = oy;
    p.z = oz;
  }
  p.w = 1.0f;
  out[i] = p;
}

template <int G>
__global__ void __launch_bounds__(256) nn_search_kernel(const GridView g, const float4* __restrict__ q, int nq,
                                                        int32_t* __restrict__ out_idx, float* __restrict__ out_d2) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) / G;
  const int lane_in_group = threadIdx.x & (G - 1);
  float4 p = make_float4(0.f, 0.f, 0.f, 0.f);
  if (i < nq) p = q[i];
  const bool valid = i < nq && finite3(p.x, p.y, p.z);
  NnBest best;
  best.d2 = pos_inf();
  best.idx = -1;
  best.j = -1;
  if (valid) best = grid_nn<G>(g, p.x, p.y, p.z, pos_inf());
  if (i < nq && lane_in_group == 0) {
    out_idx[i] = best.idx;
    out_d2[i] = best.d2;
  }
}

float stop_bound(double max_dist_sqr) {
  // smallest float that is >= max_dist_sqr (so that nothing acceptable is cut off), inf if it does not fit
  if (!(max_dist_sqr < static_cast<double>(FLT_MAX))) return INFINITY;
  if (max_dist_sqr < 0.0) return 0.0f;
  float f = static_cast<float>(max_dist_sqr);
  if (static_cast<double>(f) < max_dist_sqr) f = nextafterf(f, INFINITY);
  return f;
}

int prof_mark(peb_ctx* ctx, int slot) {
  if (!ctx->profile) return PEB_OK;
  while (static_cast<int>(ctx->prof_events.size()) <= slot) {
    cudaEvent_t e;
    PEB_CUDA(ctx, cudaEventCreate(&e));
    ctx->prof_events.push_back(e);
  }
  PEB_CUDA(ctx, cudaEventRecord(ctx->prof_events[slot], ctx->stream));
  return PEB_OK;
}

// Does this iteration launch run as a search launch and a moment launch?  Batched aligns with one lane per query on
// their default paths: launch 0, the warm launches over the k-NN graph (with or without the flatness certificate) and
// the plain warm launches.  The single align (latency-bound per launch: one more launch per iteration would cost it),
// the certificates, the debug timers and the experimental variants keep the fused kernel.
bool split_iteration(const peb_ctx* ctx, const IcpLaunch& L, size_t H, int G, bool first) {
  if (!ctx->split_moments || H < static_cast<size_t>(ctx->split_min_hyp) || H <= 1 || G != 1 || L.margin > 0.0f || L.dbg ||
      L.corr_idx)
    return false;
  if (first) return true;
  if (L.cache || (ctx->warm_upfront && L.warm && L.launch_idx >= ctx->warm_upfront_from)) return false;
  if (L.warm && L.knn) return ctx->warm_graph_queue == 0;
  return !(L.warm && ctx->warm_bin);
}

// R: the align's rejector chain (nullable): a reject launch between the two, and the moments of the kept pairs
template <bool FIRST>
int launch_split_iteration(peb_ctx* ctx, const IcpLaunch& L, size_t H, int estimator, int search_bph, const RejChain* R) {
  const dim3 sgrid(search_bph, static_cast<unsigned>(H)), mgrid(L.blocks_per_hyp, static_cast<unsigned>(H));
  // (launch 0 keeps the batched cap: its cooperative verification holds more state than a warm search)
  if (FIRST)
    PEB_LAUNCH_PDL(ctx, (icp_search_kernel<kMinBlocksBatch, true, 0>), sgrid, dim3(kIcpThreads), L);
  else if (L.warm && L.knn && L.knn_aux && L.launch_idx >= ctx->warm_graph_flat_from && L.launch_idx <= ctx->warm_graph_flat_until)
    PEB_LAUNCH_PDL(ctx, (icp_search_kernel<kMinBlocksSearch, false, 6>), sgrid, dim3(kIcpThreads), L);
  else if (L.warm && L.knn)
    PEB_LAUNCH_PDL(ctx, (icp_search_kernel<kMinBlocksSearch, false, 4>), sgrid, dim3(kIcpThreads), L);
  else
    PEB_LAUNCH_PDL(ctx, (icp_search_kernel<kMinBlocksSearch, false, 0>), sgrid, dim3(kIcpThreads), L);
  if (R) {
    PEB_LAUNCH_PDL(ctx, icp_reject_kernel, dim3(static_cast<unsigned>(H)), dim3(kRejThreads), L, *R);
    const unsigned char* kept = R->kept;
    if (estimator == PEB_ESTIMATOR_SVD)
      PEB_LAUNCH_PDL(ctx, (icp_moment_kernel<PEB_ESTIMATOR_SVD, kMinBlocksBatch, true>), mgrid, dim3(kIcpThreads), L, kept);
    else
      PEB_LAUNCH_PDL(ctx, (icp_moment_kernel<PEB_ESTIMATOR_POINT_TO_PLANE_LLS, kMinBlocksBatch, true>), mgrid, dim3(kIcpThreads), L, kept);
    return PEB_OK;
  }
  const unsigned char* none = nullptr;
  if (estimator == PEB_ESTIMATOR_SVD)
    PEB_LAUNCH_PDL(ctx, (icp_moment_kernel<PEB_ESTIMATOR_SVD, kMinBlocksBatch, false>), mgrid, dim3(kIcpThreads), L, none);
  else
    PEB_LAUNCH_PDL(ctx, (icp_moment_kernel<PEB_ESTIMATOR_POINT_TO_PLANE_LLS, kMinBlocksBatch, false>), mgrid, dim3(kIcpThreads), L, none);
  return PEB_OK;
}

// search_bph > 0: the iteration runs split, with this many search blocks per hypothesis
template <int G, bool FIRST>
int launch_one_iteration(peb_ctx* ctx, const IcpLaunch& L, size_t H, int estimator, int search_bph, const RejChain* R) {
  if (G == 1 && search_bph > 0) return launch_split_iteration<FIRST>(ctx, L, H, estimator, search_bph, R);
  dim3 grid(L.blocks_per_hyp, static_cast<unsigned>(H));
  constexpr int S = PEB_ESTIMATOR_SVD, P = PEB_ESTIMATOR_POINT_TO_PLANE_LLS;
  const bool cert = G == 1 && L.margin > 0.0f;
  const bool svd = estimator == PEB_ESTIMATOR_SVD;
#define PEB_ICP_LAUNCH(EST, MB, CERT) \
  PEB_LAUNCH_PDL(ctx, (icp_iteration_kernel<G, EST, MB, CERT, FIRST>), grid, dim3(kIcpThreads), L)
  // experimental warm search (peb_ctx_set_int "warm_upfront"); the first warm launches search balls of more than a cell
  // (the first ICP step moves the points by millimetres) and keep the narrowing walk ("warm_upfront_from", default 2)
  if (G == 1 && !FIRST && !cert && ctx->warm_upfront && L.warm && L.launch_idx >= ctx->warm_upfront_from) {
#define PEB_ICP_LAUNCH_UPF(EST, MB, RW) \
  PEB_LAUNCH_PDL(ctx, (icp_iteration_kernel<1, EST, MB, false, false, RW>), grid, dim3(kIcpThreads), L)
    if (ctx->warm_upfront == 3) {
      if (H == 1) { if (svd) PEB_ICP_LAUNCH_UPF(S, kMinBlocksSingle, 3); else PEB_ICP_LAUNCH_UPF(P, kMinBlocksSingle, 3); }
      else        { if (svd) PEB_ICP_LAUNCH_UPF(S, kMinBlocksBatch, 3);  else PEB_ICP_LAUNCH_UPF(P, kMinBlocksBatch, 3); }
    } else {
      if (H == 1) { if (svd) PEB_ICP_LAUNCH_UPF(S, kMinBlocksSingle, 2); else PEB_ICP_LAUNCH_UPF(P, kMinBlocksSingle, 2); }
      else        { if (svd) PEB_ICP_LAUNCH_UPF(S, kMinBlocksBatch, 2);  else PEB_ICP_LAUNCH_UPF(P, kMinBlocksBatch, 2); }
    }
#undef PEB_ICP_LAUNCH_UPF
    return PEB_OK;
  }
  // warm launches of a batch over the target's k-NN graph (nn_graph.cuh; "warm_graph")
  if (G == 1 && !FIRST && !cert && !L.cache && L.warm && L.knn && H > 1) {
    // ... with the unproven queries of a tile queued and walked by dense warps ("warm_graph_queue" = passes per tile)
#define PEB_ICP_LAUNCH_GQ(TQ) \
  do { \
    if (svd) PEB_LAUNCH_PDL(ctx, (icp_iteration_graphq_kernel<S, kMinBlocksBatch, TQ>), grid, dim3(kIcpThreads), L); \
    else     PEB_LAUNCH_PDL(ctx, (icp_iteration_graphq_kernel<P, kMinBlocksBatch, TQ>), grid, dim3(kIcpThreads), L); \
  } while (0)
    if (ctx->warm_graph_queue == 8) { PEB_ICP_LAUNCH_GQ(8); return PEB_OK; }
    if (ctx->warm_graph_queue == 16) { PEB_ICP_LAUNCH_GQ(16); return PEB_OK; }
#undef PEB_ICP_LAUNCH_GQ
    // ... with the flatness certificate in the launches where the queries are still beyond the plain one ("warm_graph_flat_from"
    // .. "warm_graph_flat_until"; later the plain certificate settles nearly everything and the extra record only costs)
    if (L.knn_aux && L.launch_idx >= ctx->warm_graph_flat_from && L.launch_idx <= ctx->warm_graph_flat_until) {
      if (svd) PEB_LAUNCH_PDL(ctx, (icp_iteration_kernel<1, S, kMinBlocksBatch, false, false, 6>), grid, dim3(kIcpThreads), L);
      else     PEB_LAUNCH_PDL(ctx, (icp_iteration_kernel<1, P, kMinBlocksBatch, false, false, 6>), grid, dim3(kIcpThreads), L);
      return PEB_OK;
    }
    if (svd) PEB_LAUNCH_PDL(ctx, (icp_iteration_kernel<1, S, kMinBlocksBatch, false, false, 4>), grid, dim3(kIcpThreads), L);
    else     PEB_LAUNCH_PDL(ctx, (icp_iteration_kernel<1, P, kMinBlocksBatch, false, false, 4>), grid, dim3(kIcpThreads), L);
    return PEB_OK;
  }
  // warm launches of a batch with the queries of a block binned by the size of their search ("warm_bin")
  if (G == 1 && !FIRST && !cert && !L.cache && L.warm && ctx->warm_bin && H > 1) {
    if (svd) PEB_LAUNCH_PDL(ctx, (icp_iteration_binned_kernel<S, kMinBlocksBatch>), grid, dim3(kIcpThreads), L);
    else     PEB_LAUNCH_PDL(ctx, (icp_iteration_binned_kernel<P, kMinBlocksBatch>), grid, dim3(kIcpThreads), L);
    return PEB_OK;
  }
  // warm launches with the candidate cache (nn_cache.cuh; peb_ctx_set_int "nn_cache_from")
  if (G == 1 && !FIRST && !cert && L.cache && L.warm) {
#define PEB_ICP_LAUNCH_CACHED(EST, MB) \
  PEB_LAUNCH_PDL(ctx, (icp_iteration_cached_kernel<EST, MB>), grid, dim3(kIcpThreads), L)
    if (H == 1) { if (svd) PEB_ICP_LAUNCH_CACHED(S, kMinBlocksSingle); else PEB_ICP_LAUNCH_CACHED(P, kMinBlocksSingle); }
    else        { if (svd) PEB_ICP_LAUNCH_CACHED(S, kMinBlocksBatch);  else PEB_ICP_LAUNCH_CACHED(P, kMinBlocksBatch); }
#undef PEB_ICP_LAUNCH_CACHED
    return PEB_OK;
  }
  if (H == 1) {
    if (cert) { if (svd) PEB_ICP_LAUNCH(S, kMinBlocksSingle, (G == 1)); else PEB_ICP_LAUNCH(P, kMinBlocksSingle, (G == 1)); }
    else      { if (svd) PEB_ICP_LAUNCH(S, kMinBlocksSingle, false);    else PEB_ICP_LAUNCH(P, kMinBlocksSingle, false); }
  } else {
    if (cert) { if (svd) PEB_ICP_LAUNCH(S, kMinBlocksBatch, (G == 1)); else PEB_ICP_LAUNCH(P, kMinBlocksBatch, (G == 1)); }
    else      { if (svd) PEB_ICP_LAUNCH(S, kMinBlocksBatch, false);    else PEB_ICP_LAUNCH(P, kMinBlocksBatch, false); }
  }
#undef PEB_ICP_LAUNCH
  return PEB_OK;
}

// first: launch 0 of the align
// R (nullable): the rejector chain; it comes with G = 1 and search_bph > 0
int launch_one_iteration_g(peb_ctx* ctx, int G, bool first, const IcpLaunch& L, size_t H, int estimator, int search_bph,
                           const RejChain* R = nullptr) {
#define PEB_ICP_G(GG) return first ? launch_one_iteration<GG, true>(ctx, L, H, estimator, search_bph, R) : launch_one_iteration<GG, false>(ctx, L, H, estimator, search_bph, R)
  switch (G) {
    case 1: PEB_ICP_G(1);
    case 2: PEB_ICP_G(2);
    case 4: PEB_ICP_G(4);
    case 8: PEB_ICP_G(8);
    case 16: PEB_ICP_G(16);
    default: return fail(ctx, PEB_E_INVALID_ARG, "nn group width %d is not one of 1,2,4,8,16", G);
  }
#undef PEB_ICP_G
}

int launch_fitness_g(peb_ctx* ctx, int G, const IcpLaunch& L, size_t H) {
  dim3 grid(L.blocks_per_hyp, static_cast<unsigned>(H));
  switch (G) {
    case 1: PEB_LAUNCH_PDL(ctx, icp_fitness_kernel<1>, grid, dim3(kIcpThreads), L); break;
    case 2: PEB_LAUNCH_PDL(ctx, icp_fitness_kernel<2>, grid, dim3(kIcpThreads), L); break;
    case 4: PEB_LAUNCH_PDL(ctx, icp_fitness_kernel<4>, grid, dim3(kIcpThreads), L); break;
    case 8: PEB_LAUNCH_PDL(ctx, icp_fitness_kernel<8>, grid, dim3(kIcpThreads), L); break;
    default: PEB_LAUNCH_PDL(ctx, icp_fitness_kernel<16>, grid, dim3(kIcpThreads), L); break;
  }
  return PEB_OK;
}

// blocks per hypothesis for a group width: one block handles kIcpThreads / G queries per pass;
// a single align spreads over the whole chip, batched aligns give every hypothesis a few blocks
// and let grid.y fill the machine
// factor = blocks per SM and launch, summed over all hypotheses.  0 = measured defaults (B200, C4):
// a block pays a fixed cost (state load, 17-value reduction, ticket), so fewer and larger blocks win as long
// as the launch tails are hidden (chains, per-hypothesis dependencies); small batches need enough blocks to fill the machine
int blocks_for(int n, size_t H, int G, int factor) {
  if (factor <= 0) factor = H >= 256 ? 32 : 16;  // (with per-hypothesis launch dependencies: 1024 hypotheses 89.2 ms at 24-32, 90.6 at 64)
  const int want = ceil_div(std::max(n, 1), kIcpThreads / G);
  int bph;
  if (H == 1)
    bph = std::min(want, kSmCount * 8);
  else
    bph = std::min(want, std::max(1, static_cast<int>((static_cast<size_t>(kSmCount) * factor + H - 1) / H)));
  return std::max(bph, 1);
}

// launch 0: its blocks differ a lot (patches whose common region holds hundreds of rows next to patches that hold ten), so it
// keeps the finer blocks also for small batches — a 128-hypothesis shard: 9.17 -> 9.07 ms with 32 instead of 16 per SM
int cold_blocks_factor(const peb_ctx* ctx) {
  return ctx->blocks_factor_cold > 0 ? ctx->blocks_factor_cold : (ctx->blocks_factor > 0 ? ctx->blocks_factor : 32);
}

}  // namespace

namespace {

// fills everything of the launch record that does not depend on the mode
int prepare_launch(peb_ctx* ctx, size_t H, const peb_icp_params* prm, IcpLaunch& L) {
  const int n = ctx->n_src_sorted;
  L.grid = ctx->tgt_grid.view;
  L.seed_guard2 = ctx->seed_guard * ctx->seed_guard;
  L.coop_max_rows = ctx->coop_max_rows;
  L.src = ctx->src_grid.view.pts;
  L.n_src = n;
  const int max_bph = std::max({blocks_for(n, H, ctx->nn_group, ctx->blocks_factor), blocks_for(n, H, 1, ctx->blocks_factor),
                                blocks_for(n, H, ctx->nn_group, cold_blocks_factor(ctx)), blocks_for(n, H, 1, cold_blocks_factor(ctx))});
  PEB_CUDA(ctx, ctx->work.ensure(std::max<size_t>(H * static_cast<size_t>(n), 1) * sizeof(float4)));
  PEB_CUDA(ctx, ctx->slack.ensure(std::max<size_t>(H * static_cast<size_t>(n), 1) * sizeof(float)));
  PEB_CUDA(ctx, ctx->state.ensure(H * sizeof(IcpState)));
  PEB_CUDA(ctx, ctx->partials.ensure(H * static_cast<size_t>(max_bph) * kAccMax * sizeof(double)));
  L.work = ctx->work.as<float4>();
  L.slack = ctx->slack.as<float>();
  L.margin = ctx->cert_margin * L.grid.h;
  L.states = ctx->state.as<IcpState>();
  L.partials = ctx->partials.as<double>();
  L.part_stride = max_bph;
  L.crit.max_iterations = prm->max_iterations;
  L.crit.min_correspondences = prm->min_correspondences;
  L.crit.max_similar = prm->max_iterations_similar;
  L.crit.estimator = prm->estimator;
  L.crit.mse_abs = prm->abs_mse_threshold;
  L.crit.mse_rel = prm->euclidean_fitness_epsilon;
  L.crit.translation_threshold = prm->transformation_epsilon;
  L.crit.rotation_threshold = prm->rotation_epsilon > 0 ? prm->rotation_epsilon : 1.0 - prm->transformation_epsilon;
  L.max_dist_sqr = prm->max_corr_dist * prm->max_corr_dist;
  L.use_rejector = prm->rejector_max_dist > 0 ? 1 : 0;
  L.rej_max2 = static_cast<float>(prm->rejector_max_dist * prm->rejector_max_dist);
  float stop = stop_bound(L.max_dist_sqr);
  if (L.use_rejector) stop = fminf(stop, L.rej_max2);
  L.stop_d2 = stop;
  L.fitness_max_range = prm->fitness_max_range;
  L.fitness_stop_d2 = stop_bound(prm->fitness_max_range);
  return PEB_OK;
}

}  // namespace

namespace {
int ensure_sub_streams(peb_ctx* ctx, int S) {
  while (static_cast<int>(ctx->sub_streams.size()) < S) {
    cudaStream_t st;
    cudaEvent_t ev;
    PEB_CUDA(ctx, cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    PEB_CUDA(ctx, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    ctx->sub_streams.push_back(st);
    ctx->join_events.push_back(ev);
  }
  if (!ctx->fork_event) PEB_CUDA(ctx, cudaEventCreateWithFlags(&ctx->fork_event, cudaEventDisableTiming));
  return PEB_OK;
}
}  // namespace

int icp_align_device(peb_ctx* ctx, const float* d_guesses, size_t H, const peb_icp_params* prm,
                     peb_icp_result* d_results, bool single_mode, const peb_rejector* chain, int n_chain) {
  if (!ctx->tgt_grid.valid) return fail(ctx, PEB_E_NO_TARGET, "align: no target set (peb_target_set)");
  if (!ctx->src_set) return fail(ctx, PEB_E_NO_SOURCE, "align: no source set (peb_source_set)");
  if (H == 0) return PEB_OK;
  if (prm->max_iterations < 0) return fail(ctx, PEB_E_INVALID_ARG, "align: max_iterations < 0");
  if (prm->estimator != PEB_ESTIMATOR_SVD && prm->estimator != PEB_ESTIMATOR_POINT_TO_PLANE_LLS)
    return fail(ctx, PEB_E_UNSUPPORTED, "align: unknown estimator %d (no CPU fallback)", prm->estimator);
  if (prm->estimator == PEB_ESTIMATOR_POINT_TO_PLANE_LLS && !ctx->tgt_has_normals)
    return fail(ctx, PEB_E_INVALID_ARG, "align: point-to-plane needs target normals (peb_target_set normals)");
  const int n = ctx->n_src_sorted;
  const int n_all = static_cast<int>(ctx->n_src);
  IcpLaunch L{};
  PEB_TRY(prepare_launch(ctx, H, prm, L));
  L.results = d_results;
  // a rejector chain (icp_reject_kernel): every iteration split, one lane per query, no certificate, no cache
  const bool with_chain = n_chain > 0;
  RejChain R{};
  if (with_chain) {
    L.margin = 0.0f;
    R.n = n_chain;
    bool o2o = false;
    for (int s = 0; s < n_chain; ++s) {
      R.kind[s] = chain[s].kind;
      R.min_corr[s] = chain[s].min_correspondences;
      R.value[s] = chain[s].value;
      o2o = o2o || chain[s].kind == PEB_REJECTOR_ONE_TO_ONE;
    }
    PEB_CUDA(ctx, ctx->rej_kept.ensure(std::max<size_t>(H * static_cast<size_t>(n), 1)));
    R.kept = ctx->rej_kept.as<unsigned char>();
    if (o2o) {
      const size_t bytes = std::max<size_t>(H * static_cast<size_t>(L.grid.n), 1) * sizeof(unsigned long long);
      const size_t cap0 = ctx->rej_o2o.cap;
      const cudaError_t e = ctx->rej_o2o.ensure(bytes);
      if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, PEB_E_OOM, "align: the one-to-one rejector's table of %zu hypotheses x %d target points (%.2f GB) "
                    "could not be allocated: %s", H, L.grid.n, static_cast<double>(bytes) / 1e9, cudaGetErrorString(e));
      }
      // all ones when allocated; every stage leaves it so (icp_reject_kernel)
      if (ctx->rej_o2o.cap != cap0 || !ctx->rej_o2o_clean)
        PEB_CUDA(ctx, cudaMemsetAsync(ctx->rej_o2o.p, 0xFF, ctx->rej_o2o.cap, ctx->stream));
      ctx->rej_o2o_clean = false;  // (set again once every launch of this align is queued)
      R.o2o = ctx->rej_o2o.as<unsigned long long>();
    }
  }
  if (single_mode) {
    PEB_CUDA(ctx, ctx->corr_idx.ensure(std::max(n_all, 1) * sizeof(int32_t)));
    PEB_CUDA(ctx, ctx->corr_d2.ensure(std::max(n_all, 1) * sizeof(float)));
    // non-finite source points never take part: they stay "no correspondence"
    PEB_CUDA(ctx, cudaMemsetAsync(ctx->corr_idx.p, 0xFF, std::max(n_all, 1) * sizeof(int32_t), ctx->stream));
    PEB_CUDA(ctx, cudaMemsetAsync(ctx->corr_d2.p, 0, std::max(n_all, 1) * sizeof(float), ctx->stream));
    const int cap = std::max(prm->max_iterations, 1);
    PEB_CUDA(ctx, ctx->trace.ensure(static_cast<size_t>(cap) * sizeof(Mat4)));
    L.corr_idx = ctx->corr_idx.as<int32_t>();
    L.corr_d2 = ctx->corr_d2.as<float>();
    L.trace = ctx->trace.as<Mat4>();
    L.trace_cap = cap;
    ctx->last_trace_cap = cap;
  }
  const int g_cold = with_chain ? 1 : ctx->nn_group;
  const int g_warm = ctx->warm_start ? 1 : g_cold;
  const bool per_launch = ctx->profile_level >= 2;
  const int launches = std::max(prm->max_iterations, 1);  // PCL runs the loop body at least once (do ... while)
  // Per-hypothesis dependencies between the iteration launches (see icp_iteration_kernel): needs PDL, and
  // nothing between the launches (profile level 2 and the debug timers put events there)
  // (not for a single align or a handful of hypotheses: hundreds of blocks polling one flag slow down the
  //  one thread everybody waits for — measured 0.74 -> 0.78 ms on C2)
  const bool flag_deps = !with_chain && ctx->flag_deps && ctx->use_pdl && !per_launch && !ctx->debug_timers && !single_mode && H >= 16 &&
                         launches < kEpochStopped;
  ctx->last_err_flag = nullptr;
  if (flag_deps) {
    PEB_CUDA(ctx, ctx->epochs.ensure((H + 1) * sizeof(int)));
    L.epochs = ctx->epochs.as<int>();
    L.err_flag = L.epochs + H;
    ctx->last_err_flag = L.err_flag;
  }
  PEB_LAUNCH(ctx, icp_init_kernel, ceil_div(static_cast<long long>(H + 1), 128), 128, 0, L.states, d_guesses,
             static_cast<int>(H), L.epochs);
  if (L.margin > 0.0f)  // no certificate yet (all-ones = NaN: never > 0)
    PEB_CUDA(ctx, cudaMemsetAsync(L.slack, 0xFF, std::max<size_t>(H * static_cast<size_t>(n), 1) * sizeof(float), ctx->stream));
  IcpLaunch Lc = L, Lw = L;
  // launch 0 costs several warm launches and its blocks differ a lot: finer blocks keep the machine even
  Lc.blocks_per_hyp = blocks_for(n, H, g_cold, cold_blocks_factor(ctx));
  Lc.warm = 0;
  // (a single align has too few patches to fill the machine with anchor searches: their latency
  //  would exceed what the seeds save; its cold launch keeps the plain ring search)
  if (ctx->warm_start && ctx->anchor_seed && g_cold == 1 && n >= 64 && H * static_cast<size_t>(n) >= (1u << 20) && H <= 65535) {
    const int n_anchor = ceil_div(n, 32);
    PEB_CUDA(ctx, ctx->anchors.ensure(H * static_cast<size_t>(n_anchor) * sizeof(int)));
    Lc.n_anchor = n_anchor;
    dim3 agrid(ceil_div(n_anchor, 128), static_cast<unsigned>(H));
    PEB_LAUNCH(ctx, icp_anchor_kernel, agrid, 128, 0, Lc, ctx->anchors.as<int>());
    Lc.anchors = ctx->anchors.as<int>();
  }
  Lw.blocks_per_hyp = blocks_for(n, H, g_warm, ctx->blocks_factor);
  Lw.warm = ctx->warm_start ? 1 : 0;
  // the search launches of split iterations (icp_search_kernel; one lane per query)
  const int fs = ctx->blocks_factor_search;
  const int search_bph_cold = blocks_for(n, H, 1, fs > 0 ? fs : cold_blocks_factor(ctx));
  const int search_bph_warm = blocks_for(n, H, 1, fs > 0 ? fs : ctx->blocks_factor);
  // the warm searches of a large enough batch run over the target's k-NN graph (built once per target)
  if (ctx->warm_graph && ctx->warm_start && g_warm == 1 && !single_mode &&
      (with_chain || (!(L.margin > 0.0f) && !ctx->warm_upfront && !ctx->warm_bin && ctx->nn_cache_from == 0)) &&
      H >= static_cast<size_t>(ctx->warm_graph_min_hyp) && launches > 1) {
    PEB_TRY(target_graph_ensure(ctx));
    Lw.knn = ctx->tgt_knn.as<KnnRow>();
    Lw.knn_stat = ctx->tgt_knn_stat.as<double>();
    Lw.knn_kappa = ctx->warm_graph_kappa;
    Lw.knn_peek_until = ctx->warm_graph_peek;
    Lw.knn_aux = ctx->warm_graph_flat ? ctx->tgt_knn_aux.as<float4>() : nullptr;
    if (ctx->cold_graph && Lc.anchors) {
      Lc.knn = Lw.knn;
      Lc.cold_graph = 1;
    }
  }
  // the candidate cache of the warm launches from launch nn_cache_from on (0: never)
  const int cache_from = (!with_chain && ctx->nn_cache_from > 0 && ctx->warm_start && g_warm == 1 && !(L.margin > 0.0f)) ? ctx->nn_cache_from : 0;
  NnCache* cache_buf = nullptr;
  if (cache_from > 0 && cache_from < launches) {
    PEB_CUDA(ctx, ctx->nn_cache.ensure(H * static_cast<size_t>(std::max(n, 1)) * sizeof(NnCache)));
    cache_buf = ctx->nn_cache.as<NnCache>();
    Lw.cache_r_cells = ctx->nn_cache_r;
  }
  // (per launch: Lw.cache is set from cache_from on; the fitness launch keeps the plain warm search)
  auto set_cache = [&](int it) {
    Lw.cache = (cache_buf && it >= cache_from && it < launches) ? cache_buf : nullptr;
    Lw.cache_init = it == cache_from ? 1 : 0;
  };
  // (per launch, after set_cache: the search blocks per hypothesis if iteration `it` runs split, else 0.  The split
  //  launches of an align stay a prefix of its launches: a moment launch waits for the count of search launches before it.)
  bool split_prefix = true;
  auto split_bph = [&](int it) {
    if (with_chain) return it == 0 ? search_bph_cold : search_bph_warm;
    split_prefix = split_prefix && split_iteration(ctx, it == 0 ? Lc : Lw, H, it == 0 ? g_cold : g_warm, it == 0);
    return split_prefix ? (it == 0 ? search_bph_cold : search_bph_warm) : 0;
  };
  ctx->prof_launches = 0;
  ctx->prof_chain_ends = 0;
  if (ctx->debug_timers) {
    PEB_CUDA(ctx, ctx->dbg.ensure(static_cast<size_t>(launches) * 8 * sizeof(unsigned long long)));
    PEB_CUDA(ctx, cudaMemsetAsync(ctx->dbg.p, 0, static_cast<size_t>(launches) * 8 * sizeof(unsigned long long), ctx->stream));
    Lc.dbg = Lw.dbg = ctx->dbg.as<unsigned long long>();
    ctx->dbg_launches = launches;
  }
  // profile 1: one event pair around the whole run of iteration launches (nothing between the
  // launches, so PDL overlap is what the bench measures); profile 2: a pair around every launch

  // Batched aligns run as S independent chains of launches on S streams, each over a contiguous
  // share of the hypotheses: while one chain drains the tail of a launch (its last blocks, the
  // per-hypothesis solves) the other chains' blocks fill the idle SMs.  Hypotheses never interact,
  // so the chains need no synchronisation between the fork and the join.
  int S = 1;
  if (!single_mode && !per_launch && !ctx->debug_timers) {
    const size_t want = ctx->batch_streams > 0 ? ctx->batch_streams : (H >= 512 ? 4 : 2);  // measured, B200 C4
    S = static_cast<int>(std::min<size_t>(want, H / 16));
    // gridDim.y carries the hypothesis index: very large batches are split into more chains
    S = std::max<int>(S, static_cast<int>((H + 32767) / 32768));
  }
  if (S <= 1 && H > 65535)
    return fail(ctx, PEB_E_UNSUPPORTED, "align_batch: %zu hypotheses in one launch (profile level 2 / debug timers "
                "allow at most 65535)", H);
  if (S > 1) {
    PEB_TRY(ensure_sub_streams(ctx, S));
    PEB_TRY(prof_mark(ctx, 0));
    PEB_CUDA(ctx, cudaEventRecord(ctx->fork_event, ctx->stream));
    const size_t per = (H + S - 1) / S;
    struct StreamSwap {  // the launch macros use ctx->stream
      peb_ctx* c;
      cudaStream_t keep;
      StreamSwap(peb_ctx* c_, cudaStream_t s) : c(c_), keep(c_->stream) { c->stream = s; }
      ~StreamSwap() { c->stream = keep; }
    };
    auto chunk_of = [&](const IcpLaunch& base, size_t h0) {
      IcpLaunch C = base;
      C.states += h0;
      C.work += h0 * static_cast<size_t>(n);
      C.slack += h0 * static_cast<size_t>(n);
      C.partials += h0 * static_cast<size_t>(base.part_stride) * kAccMax;
      C.results += h0;
      if (C.anchors) C.anchors += h0 * static_cast<size_t>(C.n_anchor);
      if (C.epochs) C.epochs += h0;
      if (C.cache) C.cache += h0 * static_cast<size_t>(n);
      return C;
    };
    auto rchunk_of = [&](size_t h0) {
      RejChain C = R;
      C.kept += h0 * static_cast<size_t>(n);
      if (C.o2o) C.o2o += h0 * static_cast<size_t>(L.grid.n);
      return C;
    };
    // the anchor launch above ran on the main stream for all hypotheses: the fork event orders it
    for (int c = 0; c < S; ++c) PEB_CUDA(ctx, cudaStreamWaitEvent(ctx->sub_streams[c], ctx->fork_event, 0));
    for (int it = 0; it <= launches; ++it) {
      Lc.launch_idx = Lw.launch_idx = it;
      set_cache(it);
      const int sb = it < launches ? split_bph(it) : 0;
      for (int c = 0; c < S; ++c) {
        const size_t h0 = c * per, h1 = std::min(H, h0 + per);
        if (h0 >= h1) continue;
        StreamSwap swap(ctx, ctx->sub_streams[c]);
        const RejChain Rc = rchunk_of(h0);
        const RejChain* rc = with_chain ? &Rc : nullptr;
        if (it == 0) {
          PEB_TRY(launch_one_iteration_g(ctx, g_cold, true, chunk_of(Lc, h0), h1 - h0, prm->estimator, sb, rc));
        } else if (it < launches) {
          PEB_TRY(launch_one_iteration_g(ctx, g_warm, false, chunk_of(Lw, h0), h1 - h0, prm->estimator, sb, rc));
        } else {
          // profile 1: the span ends with the last ITERATION launch of the slowest chain, as in the single-chain path
          // (peb_profile_read takes the maximum over the chains)
          PEB_TRY(prof_mark(ctx, 2 + c));
          PEB_TRY(launch_fitness_g(ctx, g_warm, chunk_of(Lw, h0), h1 - h0));
          PEB_CUDA(ctx, cudaEventRecord(ctx->join_events[c], ctx->stream));
        }
      }
    }
    for (int c = 0; c < S; ++c) PEB_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->join_events[c], 0));
    if (R.o2o) ctx->rej_o2o_clean = true;
    if (ctx->profile) {
      ctx->prof_launches = 1;  // one record: from the fork to the end of the last iteration launch of the slowest chain
      ctx->prof_span_launches = launches;
      ctx->prof_chain_ends = static_cast<int>(std::min<size_t>(S, (H + per - 1) / per));  // chains that hold hypotheses
    }
    return PEB_OK;
  }

  if (!per_launch) PEB_TRY(prof_mark(ctx, 0));
  for (int it = 0; it < launches; ++it) {
    if (per_launch) PEB_TRY(prof_mark(ctx, 2 * it));  // (a split iteration: both of its launches between the marks)
    Lc.launch_idx = Lw.launch_idx = it;
    set_cache(it);
    const int sb = split_bph(it);
    const RejChain* rc = with_chain ? &R : nullptr;
    if (it == 0)
      PEB_TRY(launch_one_iteration_g(ctx, g_cold, true, Lc, H, prm->estimator, sb, rc));
    else
      PEB_TRY(launch_one_iteration_g(ctx, g_warm, false, Lw, H, prm->estimator, sb, rc));
    if (per_launch) PEB_TRY(prof_mark(ctx, 2 * it + 1));
  }
  Lw.launch_idx = launches;  // the fitness launch needs all iteration launches of its hypothesis
  set_cache(launches);
  if (R.o2o) ctx->rej_o2o_clean = true;
  if (per_launch) {
    PEB_TRY(prof_mark(ctx, 2 * launches));
    PEB_TRY(launch_fitness_g(ctx, g_warm, Lw, H));
    PEB_TRY(prof_mark(ctx, 2 * launches + 1));
    if (ctx->profile) ctx->prof_launches = launches + 1;
  } else {
    PEB_TRY(prof_mark(ctx, 1));
    PEB_TRY(launch_fitness_g(ctx, g_warm, Lw, H));
    if (ctx->profile) {
      ctx->prof_launches = 1;        // one record: the span of all iteration launches
      ctx->prof_span_launches = launches;
    }
  }
  return PEB_OK;
}

#ifdef PEB_COOP_STATS
extern "C" __attribute__((visibility("default"))) int peb_debug_coop_stats(unsigned long long* out8, int reset) {
  if (cudaMemcpyFromSymbol(out8, g_coop_stats, 8 * sizeof(unsigned long long)) != cudaSuccess) return -1;
  if (reset) {
    unsigned long long z[8] = {};
    cudaMemcpyToSymbol(g_coop_stats, z, sizeof(z));
  }
  return 0;
}
#endif

int fitness_device(peb_ctx* ctx, const float* d_T, double max_range, peb_icp_result* d_result) {
  if (!ctx->tgt_grid.valid) return fail(ctx, PEB_E_NO_TARGET, "fitness_score: no target set (peb_target_set)");
  if (!ctx->src_set) return fail(ctx, PEB_E_NO_SOURCE, "fitness_score: no source set (peb_source_set)");
  peb_icp_params prm;
  peb_icp_params_default(&prm);
  prm.fitness_max_range = max_range;
  IcpLaunch L{};
  PEB_TRY(prepare_launch(ctx, 1, &prm, L));
  L.results = d_result;
  L.fitness_only = 1;
  L.warm = 0;  // an arbitrary transform: nothing to seed the search with
  L.blocks_per_hyp = blocks_for(ctx->n_src_sorted, 1, ctx->nn_group, ctx->blocks_factor);
  PEB_LAUNCH(ctx, icp_init_kernel, 1, 128, 0, L.states, d_T, 1, static_cast<int*>(nullptr));
  return launch_fitness_g(ctx, ctx->nn_group, L, 1);
}

int icp_output_device(peb_ctx* ctx, float4* d_out) {
  const int n = static_cast<int>(ctx->n_src);
  if (n == 0) return PEB_OK;
  PEB_LAUNCH(ctx, icp_output_kernel, ceil_div(n, 256), 256, 0, ctx->src.as<float4>(), n, ctx->state.as<IcpState>(),
             d_out);
  return PEB_OK;
}

int nn_search_device(peb_ctx* ctx, const float4* d_q, int nq, int32_t* d_idx, float* d_d2) {
  if (!ctx->tgt_grid.valid) return fail(ctx, PEB_E_NO_TARGET, "nn_search: no target set");
  if (nq == 0) return PEB_OK;
  const GridView& g = ctx->tgt_grid.view;
  switch (ctx->nn_group) {
    case 1: PEB_LAUNCH(ctx, nn_search_kernel<1>, ceil_div(nq, 256), 256, 0, g, d_q, nq, d_idx, d_d2); break;
    case 2: PEB_LAUNCH(ctx, nn_search_kernel<2>, ceil_div(2ll * nq, 256), 256, 0, g, d_q, nq, d_idx, d_d2); break;
    case 4: PEB_LAUNCH(ctx, nn_search_kernel<4>, ceil_div(4ll * nq, 256), 256, 0, g, d_q, nq, d_idx, d_d2); break;
    case 8: PEB_LAUNCH(ctx, nn_search_kernel<8>, ceil_div(8ll * nq, 256), 256, 0, g, d_q, nq, d_idx, d_d2); break;
    default: PEB_LAUNCH(ctx, nn_search_kernel<16>, ceil_div(16ll * nq, 256), 256, 0, g, d_q, nq, d_idx, d_d2); break;
  }
  return PEB_OK;
}

}  // namespace peb
