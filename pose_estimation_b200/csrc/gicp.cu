// gicp.cu — pcl::GeneralizedIterativeClosestPoint<PointXYZ, PointXYZ>::align on the device (DESIGN.md §15;
// [PCL] registration/impl/gicp.hpp, bfgs.h; the scalar arithmetic is gicp_math.cuh).
//
//   gicp_cov_*_kernel     computeCovariances: the k nearest neighbours of every point of a cloud in its own grid
//                         (knn_list.cuh, the searches of NormalEstimation), their moments, svd3, the reconstitution.
//                         Once per cloud and k, by sorted grid position.  The source is walked as its FINITE points in
//                         the order of its own grid, so non-finite rows change no sum.
//   gicp_search_kernel    one per outer iteration: the query transformation_ * output[i], its exact nearest target point
//                         (nn_search.cuh: the ring search in the first iteration, then the ball search seeded by the
//                         previous match), the pair test d2 < max_corr_dist^2 and M_i = (R C1 R^T + C2)^-1 (9 doubles).
//   gicp_bfgs_kernel      one per outer iteration: one thread-block cluster per hypothesis runs the whole inner BFGS.
//                         Every f / g evaluation sums the pairs of each block in a fixed order, then the blocks' sums in
//                         rank order through distributed shared memory.  Every thread runs the same scalar state machine
//                         on the same sums, so no decision has to be broadcast.  The cluster size depends on n_src only:
//                         a hypothesis gets the same bytes alone or inside any batch.
// The host polls a per-iteration "hypotheses still iterating" counter every kGicpPollEvery iterations.
#include <cooperative_groups.h>

#include <algorithm>
#include <cfloat>

#include "gicp_math.cuh"
#include "knn_list.cuh"

namespace cg = cooperative_groups;

namespace peb {

namespace {

constexpr int kGicpThreads = 256;
constexpr int kGicpWarps = kGicpThreads / 32;
constexpr int kGicpMaxCluster = 8;         // the portable cluster size
constexpr int kGicpPointsPerBlock = 8192;  // points per block of a cluster before the cluster grows
constexpr int kGicpPollEvery = 4;          // outer iterations between two reads of the "still iterating" counter

struct GicpState {
  float T[16];        // transformation_
  float guess[16];
  float final_t[16];  // final_transformation_ once the hypothesis has stopped
  double last_mse;
  int iterations;
  int active;
  int state;
  int converged;
  int ncorr;
  int pad;
};

struct GicpLaunch {
  GridView tgt;
  const float4* src;      // n_src FINITE source points in the order of the source's grid, .w = original index
  int n_src;
  const double* src_cov;  // n_src x 9, same order
  const double* tgt_cov;  // tgt.n x 9, sorted grid position
  GicpState* st;          // H
  int* prev;              // H x n_src: sorted position of the last match (-1: none)
  float4* tq;             // H x n_src: the pair's target point; .w = original target index, -1 = no pair
  float* d2;              // H x n_src: squared distance of the match
  double* M;              // H x n_src x 9
  int* alive;             // per outer iteration: hypotheses that go on after it
  double dist_thr;        // max_corr_dist^2 (pair iff d2 < it)
  float stop_d2;          // searches may stop once every unexamined point is farther than this
  int iter;
  int max_iterations;
  int max_inner;
  int cluster;
  double inv_rot_eps, inv_trans_eps;
};

__global__ void __launch_bounds__(256) gicp_nan_rows_kernel(double* __restrict__ out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 9 * n) out[i] = __longlong_as_double(0x7ff8000000000000ll);
}

__device__ __forceinline__ void gicp_cov_store(double* __restrict__ out, int row, const double (&acc)[9], int k) {
  double c[9];
  gicp_cov_finish(acc, k, c);
#pragma unroll
  for (int i = 0; i < 9; ++i) out[static_cast<size_t>(row) * 9 + i] = c[i];
}

// k <= K <= 32: the register list; row = sorted grid position
template <int K>
__global__ void __launch_bounds__(128, 4) gicp_cov_reglist_kernel(const GridView g, int k, double* __restrict__ out) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= g.n) return;
  const float4 p = g.pts[q];
  RegList<K> l;
  reglist_knn<K>(g, p, k, l);
  double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
  for (int s = 0; s < K; ++s) {
    if (l.j[s] >= 0) {
      const float4 c = g.pts[l.j[s]];
      gicp_cov_add(acc, c.x, c.y, c.z);
    }
  }
  gicp_cov_store(out, q, acc, k);
}

// k > 32: the shared-memory list
__global__ void gicp_cov_knn_kernel(const GridView g, int k, double* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int T = blockDim.x;
  const int q = blockIdx.x * T + threadIdx.x;
  if (q >= g.n) return;
  const float4 p = g.pts[q];
  KnnList l;
  knn_list_search(g, p, k, reinterpret_cast<unsigned long long*>(smem_raw), l);
  double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int i = 0; i < l.count; ++i) {
    const float4 c = g.pts[knn_key_pos(l.e[i * T])];
    gicp_cov_add(acc, c.x, c.y, c.z);
  }
  gicp_cov_store(out, q, acc, k);
}

// a cloud's covariances (by sorted position) in original order
__global__ void __launch_bounds__(256) gicp_cov_unsort_kernel(const GridView g, const double* __restrict__ cov,
                                                             double* __restrict__ out) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= g.n) return;
  const int orig = __float_as_int(g.pts[j].w);
#pragma unroll
  for (int i = 0; i < 9; ++i) out[static_cast<size_t>(orig) * 9 + i] = cov[static_cast<size_t>(j) * 9 + i];
}

__global__ void gicp_init_kernel(GicpState* __restrict__ st, const float* __restrict__ guesses, int H) {
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= H) return;
  GicpState s;
  const Mat4 I = mat4_identity();
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    s.T[i] = I.m[i];
    s.guess[i] = guesses ? guesses[16 * h + i] : I.m[i];
    s.final_t[i] = s.guess[i];
  }
  s.last_mse = DBL_MAX;
  s.iterations = 0;
  s.active = 1;
  s.state = PEB_NOT_CONVERGED;
  s.converged = 0;
  s.ncorr = 0;
  s.pad = 0;
  st[h] = s;
}

// grid (ceil(n_src / kGicpThreads), H)
__global__ void __launch_bounds__(kGicpThreads) gicp_search_kernel(const GicpLaunch L) {
  const int h = blockIdx.y;
  const GicpState* st = L.st + h;
  if (!st->active) return;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= L.n_src) return;
  float T[16], G[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    T[k] = st->T[k];
    G[k] = st->guess[k];
  }
  const size_t o = static_cast<size_t>(h) * L.n_src + i;
  const float4 p = L.src[i];
  float4 tq = make_float4(0.f, 0.f, 0.f, __int_as_float(-1));
  float d2 = pos_inf();
  {
    float ox, oy, oz, qx, qy, qz;
    transform_tpc(G, p.x, p.y, p.z, ox, oy, oz);  // output = transformPointCloud(input, guess)
    transform_icp(T, ox, oy, oz, qx, qy, qz);     // transformation_ * output[i]
    const int jp = L.iter > 0 ? L.prev[o] : -1;
    const NnBest best = jp >= 0 ? grid_nn_warm(L.tgt, qx, qy, qz, jp, L.stop_d2) : grid_nn<1>(L.tgt, qx, qy, qz, L.stop_d2);
    L.prev[o] = best.j;
    if (best.idx >= 0 && static_cast<double>(best.d2) < L.dist_thr) {
      const float4 t = L.tgt.pts[best.j];
      tq = make_float4(t.x, t.y, t.z, __int_as_float(best.idx));
      d2 = best.d2;
      double R[9];
      gicp_rotation_d(T, G, R);
      gicp_mahalanobis(R, L.src_cov + static_cast<size_t>(i) * 9, L.tgt_cov + static_cast<size_t>(best.j) * 9, L.M + o * 9);
    }
  }
  L.tq[o] = tq;
  L.d2[o] = d2;
}

// Sums N doubles over the cluster: every thread's values in a fixed order (xor tree in the warp, warps in order, the
// blocks' sums in rank order).  The result is in tot[0 .. N) of every block; part is double-buffered by the caller's
// parity, so one cluster barrier per reduction suffices.
template <int N>
__device__ __forceinline__ void gicp_cluster_sum(cg::cluster_group& cl, int C, double (&acc)[N], double* wsum, double* part,
                                                 double* tot, int& parity) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int v = 0; v < N; ++v) {
    double s = acc[v];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
    if (lane == 0) wsum[warp * N + v] = s;
  }
  __syncthreads();
  if (threadIdx.x < N) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kGicpWarps; ++w) s += wsum[w * N + threadIdx.x];
    part[parity * N + threadIdx.x] = s;
  }
  cl.sync();
  if (threadIdx.x < N) {
    double s = 0.0;
    for (int r = 0; r < C; ++r) s += cl.map_shared_rank(part, r)[parity * N + threadIdx.x];
    tot[threadIdx.x] = s;
  }
  parity ^= 1;
  __syncthreads();
}

// the evaluator of gicp_bfgs_minimize: f and g at x over the hypothesis' pairs (a collective of the cluster)
struct GicpClusterEval {
  const GicpLaunch* L;
  cg::cluster_group* cl;
  int h, rank, m;
  const float* G;
  double *wsum, *part, *tot;
  int parity;
  __device__ void fdf(const double* x, double& f, double* g) {
    const Mat4 Tx = gicp_apply_state(x);
    double acc[kGicpAcc];
#pragma unroll
    for (int v = 0; v < kGicpAcc; ++v) acc[v] = 0.0;
    const int C = L->cluster, n = L->n_src;
    const size_t base = static_cast<size_t>(h) * n;
    for (int i = rank * kGicpThreads + threadIdx.x; i < n; i += C * kGicpThreads) {
      const float4 t = L->tq[base + i];
      if (__float_as_int(t.w) < 0) continue;
      const float4 p = L->src[i];
      float ox, oy, oz;
      transform_tpc(G, p.x, p.y, p.z, ox, oy, oz);
      gicp_pair_add(acc, Tx.m, ox, oy, oz, t.x, t.y, t.z, L->M + (base + i) * 9);
    }
    gicp_cluster_sum<kGicpAcc>(*cl, C, acc, wsum, part, tot, parity);
    double s[kGicpAcc];
#pragma unroll
    for (int v = 0; v < kGicpAcc; ++v) s[v] = tot[v];
    gicp_fg_finish(s, m, x, f, g);
  }
};

// grid (cluster x H), cluster (cluster, 1, 1)
__global__ void __launch_bounds__(kGicpThreads, 1) gicp_bfgs_kernel(const GicpLaunch L) {
  cg::cluster_group cl = cg::this_cluster();
  __shared__ double wsum[kGicpWarps * kGicpAcc];
  __shared__ double part[2 * kGicpAcc];
  __shared__ double tot[kGicpAcc];
  const int C = L.cluster;
  const int rank = static_cast<int>(cl.block_rank());
  const int h = blockIdx.x / C;
  GicpState* st = L.st + h;
  if (!st->active) return;  // (the whole cluster: nobody touches another block's shared memory)
  float T[16], G[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    T[k] = st->T[k];
    G[k] = st->guess[k];
  }
  const int iterations0 = st->iterations;
  int parity = 0;
  // the pairs of this iteration: count and sum of d2
  double a2[2] = {0.0, 0.0};
  {
    const size_t base = static_cast<size_t>(h) * L.n_src;
    for (int i = rank * kGicpThreads + threadIdx.x; i < L.n_src; i += C * kGicpThreads) {
      if (__float_as_int(L.tq[base + i].w) >= 0) {
        a2[0] += 1.0;
        a2[1] += static_cast<double>(L.d2[base + i]);
      }
    }
  }
  gicp_cluster_sum<2>(cl, C, a2, wsum, part, tot, parity);
  const int m = static_cast<int>(tot[0]);
  const double sum_d2 = tot[1];
  GicpState s;
  s.last_mse = m > 0 ? sum_d2 / static_cast<double>(m) : DBL_MAX;
  s.ncorr = m;
  s.pad = 0;
  s.iterations = iterations0;
#pragma unroll
  for (int k = 0; k < 16; ++k) s.guess[k] = G[k];
  if (m < 4) {
    // estimateRigidTransformationBFGS throws NotEnoughPointsException below 4 pairs and the loop ends there
    // (m == 0: PCL would divide by zero); the record keeps final = previous * guess, previous = transformation_
    Mat4 Tm, Gm;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      Tm.m[k] = T[k];
      Gm.m[k] = G[k];
    }
    const Mat4 F = mat4_mul(Tm, Gm);
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      s.T[k] = T[k];
      s.final_t[k] = F.m[k];
    }
    s.active = 0;
    s.converged = 0;
    s.state = PEB_NO_CORRESPONDENCES;
  } else {
    double x[6];
    gicp_state_of(T, x);
    GicpClusterEval ev{&L, &cl, h, rank, m, G, wsum, part, tot, parity};
    gicp_bfgs_minimize(ev, x, L.max_inner);
    const Mat4 Tn = gicp_apply_state(x);
    double delta = 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
      for (int l = 0; l < 4; ++l) {
        const double ratio = (k < 3 && l < 3) ? L.inv_rot_eps : L.inv_trans_eps;
        const double c = ratio * static_cast<double>(fabsf(T[l * 4 + k] - Tn.m[l * 4 + k]));
        if (c > delta) delta = c;
      }
    s.iterations = iterations0 + 1;
    const bool stop = s.iterations >= L.max_iterations || delta < 1.0;
    Mat4 Gm;
#pragma unroll
    for (int k = 0; k < 16; ++k) Gm.m[k] = G[k];
    const Mat4 F = mat4_mul(Tn, Gm);
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      s.T[k] = Tn.m[k];
      s.final_t[k] = stop ? F.m[k] : 0.0f;
    }
    s.active = stop ? 0 : 1;
    s.converged = stop ? 1 : 0;
    s.state = stop ? (delta < 1.0 ? PEB_TRANSFORM : PEB_ITERATIONS) : PEB_NOT_CONVERGED;
  }
  if (rank == 0 && threadIdx.x == 0) {
    *st = s;
    if (s.active) atomicAdd(L.alive + L.iter, 1);
  }
  cl.sync();  // no block leaves while another may still read its shared memory
}

__global__ void gicp_final_kernel(const GicpState* __restrict__ st, int H, float* __restrict__ final16) {
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= H) return;
#pragma unroll
  for (int k = 0; k < 16; ++k) final16[16 * h + k] = st[h].final_t[k];
}

// the records: the GICP state with the fitness of getFitnessScore (icp.cu's fitness launch, written to fit)
__global__ void gicp_pack_kernel(const GicpState* __restrict__ st, const peb_icp_result* __restrict__ fit, int H,
                                 peb_icp_result* __restrict__ out) {
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= H) return;
  const GicpState s = st[h];
  peb_icp_result r;
#pragma unroll
  for (int k = 0; k < 16; ++k) r.T[k] = s.final_t[k];
  r.fitness = fit[h].fitness;
  r.last_mse = s.last_mse;
  r.iterations = s.iterations;
  r.converged = s.converged;
  r.state = s.state;
  r.n_correspondences = s.ncorr;
  out[h] = r;
}

// single align outputs: the aligned cloud (transformPointCloud(input, final)) over the original records, no pair yet
__global__ void __launch_bounds__(256) gicp_output_kernel(const float4* __restrict__ src, int n, const GicpState* __restrict__ st,
                                                          float4* __restrict__ aligned, int32_t* __restrict__ corr_idx,
                                                          float* __restrict__ corr_d2) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (aligned) {
    const float4 p = src[i];
    float x, y, z;
    transform_tpc(st->final_t, p.x, p.y, p.z, x, y, z);
    aligned[i] = make_float4(x, y, z, 1.0f);
  }
  if (corr_idx) corr_idx[i] = -1;
  if (corr_d2) corr_d2[i] = pos_inf();
}

// ... then the last iteration's pairs of the finite points, scattered to their original index
__global__ void __launch_bounds__(256) gicp_corr_kernel(const float4* __restrict__ srt, int n, const float4* __restrict__ tq,
                                                        const float* __restrict__ d2, int32_t* __restrict__ corr_idx,
                                                        float* __restrict__ corr_d2) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= n) return;
  const int orig = __float_as_int(srt[q].w);
  const int idx = __float_as_int(tq[q].w);
  if (corr_idx) corr_idx[orig] = idx;
  if (corr_d2 && idx >= 0) corr_d2[orig] = d2[q];
}

// smallest float >= d (inf if none): nothing acceptable is cut off by the search bound
float gicp_stop_bound(double d) {
  if (!(d < static_cast<double>(FLT_MAX))) return INFINITY;
  if (d < 0.0) return 0.0f;
  float f = static_cast<float>(d);
  if (static_cast<double>(f) < d) f = nextafterf(f, INFINITY);
  return f;
}

int cov_launch(peb_ctx* ctx, const GridView& g, int k, double* out) {
  if (g.n == 0) return PEB_OK;
  if (k <= 8) PEB_LAUNCH(ctx, gicp_cov_reglist_kernel<8>, ceil_div(g.n, 128), 128, 0, g, k, out);
  else if (k <= 16) PEB_LAUNCH(ctx, gicp_cov_reglist_kernel<16>, ceil_div(g.n, 128), 128, 0, g, k, out);
  else if (k <= 24) PEB_LAUNCH(ctx, gicp_cov_reglist_kernel<24>, ceil_div(g.n, 128), 128, 0, g, k, out);
  else if (k <= 32) PEB_LAUNCH(ctx, gicp_cov_reglist_kernel<32>, ceil_div(g.n, 128), 128, 0, g, k, out);
  else {
    const int T = k <= 48 ? 128 : (k <= 96 ? 64 : 32);
    PEB_LAUNCH(ctx, gicp_cov_knn_kernel, ceil_div(g.n, T), T, static_cast<size_t>(k) * T * 8, g, k, out);
  }
  return PEB_OK;
}

}  // namespace

int gicp_check_k(peb_ctx* ctx, int k) {
  if (!ctx->tgt_grid.valid) return fail(ctx, PEB_E_NO_TARGET, "gicp: no target set (peb_target_set)");
  if (!ctx->src_set) return fail(ctx, PEB_E_NO_SOURCE, "gicp: no source set (peb_source_set)");
  if (k < 1) return fail(ctx, PEB_E_INVALID_ARG, "gicp: k_correspondences must be >= 1 (got %d)", k);
  if (k > 192) return fail(ctx, PEB_E_UNSUPPORTED, "gicp: k_correspondences = %d > 192 has no CUDA path (no CPU fallback)", k);
  if (k > ctx->tgt_grid.view.n || k > ctx->src_grid.view.n)
    return fail(ctx, PEB_E_INVALID_ARG, "gicp: k_correspondences = %d exceeds the finite points of the source (%d) or target (%d)", k,
                ctx->src_grid.view.n, ctx->tgt_grid.view.n);
  return PEB_OK;
}

// computeCovariances of both clouds for k, unless the context still holds them
int gicp_covariances_ensure(peb_ctx* ctx, int k) {
  PEB_TRY(gicp_check_k(ctx, k));
  if (ctx->gicp_src_k != k) {
    const GridView& g = ctx->src_grid.view;
    PEB_CUDA(ctx, ctx->gicp_src_cov.ensure(std::max<size_t>(g.n, 1) * 9 * sizeof(double)));
    PEB_TRY(cov_launch(ctx, g, k, ctx->gicp_src_cov.as<double>()));
    ctx->gicp_src_k = k;
  }
  if (ctx->gicp_tgt_k != k) {
    const GridView& g = ctx->tgt_grid.view;
    PEB_CUDA(ctx, ctx->gicp_tgt_cov.ensure(std::max<size_t>(g.n, 1) * 9 * sizeof(double)));
    PEB_TRY(cov_launch(ctx, g, k, ctx->gicp_tgt_cov.as<double>()));
    ctx->gicp_tgt_k = k;
  }
  return PEB_OK;
}

int gicp_covariances_device(peb_ctx* ctx, int which, int k, double* d_out9) {
  PEB_TRY(gicp_covariances_ensure(ctx, k));
  const int n = static_cast<int>(which == 0 ? ctx->n_src : ctx->n_tgt);
  if (n == 0) return PEB_OK;
  const GridView& g = which == 0 ? ctx->src_grid.view : ctx->tgt_grid.view;
  const double* cov = which == 0 ? ctx->gicp_src_cov.as<double>() : ctx->gicp_tgt_cov.as<double>();
  PEB_LAUNCH(ctx, gicp_nan_rows_kernel, ceil_div(9ll * n, 256), 256, 0, d_out9, n);
  if (g.n > 0) PEB_LAUNCH(ctx, gicp_cov_unsort_kernel, ceil_div(g.n, 256), 256, 0, g, cov, d_out9);
  return PEB_OK;
}

int gicp_align_device(peb_ctx* ctx, const float* d_guesses, size_t H, const peb_gicp_params* prm, peb_icp_result* d_results,
                      float4* d_aligned, int32_t* d_corr_idx, float* d_corr_d2) {
  if (H == 0) return PEB_OK;
  PEB_TRY(gicp_covariances_ensure(ctx, prm->k_correspondences));
  const int n = ctx->src_grid.view.n;  // the finite source points, in the order of the source's grid
  const size_t hn = H * static_cast<size_t>(std::max(n, 1));
  PEB_CUDA(ctx, ctx->gicp_state.ensure(H * sizeof(GicpState)));
  PEB_CUDA(ctx, ctx->gicp_prev.ensure(hn * sizeof(int)));
  PEB_CUDA(ctx, ctx->gicp_tq.ensure(hn * sizeof(float4)));
  PEB_CUDA(ctx, ctx->gicp_d2.ensure(hn * sizeof(float)));
  {
    const cudaError_t e = ctx->gicp_M.ensure(hn * 9 * sizeof(double));
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(ctx, e == cudaErrorMemoryAllocation ? PEB_E_OOM : PEB_E_CUDA,
                  "gicp: the Mahalanobis matrices of %zu hypotheses x %d points (%.2f GB) cannot be allocated: %s", H, n,
                  static_cast<double>(hn) * 72.0 / 1e9, cudaGetErrorString(e));
    }
  }
  const int max_it = std::max(prm->max_iterations, 1);
  PEB_CUDA(ctx, ctx->gicp_alive.ensure(static_cast<size_t>(max_it) * sizeof(int)));
  PEB_CUDA(ctx, ctx->gicp_final.ensure(H * 16 * sizeof(float)));
  PEB_CUDA(ctx, ctx->gicp_fit.ensure(H * sizeof(peb_icp_result)));
  PEB_CUDA(ctx, ctx->h_small.ensure(4096));
  PEB_CUDA(ctx, cudaMemsetAsync(ctx->gicp_alive.p, 0, static_cast<size_t>(max_it) * sizeof(int), ctx->stream));
  GicpState* st = ctx->gicp_state.as<GicpState>();
  PEB_LAUNCH(ctx, gicp_init_kernel, ceil_div(static_cast<long long>(H), 128), 128, 0, st, d_guesses, static_cast<int>(H));

  GicpLaunch L{};
  L.tgt = ctx->tgt_grid.view;
  L.src = ctx->src_grid.view.pts;
  L.n_src = n;
  L.src_cov = ctx->gicp_src_cov.as<double>();
  L.tgt_cov = ctx->gicp_tgt_cov.as<double>();
  L.st = st;
  L.prev = ctx->gicp_prev.as<int>();
  L.tq = ctx->gicp_tq.as<float4>();
  L.d2 = ctx->gicp_d2.as<float>();
  L.M = ctx->gicp_M.as<double>();
  L.alive = ctx->gicp_alive.as<int>();
  L.dist_thr = prm->max_corr_dist * prm->max_corr_dist;
  L.stop_d2 = gicp_stop_bound(L.dist_thr);
  L.max_iterations = max_it;
  L.max_inner = prm->max_inner_iterations;
  L.cluster = std::min(kGicpMaxCluster, std::max(1, ceil_div(n, kGicpPointsPerBlock)));
  L.inv_rot_eps = 1.0 / prm->rotation_epsilon;
  L.inv_trans_eps = 1.0 / prm->transformation_epsilon;

  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(L.cluster * H));
  cfg.blockDim = dim3(kGicpThreads);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = ctx->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = static_cast<unsigned>(L.cluster);
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  int* h_alive = ctx->h_small.as<int>() + 96;
  const dim3 sgrid(static_cast<unsigned>(ceil_div(std::max(n, 1), kGicpThreads)), static_cast<unsigned>(H));
  for (int it = 0; it < max_it; ++it) {
    L.iter = it;
    PEB_LAUNCH(ctx, gicp_search_kernel, sgrid, kGicpThreads, 0, L);
    ctx->launches++;
    PEB_CUDA(ctx, cudaLaunchKernelEx(&cfg, gicp_bfgs_kernel, L));
    if ((it + 1) % kGicpPollEvery == 0 && it + 1 < max_it) {
      PEB_CUDA(ctx, cudaMemcpyAsync(h_alive, ctx->gicp_alive.as<int>() + it, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
      PEB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
      if (*h_alive == 0) break;
    }
  }
  float* d_final = ctx->gicp_final.as<float>();
  PEB_LAUNCH(ctx, gicp_final_kernel, ceil_div(static_cast<long long>(H), 128), 128, 0, st, static_cast<int>(H), d_final);
  PEB_TRY(fitness_batch_device(ctx, d_final, H, prm->fitness_max_range, ctx->gicp_fit.as<peb_icp_result>()));
  PEB_LAUNCH(ctx, gicp_pack_kernel, ceil_div(static_cast<long long>(H), 128), 128, 0, st, ctx->gicp_fit.as<peb_icp_result>(),
             static_cast<int>(H), d_results);
  const int n_all = static_cast<int>(ctx->n_src);
  if (n_all > 0 && (d_aligned || d_corr_idx || d_corr_d2)) {
    PEB_LAUNCH(ctx, gicp_output_kernel, ceil_div(n_all, 256), 256, 0, ctx->src.as<float4>(), n_all, st, d_aligned, d_corr_idx, d_corr_d2);
    if (n > 0 && (d_corr_idx || d_corr_d2))
      PEB_LAUNCH(ctx, gicp_corr_kernel, ceil_div(n, 256), 256, 0, L.src, n, L.tq, L.d2, d_corr_idx, d_corr_d2);
  }
  return PEB_OK;
}

}  // namespace peb
