// common.cuh — context, buffers and launch helpers shared by every translation unit of
// libpe_b200.so.  sm_100a only; the whole library is compiled with -fmad=false so that float
// expressions keep PCL's source-level rounding (SURVEY.md H1); fused operations are written
// explicitly (fma()) where they are wanted.
#pragma once

#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/pe_b200.h"

#define PEB_HD __host__ __device__ __forceinline__

namespace peb {

constexpr int kSmCount = 148;  // B200: 2 dies x 74 SMs; grids are sized in multiples of this

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T>
  T* as() const {
    return static_cast<T*>(p);
  }
};

struct PinnedBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMallocHost(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T>
  T* as() const {
    return static_cast<T*>(p);
  }
};

// The uniform grid over a cloud (the kd-tree replacement, SURVEY.md 8a-2').  Points are sorted
// by cell id (x fastest), cell_start has n_cells + 1 entries, so the points of the x-run of
// cells [c0, c1] of one (y, z) row are the contiguous range [cell_start[c0], cell_start[c1 + 1]).
struct GridView {
  const float4* pts;            // sorted; .w carries the ORIGINAL index (int bits)
  const float4* normals;        // sorted like pts (nullable)
  const uint32_t* cell_start;   // n_cells + 1
  float ox, oy, oz;             // origin = min corner of the finite bounding box
  float h, inv_h;               // cell edge and its reciprocal
  int dx, dy, dz;               // cells per axis
  int n;                        // finite points
};

struct Grid {
  DevBuf pts, normals, cell_start, keys, vals, keys_tmp, vals_tmp;
  GridView view{};
  long long n_cells = 0;
  int n_input = 0;    // records handed in (including non-finite)
  bool valid = false;
};

}  // namespace peb

// ---- the context ---------------------------------------------------------------------------
struct peb_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  uint64_t launches = 0;
  int nn_group = 1;             // lanes that share one COLD nearest-neighbour query (1, 2, 4, 8, 16)
  float grid_occupancy = 5.0f;  // wanted mean points per occupied cell of the target grid.  Round 1 (every warm query walks the grid), C4 / C2:
                                // 1.0 93.3 ms, 1.5 94.1, 2.0 97.1, 2.5 93.4, 3.0 91.8, 3.5 91.5, 4.0 91.2, 5.0 92.7, 6.0 95.4, 8.0 101.0 per
                                // 1024-hypothesis batch; single align 0.736 ms at 2.0, 0.721 at 3.0, 0.729 at 4.0.  Round 2 (near queries are
                                // settled by the k-NN graph, only the larger balls still walk): 2.0 70.1 ms, 2.75 67.1, 3.5 64.5, 4.5 63.1,
                                // 5.0 62.8, 6.0 62.5, 7.0 62.6, 8.0 62.9; single align 0.722 ms at 3.5, 0.733 at 5.0, 0.741 at 6.0, 0.751 at 7.0;
                                // a 128-hypothesis shard 8.83 ms at 3.5, 8.49 at 5.0
  bool warm_start = true;       // iterations >= 1 seed the search with the previous match
  int warm_upfront = 0;         // experimental: warm searches fetch the row bounds of their ball up front (nn_upfront.cuh):
                                // 0 = off, 1 or 2 = boxes up to 2 x 2 rows, 3 = up to 3 x 3; unmeasured
  int warm_upfront_from = 2;    // ... from this iteration launch on (launch 1 searches balls of 1.3 cells: 61 % of its warps hold a lane beyond 3 x 3 rows)
  int warm_graph = 1;           // batched warm launches search over the target's k-NN graph (nn_graph.cuh) instead of walking the grid
  float warm_graph_kappa = 0.0f; // > 0: a hypothesis takes the graph once 4 * MSE * kappa < mean outer bound of the rows; 0: from launch 1 on (measured flat from 0 to 0.6 once hopeless rows are skipped)
  int warm_graph_queue = 0;     // (measured: -7 %, off) graph launches: every warp queues the unproven queries of a tile of 8 / 16 passes and
                                // walks the grid for them 32 at a time (icp.cu : icp_iteration_graphq_kernel); 0 = every lane walks for itself
  int warm_graph_flat = 1;      // graph searches also try the flatness certificate (nn_graph.cuh : knn_aux_of) ...
  int warm_graph_flat_from = 2, warm_graph_flat_until = 15;  // ... in these iteration launches
  int warm_graph_peek = 1;      // (measured: launch 1 5.0 -> 4.6 ms, nothing after it) graph launches 1 .. this: a query whose row cannot certify looks at the four nearest neighbours of its previous match before it walks
  int cold_graph = 1;           // launch 0 of a batch with a graph: candidates by greedy descent from the patch's anchor match instead of the 3 x 3 x 3 probe
  int warm_graph_min_hyp = 32;  // ... for batches of at least this many hypotheses (the graph costs one k-NN pass over the target)
  int warm_bin = 0;             // (measured: -6 %, off) batched warm launches bin the queries of a block by the rows their search walks (icp.cu : icp_iteration_binned_kernel)
  bool anchor_seed = true;      // iteration 0: one cold search per 32-point patch seeds the patch
  int coop_max_rows = 1024;     // first iteration of a batch: a patch verifies its 32 candidates together (nn_search.cuh) up to this many grid rows
  float seed_guard = 10.0f;     // seeds farther than this many cells from the query are not used
  int batch_streams = 0;        // batched aligns: independent chains of launches (see icp.cu); 0 = auto
  std::vector<cudaStream_t> sub_streams;
  std::vector<cudaEvent_t> join_events;
  cudaEvent_t fork_event = nullptr;
  int blocks_factor = 0;        // batched aligns: ~this many blocks per SM and launch in total; 0 = auto
  int blocks_factor_cold = 0;   // the same for launch 0 of a batched align; 0 = like blocks_factor
  int blocks_factor_search = 0; // the same for the search launches of split iterations; 0 = like the launch's moment launch
  int split_moments = 1;        // batched iterations run as a search launch and a moment launch (icp.cu : icp_search_kernel)
  int split_min_hyp = 256;      // ... in batches of at least this many hypotheses (a 128-hypothesis shard: 8.27 / 8.58 ms fused,
                                // 8.27 / 8.66 split at PEB_HYP_OFFSET 0 / 512, B200)
  bool flag_deps = true;        // warm launches wait per hypothesis (epoch flags) instead of for the whole previous grid
  peb::DevBuf epochs;           // H solved-iteration counters + 1 error flag
  int* last_err_flag = nullptr; // device address of that flag for the last batched align (nullptr: whole-grid dependencies)
  bool use_pdl = true;          // programmatic dependent launch between the ICP launches of an align
  bool debug_timers = false;    // development: %globaltimer stamps of the phases of every iteration launch
  peb::DevBuf dbg;
  int dbg_launches = 0;
  peb::DevBuf anchors;          // H x ceil(n / 32) sorted positions
  int nn_cache_from = 0;        // warm launches from this one on answer from the candidate cache (nn_cache.cuh); 0: off
  float nn_cache_r = 0.75f;     // radius (cells) a cache entry's collecting search covers
  peb::DevBuf nn_cache;         // H x n_src entries of 32 bytes
  float cert_margin = 0.0f;     // > 0: warm searches cover this fraction of a cell beyond the match, which
                                // buys a certificate that lets later iterations skip the search while the
                                // point has moved less than half of it.  Off by default: on surface scans the
                                // runner-up is ~0.2 mm behind the winner and point-to-point ICP creeps by
                                // tens of micrometres per iteration, so certificates expire at once and the
                                // larger ball only costs time (measured: 6738 -> 5442 hyp/s at 0.25 h).

  peb::PinnedBuf h_stage;    // host repack / readback staging
  peb::PinnedBuf h_small;    // small results (bbox, counters, peb_icp_result)
  peb::DevBuf d_small;       // device side of h_small
  peb::DevBuf d_scratch;     // plane RANSAC staging
  peb::DevBuf sort_scratch;  // radix sort: digit histograms, tile tickets, look-back words (sort_scan.cuh : SortPlan)
  peb::DevBuf scan_scratch[4];  // single-pass scans: look-back words + ticket + total per slot (sort_scan.cuh : ScanState)
  peb::DevBuf d_stage;       // raw host records before the repack kernel

  // target (scene)
  peb::DevBuf tgt_raw;       // float4 xyz(w) in original order
  peb::DevBuf tgt_nrm_raw;   // float4 normals in original order (if any)
  size_t n_tgt = 0;
  bool tgt_has_normals = false;
  bool tgt_staged = false;            // tgt_raw (+ normals) holds a cloud; tgt_stage_event orders a replica's copy after it
  cudaEvent_t tgt_stage_event = nullptr;
  peb::Grid tgt_grid;
  peb::DevBuf tgt_knn;                // k-nearest-neighbour graph of the target grid's points (nn_graph.cuh), 64 bytes per point,
  peb::DevBuf tgt_knn_aux;            // ... and the flatness certificate's (direction, height bound) per point, 16 bytes
  peb::DevBuf tgt_knn_stat;           // two doubles: sum and count of the rows' finite outer bounds
  bool tgt_knn_valid = false;         // built by the first batched align on this target that uses it

  // source (model)
  peb::DevBuf src;           // float4 xyz1, original order
  size_t n_src = 0;
  bool src_set = false;
  bool src_staged = false;
  cudaEvent_t src_stage_event = nullptr;
  // the finite source points sorted by the cells of a coarse grid over the source itself
  // (~32 points per cell = one warp per compact patch): neighbouring threads get neighbouring
  // queries, i.e. the same grid rows, the same ring counts and L1 hits.  .w = original index.
  peb::Grid src_grid;
  int n_src_sorted = 0;
  float src_sort_occupancy = 32.0f;

  // ICP working set
  peb::DevBuf work;          // float4 working clouds
  peb::DevBuf slack;         // float per working point: remaining certificate of its match
  peb::DevBuf corr_idx, corr_d2;
  peb::DevBuf partials;      // per-block double partial sums
  peb::DevBuf rej_kept;      // rejector chains: one kept byte per working point (icp.cu : icp_reject_kernel)
  peb::DevBuf rej_o2o;       // ... the one-to-one rejector's H x target-point keys, all ones between aligns
  bool rej_o2o_clean = false;  // rej_o2o holds all ones (an align that stopped queueing half-way may have left keys)
  peb::DevBuf state;         // IcpState per hypothesis
  peb::DevBuf trace;         // per-iteration increments of the last single align
  peb::DevBuf d_guesses, d_results, d_aligned;
  int last_trace_cap = 0;
  int last_iterations = 0;
  // optional per-launch timing of the ICP kernels (bench.py's roofline leg): event pairs around
  // every iteration launch + the fitness launch of the last align
  bool profile = false;
  std::vector<cudaEvent_t> prof_events;
  int prof_launches = 0;
  int profile_level = 0;        // 1: one event pair around all iteration launches, 2: one per launch
  int prof_span_launches = 0;
  int prof_chain_ends = 0;      // > 0: the last align ran as this many chains; events 2 .. 2 + chains - 1 end their iteration launches
  peb::DevBuf nn_q, nn_idx, nn_d2;   // peb_nn_search staging

  // voxel grid / normals scratch
  peb::Grid aux_grid;
  peb::DevBuf vg_in, vg_out, vg_flags, vg_scan, vg_starts;
  peb::DevBuf nrm_in, nrm_out;
  peb::DevBuf brute_keys;    // brute-force validator: one 64-bit (distance, index) key per query, merged over the target segments with atomicMin
  peb::DevBuf cv_arena;      // cv::ppf_match_3d::ICP mode: all device buffers of a call
  peb::PinnedBuf h_cv;       // cv ICP mode: pose tables (two, alternating) + accumulator read-back
  peb::PinnedBuf h_sac;      // plane RANSAC: sample indices / coordinates, candidate planes, counts, moment records
};

namespace peb {

int fail(peb_ctx* ctx, int code, const char* fmt, ...);

#define PEB_CUDA(ctx, expr)                                                                   \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess) {                                                                  \
      cudaGetLastError();                                                                     \
      return peb::fail((ctx), _e == cudaErrorMemoryAllocation ? PEB_E_OOM : PEB_E_CUDA,       \
                       "%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
    }                                                                                         \
  } while (0)

#define PEB_TRY(expr)          \
  do {                         \
    int _rc = (expr);          \
    if (_rc != PEB_OK) return _rc; \
  } while (0)

// launch + count (bench.py's gpu_launches reads the counter)
#define PEB_LAUNCH(ctx, kernel, grid, block, smem, ...)                        \
  do {                                                                         \
    kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);           \
    (ctx)->launches++;                                                         \
    PEB_CUDA((ctx), cudaGetLastError());                                       \
  } while (0)

// Launch with programmatic dependent launch (PDL): the kernel may be scheduled while the previous
// kernel of the stream is still draining; it must execute pdl_wait() before it touches anything the
// previous kernel wrote.  Hides the ~3 us launch gap between the dependent ICP iteration launches.
#define PEB_LAUNCH_PDL(ctx, kernel, grid_, block_, ...)                                   \
  do {                                                                                    \
    cudaLaunchConfig_t _cfg = {};                                                         \
    _cfg.gridDim = (grid_);                                                               \
    _cfg.blockDim = (block_);                                                             \
    _cfg.dynamicSmemBytes = 0;                                                            \
    _cfg.stream = (ctx)->stream;                                                          \
    cudaLaunchAttribute _attr[1];                                                         \
    _attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                     \
    _attr[0].val.programmaticStreamSerializationAllowed = (ctx)->use_pdl ? 1 : 0;         \
    _cfg.attrs = _attr;                                                                   \
    _cfg.numAttrs = 1;                                                                    \
    (ctx)->launches++;                                                                    \
    PEB_CUDA((ctx), cudaLaunchKernelEx(&_cfg, kernel, __VA_ARGS__));                      \
  } while (0)

static inline int ceil_div(long long a, long long b) { return static_cast<int>((a + b - 1) / b); }

// ---- stages implemented in the other translation units -------------------------------------
// radix_sort.cu
int sort_pairs(peb_ctx* ctx, uint32_t* keys, uint32_t* vals, uint32_t* keys_tmp, uint32_t* vals_tmp, int n,
               int key_bits, uint32_t** keys_out, uint32_t** vals_out);
int exclusive_scan_u32(peb_ctx* ctx, const uint32_t* in, uint32_t* out, int n, uint32_t* d_total);
// grid.cu
int grid_build(peb_ctx* ctx, Grid* g, const float4* d_pts, const float4* d_normals, int n, float occupancy);
int bbox_finite(peb_ctx* ctx, const float4* d_pts, int n, float mn[3], float mx[3], int* n_finite);
// icp.cu
// chain / n_chain: a rejector chain, checked by the caller (n_chain 0: none)
int icp_align_device(peb_ctx* ctx, const float* d_guesses /*nullable: identity*/, size_t H, const peb_icp_params* prm,
                     peb_icp_result* d_results, bool single_mode, const peb_rejector* chain = nullptr, int n_chain = 0);
// multi.cu: fn(ctx i, lo, hi) on every context of m with its shard [lo, hi) of n_items (skipped when empty), device 0's
// on the calling thread; the first failing context is reported in m's error text
int multi_run_sharded(peb_multi* m, const char* what, size_t n_items, int (*fn)(peb_ctx*, size_t lo, size_t hi, void* user),
                      void* user);
// m's error text
int multi_set_error(peb_multi* m, int code, const char* msg);
int icp_output_device(peb_ctx* ctx, float4* d_out);
int nn_search_device(peb_ctx* ctx, const float4* d_q, int nq, int32_t* d_idx, float* d_d2);
// fitness of one transform (device, 16 floats); the record's n_correspondences carries the inlier count
int fitness_device(peb_ctx* ctx, const float* d_T, double max_range, peb_icp_result* d_result);
// brute.cu
int nn_bruteforce_device(peb_ctx* ctx, const float4* d_q, int nq, int32_t* d_idx, float* d_d2);
// voxel.cu
int voxel_grid_device(peb_ctx* ctx, const float4* d_in, int n, float lx, float ly, float lz, unsigned min_pts,
                      float4* d_out, size_t* out_n);
// prefilter.cu
int scene_prefilter_device(peb_ctx* ctx, const float4* d_in, int n, const peb_prefilter_params* prm, float4* d_out,
                           size_t* out_n);
// sac.cu
int sac_plane_device(peb_ctx* ctx, const float4* d_pts, int n, const peb_sac_params* prm, float out_coeff[4],
                     int32_t* d_out_inliers, size_t* out_n_inliers, int32_t* out_iterations);
// cvicp.cu (host pointers in, results on the host)
int cvicp_register_device(peb_ctx* ctx, const float* h_model, size_t n_model, const float* h_scene, size_t n_scene,
                          const peb_cvicp_params* prm, double* poses, size_t n_poses, double* residuals);
// normals.cu
int target_graph_ensure(peb_ctx* ctx);  // builds ctx->tgt_knn for the current target grid if it is not there yet
int normals_knn_device(peb_ctx* ctx, const float4* d_in, int n, int k, const float vp[3], float* d_out8,
                       int32_t* d_out_nn /*nullable, n x k original indices*/);
// cv::ppf_match_3d::computeNormalsPC3d: d_out6 = n rows of x y z nx ny nz (DESIGN.md §13)
int cv_normals_device(peb_ctx* ctx, const float4* d_in, int n, int k, bool flip, const float vp[3], float* d_out6,
                      int32_t* d_out_nn /*nullable, n x k original indices*/);

}  // namespace peb
