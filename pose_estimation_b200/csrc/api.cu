// api.cu — the C ABI of libpe_b200.so (include/pe_b200.h): argument checking, host <-> device
// staging and the mapping of every entry point onto the CUDA stages.  No exceptions leave this
// file and there is no CPU implementation behind any entry point: if the device path cannot run,
// the call fails with a peb_status and a message.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <new>

#include "block_select.cuh"
#include "core_math.cuh"

namespace peb {

int fail(peb_ctx* ctx, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf;
  return code;
}

namespace {

thread_local std::string g_create_error;

// raw records (x, y, z at the head of every `stride` bytes) -> float4 (x, y, z, w_fill)
__global__ void __launch_bounds__(256) repack_kernel(const unsigned char* __restrict__ raw, size_t stride, int n,
                                                     float w_fill, float4* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* r = reinterpret_cast<const float*>(raw + static_cast<size_t>(i) * stride);
  out[i] = make_float4(r[0], r[1], r[2], w_fill);
}

int check_cloud(peb_ctx* ctx, const char* what, const void* pts, size_t n, size_t stride) {
  if (n > 0 && !pts) return fail(ctx, PEB_E_INVALID_ARG, "%s: null pointer with n = %zu", what, n);
  if (stride < 12 || (stride & 3)) return fail(ctx, PEB_E_INVALID_ARG, "%s: stride %zu is not a multiple of 4 >= 12", what, stride);
  if (n > static_cast<size_t>(INT32_MAX) / 2) return fail(ctx, PEB_E_INVALID_ARG, "%s: %zu points exceed the 2^30 limit", what, n);
  return PEB_OK;
}

// host records -> device float4 array (dst must hold n float4)
int upload_cloud(peb_ctx* ctx, const void* pts, size_t n, size_t stride, float w_fill, float4* d_dst) {
  if (n == 0) return PEB_OK;
  const size_t bytes = (n - 1) * stride + 12;  // the last record may be shorter than the stride
  PEB_CUDA(ctx, ctx->d_stage.ensure(bytes));
  PEB_CUDA(ctx, cudaMemcpyAsync(ctx->d_stage.p, pts, bytes, cudaMemcpyHostToDevice, ctx->stream));
  PEB_LAUNCH(ctx, repack_kernel, ceil_div(static_cast<long long>(n), 256), 256, 0,
             static_cast<const unsigned char*>(ctx->d_stage.p), stride, static_cast<int>(n), w_fill, d_dst);
  return PEB_OK;
}

int sync(peb_ctx* ctx) {
  PEB_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return PEB_OK;
}

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

int target_finish(peb_ctx* ctx, size_t n, bool has_normals) {
  ctx->tgt_knn_valid = false;
  ctx->n_tgt = n;
  ctx->tgt_has_normals = has_normals;
  return grid_build(ctx, &ctx->tgt_grid, ctx->tgt_raw.as<float4>(), has_normals ? ctx->tgt_nrm_raw.as<float4>() : nullptr,
                    static_cast<int>(n), ctx->grid_occupancy);
}

int source_finish(peb_ctx* ctx, size_t n) {
  ctx->n_src = n;
  PEB_TRY(grid_build(ctx, &ctx->src_grid, ctx->src.as<float4>(), nullptr, static_cast<int>(n), ctx->src_sort_occupancy));
  ctx->n_src_sorted = ctx->src_grid.view.n;
  ctx->src_set = true;
  return PEB_OK;
}

// records (creating it on first use) the event that orders a replica's copy after this context's staging
int mark_staged(peb_ctx* ctx, cudaEvent_t* ev) {
  if (!*ev) PEB_CUDA(ctx, cudaEventCreateWithFlags(ev, cudaEventDisableTiming));
  PEB_CUDA(ctx, cudaEventRecord(*ev, ctx->stream));
  return PEB_OK;
}

int upload_guesses(peb_ctx* ctx, const float* guesses, size_t H, const float** d_out) {
  *d_out = nullptr;
  if (!guesses) return PEB_OK;
  PEB_CUDA(ctx, ctx->d_guesses.ensure(H * 16 * sizeof(float)));
  PEB_CUDA(ctx, cudaMemcpyAsync(ctx->d_guesses.p, guesses, H * 16 * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  *d_out = ctx->d_guesses.as<float>();
  return PEB_OK;
}

// No C++ exception leaves the library (include/pe_b200.h): the entry points whose host side allocates (std::vector
// staging of the RANSAC candidates and the cv ICP pose tables, stream / event lists, error strings) run behind this.
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

// peb_debug_select_nth: one 1024-thread block per requested rank
struct DebugLoad {
  const float* v;
  __device__ float operator()(int i) const { return v[i]; }
};
template <bool SKIP_NEG>
__global__ void __launch_bounds__(1024) debug_select_nth_kernel(const float* __restrict__ v, int m, const int32_t* __restrict__ nths,
                                                                float* __restrict__ out) {
  __shared__ unsigned hist[2048];
  __shared__ unsigned st[2];
  __shared__ unsigned wsum[32];
  const float r = block_select_nth<DebugLoad, SKIP_NEG>(DebugLoad{v}, m, nths[blockIdx.x], hist, st, wsum);
  if (threadIdx.x == 0) out[blockIdx.x] = r;
}
}  // namespace
}  // namespace peb

using namespace peb;

extern "C" {

PEB_API const char* peb_version(void) { return "pe_b200 0.1 (sm_100a)"; }

PEB_API void peb_icp_params_default(peb_icp_params* p) {
  if (!p) return;
  p->max_iterations = 10;
  p->min_correspondences = 3;
  p->estimator = PEB_ESTIMATOR_SVD;
  p->max_iterations_similar = 0;
  p->max_corr_dist = sqrt(DBL_MAX);
  p->transformation_epsilon = 0.0;
  p->rotation_epsilon = 0.0;
  p->euclidean_fitness_epsilon = -DBL_MAX;
  p->abs_mse_threshold = 1e-12;
  p->rejector_max_dist = 0.0;
  p->fitness_max_range = DBL_MAX;
}

PEB_API int peb_ctx_create(int device, peb_ctx** out) {
  if (!out) return PEB_E_INVALID_ARG;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    cudaGetLastError();
    g_create_error = std::string("peb_ctx_create: no CUDA device (") + cudaGetErrorString(e) +
                     "); libpe_b200 has no CPU fallback";
    return PEB_E_CUDA;
  }
  if (device < 0 || device >= count) {
    g_create_error = "peb_ctx_create: device index out of range";
    return PEB_E_INVALID_ARG;
  }
  cudaDeviceProp prop{};
  cudaGetDeviceProperties(&prop, device);
  if (prop.major != 10) {
    g_create_error = std::string("peb_ctx_create: device '") + prop.name + "' is sm_" + std::to_string(prop.major) +
                     std::to_string(prop.minor) + "; this library carries sm_100a code only";
    return PEB_E_UNSUPPORTED;
  }
  peb_ctx* ctx = new (std::nothrow) peb_ctx();
  if (!ctx) return PEB_E_OOM;
  ctx->device = device;
  DeviceGuard guard(device);
  e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = ctx->d_small.ensure(1 << 20);
  if (e == cudaSuccess) e = ctx->h_small.ensure(1 << 16);
  if (e != cudaSuccess) {
    g_create_error = std::string("peb_ctx_create: ") + cudaGetErrorString(e);
    cudaGetLastError();
    peb_ctx_destroy(ctx);
    return PEB_E_CUDA;
  }
  *out = ctx;
  return PEB_OK;
}

PEB_API void peb_ctx_destroy(peb_ctx* ctx) {
  if (!ctx) return;
  DeviceGuard guard(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  DevBuf* bufs[] = {&ctx->d_small, &ctx->d_scratch, &ctx->d_stage, &ctx->tgt_raw, &ctx->tgt_nrm_raw, &ctx->src, &ctx->work, &ctx->slack, &ctx->anchors, &ctx->nn_cache, &ctx->dbg,
                    &ctx->corr_idx, &ctx->corr_d2, &ctx->partials, &ctx->state, &ctx->trace, &ctx->d_guesses,
                    &ctx->d_results, &ctx->d_aligned, &ctx->vg_in, &ctx->vg_out, &ctx->vg_flags, &ctx->vg_scan,
                    &ctx->vg_starts, &ctx->nrm_in, &ctx->nrm_out, &ctx->brute_keys, &ctx->nn_q, &ctx->nn_idx, &ctx->nn_d2, &ctx->epochs, &ctx->cv_arena};
  for (DevBuf* b : bufs) b->release();
  ctx->sort_scratch.release();
  for (DevBuf& b : ctx->scan_scratch) b.release();
  for (Grid* g : {&ctx->tgt_grid, &ctx->aux_grid, &ctx->src_grid}) {
    g->pts.release();
    g->normals.release();
    g->cell_start.release();
    g->keys.release();
    g->vals.release();
    g->keys_tmp.release();
    g->vals_tmp.release();
  }
  for (cudaEvent_t e : ctx->prof_events) cudaEventDestroy(e);
  for (cudaEvent_t e : ctx->join_events) cudaEventDestroy(e);
  for (cudaStream_t st : ctx->sub_streams) cudaStreamDestroy(st);
  if (ctx->fork_event) cudaEventDestroy(ctx->fork_event);
  if (ctx->tgt_stage_event) cudaEventDestroy(ctx->tgt_stage_event);
  if (ctx->src_stage_event) cudaEventDestroy(ctx->src_stage_event);
  ctx->h_stage.release();
  ctx->h_small.release();
  ctx->h_sac.release();
  ctx->h_cv.release();
  if (ctx->stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

PEB_API const char* peb_last_error(const peb_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }
PEB_API void* peb_ctx_stream(peb_ctx* ctx) { return ctx ? static_cast<void*>(ctx->stream) : nullptr; }
PEB_API uint64_t peb_ctx_launch_count(const peb_ctx* ctx) { return ctx ? ctx->launches : 0; }

PEB_API int peb_ctx_set_int(peb_ctx* ctx, const char* key, int value) {
  if (!ctx || !key) return PEB_E_INVALID_ARG;
  if (!strcmp(key, "nn_group")) {
    if (value != 1 && value != 2 && value != 4 && value != 8 && value != 16)
      return fail(ctx, PEB_E_INVALID_ARG, "nn_group must be 1, 2, 4, 8 or 16");
    ctx->nn_group = value;
    return PEB_OK;
  }
  if (!strcmp(key, "grid_occupancy_x100")) {
    if (value < 25 || value > 6400) return fail(ctx, PEB_E_INVALID_ARG, "grid_occupancy_x100 out of [25, 6400]");
    ctx->grid_occupancy = value / 100.0f;
    return PEB_OK;
  }
  if (!strcmp(key, "source_sort_occupancy")) {
    if (value < 1 || value > 1024) return fail(ctx, PEB_E_INVALID_ARG, "source_sort_occupancy out of [1, 1024]");
    ctx->src_sort_occupancy = static_cast<float>(value);
    return PEB_OK;
  }
  if (!strcmp(key, "cert_margin_x1000")) {
    if (value < 0 || value > 4000) return fail(ctx, PEB_E_INVALID_ARG, "cert_margin_x1000 out of [0, 4000]");
    ctx->cert_margin = value / 1000.0f;
    return PEB_OK;
  }
  if (!strcmp(key, "seed_guard_x10")) {
    if (value < 0 || value > 100000) return fail(ctx, PEB_E_INVALID_ARG, "seed_guard_x10 out of [0, 100000]");
    ctx->seed_guard = value / 10.0f;
    return PEB_OK;
  }
  if (!strcmp(key, "batch_streams")) {
    if (value < 0 || value > 32) return fail(ctx, PEB_E_INVALID_ARG, "batch_streams out of [0, 32]");
    ctx->batch_streams = value;
    return PEB_OK;
  }
  if (!strcmp(key, "blocks_factor")) {
    if (value < 0 || value > 4096) return fail(ctx, PEB_E_INVALID_ARG, "blocks_factor out of [0, 4096]");
    ctx->blocks_factor = value;
    return PEB_OK;
  }
  if (!strcmp(key, "coop_max_rows")) {
    if (value < 0 || value > (1 << 20)) return fail(ctx, PEB_E_INVALID_ARG, "coop_max_rows out of [0, 2^20]");
    ctx->coop_max_rows = value;
    return PEB_OK;
  }
  if (!strcmp(key, "blocks_factor_cold")) {
    if (value < 0 || value > 4096) return fail(ctx, PEB_E_INVALID_ARG, "blocks_factor_cold out of [0, 4096]");
    ctx->blocks_factor_cold = value;
    return PEB_OK;
  }
  if (!strcmp(key, "blocks_factor_search")) {
    if (value < 0 || value > 4096) return fail(ctx, PEB_E_INVALID_ARG, "blocks_factor_search out of [0, 4096]");
    ctx->blocks_factor_search = value;
    return PEB_OK;
  }
  if (!strcmp(key, "split_moments")) {
    if (value < 0 || value > 1) return fail(ctx, PEB_E_INVALID_ARG, "split_moments must be 0 or 1");
    ctx->split_moments = value;
    return PEB_OK;
  }
  if (!strcmp(key, "split_min_hyp")) {
    if (value < 2) return fail(ctx, PEB_E_INVALID_ARG, "split_min_hyp must be >= 2 (batches only)");
    ctx->split_min_hyp = value;
    return PEB_OK;
  }
  if (!strcmp(key, "flag_deps")) {
    ctx->flag_deps = value != 0;
    return PEB_OK;
  }
  if (!strcmp(key, "pdl")) {
    ctx->use_pdl = value != 0;
    return PEB_OK;
  }
  if (!strcmp(key, "debug_timers")) {
    ctx->debug_timers = value != 0;
    return PEB_OK;
  }
  if (!strcmp(key, "anchor_seed")) {
    ctx->anchor_seed = value != 0;
    return PEB_OK;
  }
  if (!strcmp(key, "warm_start")) {
    ctx->warm_start = value != 0;
    return PEB_OK;
  }
  if (!strcmp(key, "warm_graph")) {
    if (value < 0 || value > 1) return fail(ctx, PEB_E_INVALID_ARG, "warm_graph must be 0 or 1");
    ctx->warm_graph = value;
    return PEB_OK;
  }
  if (!strcmp(key, "warm_graph_kappa_x100")) {
    if (value < 0 || value > 100000) return fail(ctx, PEB_E_INVALID_ARG, "warm_graph_kappa_x100 out of [0, 100000]");
    ctx->warm_graph_kappa = value / 100.0f;
    return PEB_OK;
  }
  if (!strcmp(key, "warm_graph_queue")) {
    if (value != 0 && value != 8 && value != 16) return fail(ctx, PEB_E_INVALID_ARG, "warm_graph_queue must be 0, 8 or 16");
    ctx->warm_graph_queue = value;
    return PEB_OK;
  }
  if (!strcmp(key, "warm_graph_flat")) {
    if (value < 0 || value > 1) return fail(ctx, PEB_E_INVALID_ARG, "warm_graph_flat must be 0 or 1");
    ctx->warm_graph_flat = value;
    return PEB_OK;
  }
  if (!strcmp(key, "warm_graph_flat_from") || !strcmp(key, "warm_graph_flat_until")) {
    if (value < 0) return fail(ctx, PEB_E_INVALID_ARG, "%s must be >= 0", key);
    (key[16] == 'f' ? ctx->warm_graph_flat_from : ctx->warm_graph_flat_until) = value;
    return PEB_OK;
  }
  if (!strcmp(key, "warm_graph_peek")) {
    if (value < 0) return fail(ctx, PEB_E_INVALID_ARG, "warm_graph_peek must be >= 0");
    ctx->warm_graph_peek = value;
    return PEB_OK;
  }
  if (!strcmp(key, "cold_graph")) {
    if (value < 0 || value > 1) return fail(ctx, PEB_E_INVALID_ARG, "cold_graph must be 0 or 1");
    ctx->cold_graph = value;
    return PEB_OK;
  }
  if (!strcmp(key, "warm_graph_min_hyp")) {
    if (value < 2) return fail(ctx, PEB_E_INVALID_ARG, "warm_graph_min_hyp must be >= 2 (batches only)");
    ctx->warm_graph_min_hyp = value;
    return PEB_OK;
  }
  if (!strcmp(key, "warm_bin")) {
    if (value < 0 || value > 1) return fail(ctx, PEB_E_INVALID_ARG, "warm_bin must be 0 or 1");
    ctx->warm_bin = value;
    return PEB_OK;
  }
  if (!strcmp(key, "warm_upfront")) {
    if (value < 0 || value > 3) return fail(ctx, PEB_E_INVALID_ARG, "warm_upfront must be 0 (off), 1 / 2 (2 x 2 rows) or 3 (3 x 3 rows)");
    ctx->warm_upfront = value;
    return PEB_OK;
  }
  if (!strcmp(key, "nn_cache_from")) {
    if (value < 0) return fail(ctx, PEB_E_INVALID_ARG, "nn_cache_from must be >= 0 (0: off; launch 0 is never a warm launch)");
    ctx->nn_cache_from = value;
    return PEB_OK;
  }
  if (!strcmp(key, "nn_cache_r_x100")) {
    if (value < 5 || value > 400) return fail(ctx, PEB_E_INVALID_ARG, "nn_cache_r_x100 out of [5, 400]");
    ctx->nn_cache_r = value / 100.0f;
    return PEB_OK;
  }
  if (!strcmp(key, "warm_upfront_from")) {
    if (value < 1) return fail(ctx, PEB_E_INVALID_ARG, "warm_upfront_from must be >= 1 (launch 0 is never a warm launch)");
    ctx->warm_upfront_from = value;
    return PEB_OK;
  }
  if (!strcmp(key, "profile")) {
    if (value < 0 || value > 2) return fail(ctx, PEB_E_INVALID_ARG, "profile must be 0, 1 or 2");
    ctx->profile = value != 0;
    ctx->profile_level = value;
    ctx->prof_launches = 0;
    return PEB_OK;
  }
  return fail(ctx, PEB_E_INVALID_ARG, "unknown option '%s'", key);
}

// Waits for everything queued on the context; PEB_E_CUDA if the last batched align raised its internal-error flag
// (the asynchronous *_dev entry points cannot report it when they return).
PEB_API int peb_sync(peb_ctx* ctx) {
  if (!ctx) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  int* h_flag = ctx->h_small.as<int>() + 64;
  *h_flag = 0;
  if (ctx->last_err_flag)
    PEB_CUDA(ctx, cudaMemcpyAsync(h_flag, ctx->last_err_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  PEB_TRY(sync(ctx));
  if (*h_flag != 0)
    return fail(ctx, PEB_E_CUDA, "a per-hypothesis dependency wait of the last batched align ran into its bound (internal "
                                 "error; peb_ctx_set_int(ctx, \"flag_deps\", 0) restores whole-grid dependencies)");
  return PEB_OK;
}

// ---- VoxelGrid ---------------------------------------------------------------------------------
PEB_API int peb_voxel_grid_dev(peb_ctx* ctx, const void* d_xyz4, size_t n, float lx, float ly, float lz, unsigned min_pts,
                               void* d_out_xyz4, size_t* out_n) {
  if (!ctx || !out_n) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  if (n > 0 && (!d_xyz4 || !d_out_xyz4)) return fail(ctx, PEB_E_INVALID_ARG, "voxel_grid_dev: null device pointer");
  if (n > static_cast<size_t>(INT32_MAX) / 2) return fail(ctx, PEB_E_INVALID_ARG, "voxel_grid: too many points");
  return voxel_grid_device(ctx, static_cast<const float4*>(d_xyz4), static_cast<int>(n), lx, ly, lz, min_pts,
                           static_cast<float4*>(d_out_xyz4), out_n);
}

PEB_API int peb_voxel_grid(peb_ctx* ctx, const void* pts, size_t n, size_t stride, float lx, float ly, float lz,
                           unsigned min_pts, float* out_xyz4, size_t* out_n) {
  if (!ctx || !out_n) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  *out_n = 0;
  PEB_TRY(check_cloud(ctx, "voxel_grid", pts, n, stride));
  if (n > 0 && !out_xyz4) return fail(ctx, PEB_E_INVALID_ARG, "voxel_grid: null output");
  PEB_CUDA(ctx, ctx->vg_in.ensure(n * sizeof(float4)));
  PEB_CUDA(ctx, ctx->vg_out.ensure(n * sizeof(float4)));
  PEB_TRY(upload_cloud(ctx, pts, n, stride, 1.0f, ctx->vg_in.as<float4>()));
  size_t m = 0;
  PEB_TRY(voxel_grid_device(ctx, ctx->vg_in.as<float4>(), static_cast<int>(n), lx, ly, lz, min_pts,
                            ctx->vg_out.as<float4>(), &m));
  if (m > 0)
    PEB_CUDA(ctx, cudaMemcpyAsync(out_xyz4, ctx->vg_out.p, m * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
  PEB_TRY(sync(ctx));
  *out_n = m;
  return PEB_OK;
}

// ---- scene pre-filter ----------------------------------------------------------------------------
PEB_API int peb_scene_prefilter_dev(peb_ctx* ctx, const void* d_xyz4, size_t n, const peb_prefilter_params* params,
                                    void* d_out_xyz4, size_t* out_n) {
  if (!ctx || !params || !out_n) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  if (n > 0 && (!d_xyz4 || !d_out_xyz4)) return fail(ctx, PEB_E_INVALID_ARG, "scene_prefilter_dev: null device pointer");
  if (n > static_cast<size_t>(INT32_MAX) / 2) return fail(ctx, PEB_E_INVALID_ARG, "scene_prefilter: too many points");
  return scene_prefilter_device(ctx, static_cast<const float4*>(d_xyz4), static_cast<int>(n), params,
                                static_cast<float4*>(d_out_xyz4), out_n);
}

PEB_API int peb_scene_prefilter(peb_ctx* ctx, const void* pts, size_t n, size_t stride, const peb_prefilter_params* params,
                                float* out_xyz4, size_t* out_n) {
  if (!ctx || !params || !out_n) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  *out_n = 0;
  PEB_TRY(check_cloud(ctx, "scene_prefilter", pts, n, stride));
  if (n > 0 && !out_xyz4) return fail(ctx, PEB_E_INVALID_ARG, "scene_prefilter: null output");
  PEB_CUDA(ctx, ctx->vg_in.ensure(n * sizeof(float4)));
  PEB_CUDA(ctx, ctx->vg_out.ensure(n * sizeof(float4)));
  PEB_TRY(upload_cloud(ctx, pts, n, stride, 1.0f, ctx->vg_in.as<float4>()));
  size_t m = 0;
  PEB_TRY(scene_prefilter_device(ctx, ctx->vg_in.as<float4>(), static_cast<int>(n), params, ctx->vg_out.as<float4>(), &m));
  if (m > 0)
    PEB_CUDA(ctx, cudaMemcpyAsync(out_xyz4, ctx->vg_out.p, m * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
  PEB_TRY(sync(ctx));
  *out_n = m;
  return PEB_OK;
}

// ---- SACSegmentation (plane, RANSAC) --------------------------------------------------------------
PEB_API void peb_sac_params_default(peb_sac_params* p) {
  if (!p) return;
  // [PCL] segmentation/sac_segmentation.h : SACSegmentation() defaults; seed of SampleConsensusModel(random = false)
  p->distance_threshold = 0.0;
  p->probability = 0.99;
  p->max_iterations = 50;
  p->optimize_coefficients = 1;
  p->seed = 12345u;
  p->reserved = 0;
}

static int sac_plane_dev_impl(peb_ctx* ctx, const void* d_xyz4, size_t n, const peb_sac_params* params, float out_coeff[4],
                              int32_t* d_out_inliers, size_t* out_n_inliers, int32_t* out_iterations) {
  if (!ctx || !params || !out_coeff || !out_n_inliers) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  if (n > 0 && !d_xyz4) return fail(ctx, PEB_E_INVALID_ARG, "sac_plane_dev: null device pointer");
  if (n > static_cast<size_t>(INT32_MAX) / 2) return fail(ctx, PEB_E_INVALID_ARG, "sac_plane: too many points");
  return sac_plane_device(ctx, static_cast<const float4*>(d_xyz4), static_cast<int>(n), params, out_coeff, d_out_inliers,
                          out_n_inliers, out_iterations);
}

static int sac_plane_impl(peb_ctx* ctx, const void* pts, size_t n, size_t stride, const peb_sac_params* params,
                          float out_coeff[4], int32_t* out_inliers, size_t* out_n_inliers, int32_t* out_iterations) {
  if (!ctx || !params || !out_coeff || !out_n_inliers) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  *out_n_inliers = 0;
  PEB_TRY(check_cloud(ctx, "sac_plane", pts, n, stride));
  PEB_CUDA(ctx, ctx->vg_in.ensure(std::max<size_t>(n, 1) * sizeof(float4)));
  PEB_CUDA(ctx, ctx->vg_out.ensure(std::max<size_t>(n, 1) * sizeof(int32_t)));
  PEB_TRY(upload_cloud(ctx, pts, n, stride, 1.0f, ctx->vg_in.as<float4>()));
  size_t m = 0;
  PEB_TRY(sac_plane_device(ctx, ctx->vg_in.as<float4>(), static_cast<int>(n), params, out_coeff,
                           out_inliers ? ctx->vg_out.as<int32_t>() : nullptr, &m, out_iterations));
  if (out_inliers && m > 0)
    PEB_CUDA(ctx, cudaMemcpyAsync(out_inliers, ctx->vg_out.p, m * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  PEB_TRY(sync(ctx));
  *out_n_inliers = m;
  return PEB_OK;
}

// ---- create_surface_match_pc in one call ---------------------------------------------------------------
static int scene_prepare_impl(peb_ctx* ctx, const void* pts, size_t n, size_t stride, const peb_prefilter_params* filter,
                              int num_planes, const peb_sac_params* sac, float leaf, float* out_xyz4, size_t* out_n,
                              float* out_planes) {
  if (!ctx || !filter || !out_n) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  *out_n = 0;
  PEB_TRY(check_cloud(ctx, "scene_prepare", pts, n, stride));
  if (num_planes < 0 || num_planes > PEB_PREFILTER_MAX_PLANES)
    return fail(ctx, PEB_E_INVALID_ARG, "scene_prepare: num_planes %d out of [0, %d]", num_planes, PEB_PREFILTER_MAX_PLANES);
  if (num_planes > 0 && !sac) return fail(ctx, PEB_E_INVALID_ARG, "scene_prepare: plane removal needs RANSAC parameters");
  if (n > 0 && !out_xyz4) return fail(ctx, PEB_E_INVALID_ARG, "scene_prepare: null output");
  if (n == 0) return PEB_OK;
  PEB_CUDA(ctx, ctx->vg_in.ensure(n * sizeof(float4)));
  PEB_CUDA(ctx, ctx->vg_out.ensure(n * sizeof(float4)));
  float4* cur = ctx->vg_in.as<float4>();
  float4* other = ctx->vg_out.as<float4>();
  PEB_TRY(upload_cloud(ctx, pts, n, stride, 1.0f, cur));
  size_t m = 0;
  peb_prefilter_params f = *filter;
  f.n_planes = 0;  // :246-256, NaN removal + sphere filter
  PEB_TRY(scene_prefilter_device(ctx, cur, static_cast<int>(n), &f, other, &m));
  std::swap(cur, other);
  for (int k = 0; k < num_planes; ++k) {  // remove_planes, recursively in the reference
    float coeff[4] = {0.f, 0.f, 0.f, 0.f};
    size_t n_inl = 0;
    PEB_TRY(sac_plane_device(ctx, cur, static_cast<int>(m), sac, coeff, nullptr, &n_inl, nullptr));
    if (out_planes) std::copy(coeff, coeff + 4, out_planes + 4 * k);
    if (coeff[0] == 0.f && coeff[1] == 0.f && coeff[2] == 0.f && coeff[3] == 0.f) continue;  // no model: nothing is near "the plane"
    peb_prefilter_params band{};
    band.plane_band = filter->plane_band;
    band.n_planes = 1;
    std::copy(coeff, coeff + 4, band.planes);
    size_t kept = 0;
    PEB_TRY(scene_prefilter_device(ctx, cur, static_cast<int>(m), &band, other, &kept));
    std::swap(cur, other);
    m = kept;
  }
  if (leaf > 0.0f && m > 0) {
    size_t v = 0;
    PEB_TRY(voxel_grid_device(ctx, cur, static_cast<int>(m), leaf, leaf, leaf, 0, other, &v));
    std::swap(cur, other);
    m = v;
  }
  if (m > 0) PEB_CUDA(ctx, cudaMemcpyAsync(out_xyz4, cur, m * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
  PEB_TRY(sync(ctx));
  *out_n = m;
  return PEB_OK;
}

// ---- cv::ppf_match_3d::ICP::registerModelToScene ----------------------------------------------------
static int cvicp_register_impl(peb_ctx* ctx, const float* model_xyzn, size_t n_model, const float* scene_xyzn, size_t n_scene,
                               const peb_cvicp_params* params, double* poses, size_t n_poses, double* out_residuals) {
  if (!ctx || !params) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  if (n_poses == 0) return PEB_OK;
  if (!model_xyzn || !scene_xyzn || !poses) return fail(ctx, PEB_E_INVALID_ARG, "cvicp_register: null model / scene / poses");
  return cvicp_register_device(ctx, model_xyzn, n_model, scene_xyzn, n_scene, params, poses, n_poses, out_residuals);
}

// ---- NormalEstimation ---------------------------------------------------------------------------
PEB_API int peb_normals_knn_dev(peb_ctx* ctx, const void* d_xyz4, size_t n, int k, const float viewpoint[3],
                                void* d_out_normal8) {
  if (!ctx) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  if (n > 0 && (!d_xyz4 || !d_out_normal8)) return fail(ctx, PEB_E_INVALID_ARG, "normals_knn_dev: null device pointer");
  if (n > static_cast<size_t>(INT32_MAX) / 2) return fail(ctx, PEB_E_INVALID_ARG, "normals_knn: too many points");
  const float zero[3] = {0.f, 0.f, 0.f};
  return normals_knn_device(ctx, static_cast<const float4*>(d_xyz4), static_cast<int>(n), k, viewpoint ? viewpoint : zero,
                            static_cast<float*>(d_out_normal8), nullptr);
}

PEB_API int peb_normals_knn_ex(peb_ctx* ctx, const void* pts, size_t n, size_t stride, int k, const float viewpoint[3],
                               float* out_normal8, int32_t* out_nn_idx) {
  if (!ctx) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  PEB_TRY(check_cloud(ctx, "normals_knn", pts, n, stride));
  if (n > 0 && !out_normal8) return fail(ctx, PEB_E_INVALID_ARG, "normals_knn: null output");
  if (k < 1) return fail(ctx, PEB_E_INVALID_ARG, "normals_knn: k must be >= 1 (got %d)", k);
  const float zero[3] = {0.f, 0.f, 0.f};
  PEB_CUDA(ctx, ctx->nrm_in.ensure(n * sizeof(float4)));
  PEB_CUDA(ctx, ctx->nrm_out.ensure(n * 8 * sizeof(float)));
  int32_t* d_nn = nullptr;
  if (out_nn_idx) {
    PEB_CUDA(ctx, ctx->nn_idx.ensure(n * static_cast<size_t>(k) * sizeof(int32_t)));
    d_nn = ctx->nn_idx.as<int32_t>();
  }
  PEB_TRY(upload_cloud(ctx, pts, n, stride, 1.0f, ctx->nrm_in.as<float4>()));
  PEB_TRY(normals_knn_device(ctx, ctx->nrm_in.as<float4>(), static_cast<int>(n), k, viewpoint ? viewpoint : zero,
                             ctx->nrm_out.as<float>(), d_nn));
  if (n > 0) {
    PEB_CUDA(ctx, cudaMemcpyAsync(out_normal8, ctx->nrm_out.p, n * 8 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    if (out_nn_idx)
      PEB_CUDA(ctx, cudaMemcpyAsync(out_nn_idx, d_nn, n * static_cast<size_t>(k) * sizeof(int32_t), cudaMemcpyDeviceToHost,
                                    ctx->stream));
  }
  return sync(ctx);
}

PEB_API int peb_normals_knn(peb_ctx* ctx, const void* pts, size_t n, size_t stride, int k, const float viewpoint[3],
                            float* out_normal8) {
  return peb_normals_knn_ex(ctx, pts, n, stride, k, viewpoint, out_normal8, nullptr);
}

// ---- cv::ppf_match_3d::computeNormalsPC3d -------------------------------------------------------
PEB_API int peb_cv_normals_dev(peb_ctx* ctx, const void* d_xyz4, size_t n, int k, int flip_viewpoint, const float viewpoint[3],
                               void* d_out_xyzn6) {
  if (!ctx) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  if (n > 0 && (!d_xyz4 || !d_out_xyzn6)) return fail(ctx, PEB_E_INVALID_ARG, "cv_normals_dev: null device pointer");
  if (n > static_cast<size_t>(INT32_MAX) / 2) return fail(ctx, PEB_E_INVALID_ARG, "cv_normals: too many points");
  const float zero[3] = {0.f, 0.f, 0.f};
  return cv_normals_device(ctx, static_cast<const float4*>(d_xyz4), static_cast<int>(n), k, flip_viewpoint != 0,
                           viewpoint ? viewpoint : zero, static_cast<float*>(d_out_xyzn6), nullptr);
}

PEB_API int peb_cv_normals(peb_ctx* ctx, const void* pts, size_t n, size_t stride, int k, int flip_viewpoint,
                           const float viewpoint[3], float* out_xyzn6, int32_t* out_nn_idx) {
  if (!ctx) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  PEB_TRY(check_cloud(ctx, "cv_normals", pts, n, stride));
  if (n > 0 && !out_xyzn6) return fail(ctx, PEB_E_INVALID_ARG, "cv_normals: null output");
  if (k < 1) return fail(ctx, PEB_E_INVALID_ARG, "cv_normals: k must be >= 1 (got %d)", k);
  if (k > 192) return fail(ctx, PEB_E_UNSUPPORTED, "cv_normals: k = %d > 192 has no CUDA path (no CPU fallback)", k);
  if (n == 0) return PEB_OK;
  const float zero[3] = {0.f, 0.f, 0.f};
  PEB_CUDA(ctx, ctx->nrm_in.ensure(n * sizeof(float4)));
  PEB_CUDA(ctx, ctx->nrm_out.ensure(n * 6 * sizeof(float)));
  int32_t* d_nn = nullptr;
  if (out_nn_idx) {
    PEB_CUDA(ctx, ctx->nn_idx.ensure(n * static_cast<size_t>(k) * sizeof(int32_t)));
    d_nn = ctx->nn_idx.as<int32_t>();
  }
  PEB_TRY(upload_cloud(ctx, pts, n, stride, 1.0f, ctx->nrm_in.as<float4>()));
  PEB_TRY(cv_normals_device(ctx, ctx->nrm_in.as<float4>(), static_cast<int>(n), k, flip_viewpoint != 0,
                            viewpoint ? viewpoint : zero, ctx->nrm_out.as<float>(), d_nn));
  PEB_CUDA(ctx, cudaMemcpyAsync(out_xyzn6, ctx->nrm_out.p, n * 6 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  if (out_nn_idx)
    PEB_CUDA(ctx, cudaMemcpyAsync(out_nn_idx, d_nn, n * static_cast<size_t>(k) * sizeof(int32_t), cudaMemcpyDeviceToHost,
                                  ctx->stream));
  return sync(ctx);
}

// ---- target / source -----------------------------------------------------------------------------
PEB_API int peb_target_stage(peb_ctx* ctx, const void* pts, size_t n, size_t stride, const void* normals, size_t nstride) {
  if (!ctx) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  ctx->tgt_grid.valid = false;
  ctx->tgt_staged = false;
  PEB_TRY(check_cloud(ctx, "target_set", pts, n, stride));
  if (normals) PEB_TRY(check_cloud(ctx, "target_set(normals)", normals, n, nstride));
  PEB_CUDA(ctx, ctx->tgt_raw.ensure(n * sizeof(float4)));
  PEB_TRY(upload_cloud(ctx, pts, n, stride, 1.0f, ctx->tgt_raw.as<float4>()));
  if (normals) {
    PEB_CUDA(ctx, ctx->tgt_nrm_raw.ensure(n * sizeof(float4)));
    PEB_TRY(upload_cloud(ctx, normals, n, nstride, 0.0f, ctx->tgt_nrm_raw.as<float4>()));
  }
  ctx->n_tgt = n;
  ctx->tgt_has_normals = normals != nullptr;
  PEB_TRY(mark_staged(ctx, &ctx->tgt_stage_event));
  ctx->tgt_staged = true;
  return PEB_OK;
}

PEB_API int peb_target_build(peb_ctx* ctx) {
  if (!ctx) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  if (!ctx->tgt_staged) return fail(ctx, PEB_E_NO_TARGET, "target_build: no staged target (peb_target_stage / peb_target_clone)");
  return target_finish(ctx, ctx->n_tgt, ctx->tgt_has_normals);
}

PEB_API int peb_target_set(peb_ctx* ctx, const void* pts, size_t n, size_t stride, const void* normals, size_t nstride) {
  const int rc = peb_target_stage(ctx, pts, n, stride, normals, nstride);
  return rc != PEB_OK ? rc : peb_target_build(ctx);
}

// dst's target becomes a replica of src's staged cloud: device-to-device (NVLink between peers), ordered after
// src's staging by an event, then the same deterministic grid build => the replicas are identical
PEB_API int peb_target_clone(peb_ctx* dst, peb_ctx* src) {
  if (!dst || !src) return PEB_E_INVALID_ARG;
  DeviceGuard guard(dst->device);
  dst->tgt_grid.valid = false;
  dst->tgt_staged = false;
  if (!src->tgt_staged) return fail(dst, PEB_E_NO_TARGET, "target_clone: the source context has no staged target");
  if (dst == src) return peb_target_build(dst);
  const size_t n = src->n_tgt;
  PEB_CUDA(dst, dst->tgt_raw.ensure(n * sizeof(float4)));
  PEB_CUDA(dst, cudaStreamWaitEvent(dst->stream, src->tgt_stage_event, 0));
  if (n) PEB_CUDA(dst, cudaMemcpyPeerAsync(dst->tgt_raw.p, dst->device, src->tgt_raw.p, src->device, n * sizeof(float4), dst->stream));
  if (src->tgt_has_normals) {
    PEB_CUDA(dst, dst->tgt_nrm_raw.ensure(n * sizeof(float4)));
    if (n) PEB_CUDA(dst, cudaMemcpyPeerAsync(dst->tgt_nrm_raw.p, dst->device, src->tgt_nrm_raw.p, src->device, n * sizeof(float4), dst->stream));
  }
  dst->n_tgt = n;
  dst->tgt_has_normals = src->tgt_has_normals;
  PEB_TRY(mark_staged(dst, &dst->tgt_stage_event));
  dst->tgt_staged = true;
  return target_finish(dst, n, dst->tgt_has_normals);
}

PEB_API int peb_target_set_dev(peb_ctx* ctx, const void* d_xyz4, size_t n, const void* d_normal4) {
  if (!ctx) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  ctx->tgt_grid.valid = false;
  ctx->tgt_staged = false;
  if (n > 0 && !d_xyz4) return fail(ctx, PEB_E_INVALID_ARG, "target_set_dev: null device pointer");
  if (n > static_cast<size_t>(INT32_MAX) / 2) return fail(ctx, PEB_E_INVALID_ARG, "target_set: too many points");
  PEB_CUDA(ctx, ctx->tgt_raw.ensure(n * sizeof(float4)));
  if (n) PEB_CUDA(ctx, cudaMemcpyAsync(ctx->tgt_raw.p, d_xyz4, n * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream));
  if (d_normal4) {
    PEB_CUDA(ctx, ctx->tgt_nrm_raw.ensure(n * sizeof(float4)));
    if (n) PEB_CUDA(ctx, cudaMemcpyAsync(ctx->tgt_nrm_raw.p, d_normal4, n * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream));
  }
  ctx->n_tgt = n;
  ctx->tgt_has_normals = d_normal4 != nullptr;
  PEB_TRY(mark_staged(ctx, &ctx->tgt_stage_event));
  ctx->tgt_staged = true;
  return target_finish(ctx, n, d_normal4 != nullptr);
}

PEB_API int peb_source_stage(peb_ctx* ctx, const void* pts, size_t n, size_t stride) {
  if (!ctx) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  ctx->src_set = false;
  ctx->src_staged = false;
  PEB_TRY(check_cloud(ctx, "source_set", pts, n, stride));
  PEB_CUDA(ctx, ctx->src.ensure(n * sizeof(float4)));
  PEB_TRY(upload_cloud(ctx, pts, n, stride, 1.0f, ctx->src.as<float4>()));
  ctx->n_src = n;
  PEB_TRY(mark_staged(ctx, &ctx->src_stage_event));
  ctx->src_staged = true;
  return PEB_OK;
}

PEB_API int peb_source_build(peb_ctx* ctx) {
  if (!ctx) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  if (!ctx->src_staged) return fail(ctx, PEB_E_NO_SOURCE, "source_build: no staged source (peb_source_stage / peb_source_clone)");
  return source_finish(ctx, ctx->n_src);
}

PEB_API int peb_source_set(peb_ctx* ctx, const void* pts, size_t n, size_t stride) {
  const int rc = peb_source_stage(ctx, pts, n, stride);
  return rc != PEB_OK ? rc : peb_source_build(ctx);
}

PEB_API int peb_source_clone(peb_ctx* dst, peb_ctx* src) {
  if (!dst || !src) return PEB_E_INVALID_ARG;
  DeviceGuard guard(dst->device);
  dst->src_set = false;
  dst->src_staged = false;
  if (!src->src_staged) return fail(dst, PEB_E_NO_SOURCE, "source_clone: the source context has no staged source");
  if (dst == src) return peb_source_build(dst);
  const size_t n = src->n_src;
  PEB_CUDA(dst, dst->src.ensure(n * sizeof(float4)));
  PEB_CUDA(dst, cudaStreamWaitEvent(dst->stream, src->src_stage_event, 0));
  if (n) PEB_CUDA(dst, cudaMemcpyPeerAsync(dst->src.p, dst->device, src->src.p, src->device, n * sizeof(float4), dst->stream));
  dst->n_src = n;
  PEB_TRY(mark_staged(dst, &dst->src_stage_event));
  dst->src_staged = true;
  return source_finish(dst, n);
}

// direct loads / copies between the two devices where the hardware allows it (NVLink / NVSwitch on a B200 box);
// without it cudaMemcpyPeerAsync stages through the host and still works
PEB_API int peb_ctx_enable_peer(peb_ctx* ctx, const peb_ctx* peer) {
  if (!ctx || !peer) return PEB_E_INVALID_ARG;
  if (ctx->device == peer->device) return PEB_OK;
  DeviceGuard guard(ctx->device);
  int can = 0;
  if (cudaDeviceCanAccessPeer(&can, ctx->device, peer->device) == cudaSuccess && can) {
    const cudaError_t e = cudaDeviceEnablePeerAccess(peer->device, 0);
    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) can = 0;
  }
  cudaGetLastError();
  return can ? PEB_OK : PEB_E_UNSUPPORTED;
}

PEB_API int peb_source_set_dev(peb_ctx* ctx, const void* d_xyz4, size_t n) {
  if (!ctx) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  ctx->src_set = false;
  ctx->src_staged = false;
  if (n > 0 && !d_xyz4) return fail(ctx, PEB_E_INVALID_ARG, "source_set_dev: null device pointer");
  if (n > static_cast<size_t>(INT32_MAX) / 2) return fail(ctx, PEB_E_INVALID_ARG, "source_set: too many points");
  PEB_CUDA(ctx, ctx->src.ensure(n * sizeof(float4)));
  if (n) PEB_CUDA(ctx, cudaMemcpyAsync(ctx->src.p, d_xyz4, n * sizeof(float4), cudaMemcpyDeviceToDevice, ctx->stream));
  ctx->n_src = n;
  PEB_TRY(mark_staged(ctx, &ctx->src_stage_event));
  ctx->src_staged = true;
  return source_finish(ctx, n);
}

// ---- nearest neighbour ------------------------------------------------------------------------------
static int nn_common(peb_ctx* ctx, const void* queries, size_t nq, size_t stride, int32_t* out_idx, float* out_d2,
                     bool brute) {
  if (!ctx) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  PEB_TRY(check_cloud(ctx, "nn_search", queries, nq, stride));
  if (nq > 0 && (!out_idx || !out_d2)) return fail(ctx, PEB_E_INVALID_ARG, "nn_search: null output");
  if (!ctx->tgt_grid.valid) return fail(ctx, PEB_E_NO_TARGET, "nn_search: no target set (peb_target_set)");
  PEB_CUDA(ctx, ctx->nn_q.ensure(nq * sizeof(float4)));
  PEB_CUDA(ctx, ctx->nn_idx.ensure(nq * sizeof(int32_t)));
  PEB_CUDA(ctx, ctx->nn_d2.ensure(nq * sizeof(float)));
  PEB_TRY(upload_cloud(ctx, queries, nq, stride, 1.0f, ctx->nn_q.as<float4>()));
  if (brute)
    PEB_TRY(nn_bruteforce_device(ctx, ctx->nn_q.as<float4>(), static_cast<int>(nq), ctx->nn_idx.as<int32_t>(), ctx->nn_d2.as<float>()));
  else
    PEB_TRY(nn_search_device(ctx, ctx->nn_q.as<float4>(), static_cast<int>(nq), ctx->nn_idx.as<int32_t>(), ctx->nn_d2.as<float>()));
  if (nq) {
    PEB_CUDA(ctx, cudaMemcpyAsync(out_idx, ctx->nn_idx.p, nq * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    PEB_CUDA(ctx, cudaMemcpyAsync(out_d2, ctx->nn_d2.p, nq * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  }
  return sync(ctx);
}

PEB_API int peb_nn_search(peb_ctx* ctx, const void* queries, size_t nq, size_t stride, int32_t* out_idx, float* out_d2) {
  return nn_common(ctx, queries, nq, stride, out_idx, out_d2, false);
}
PEB_API int peb_nn_search_bruteforce(peb_ctx* ctx, const void* queries, size_t nq, size_t stride, int32_t* out_idx,
                                     float* out_d2) {
  return nn_common(ctx, queries, nq, stride, out_idx, out_d2, true);
}

// ---- ICP ---------------------------------------------------------------------------------------------
// a rejector chain from the caller (include/pe_b200.h : peb_rejector): "" if it is valid, else why not
static std::string chain_error(const peb_rejector* chain, size_t n_chain) {
  if (n_chain == 0) return "";
  if (!chain) return "null rejector chain with n_chain > 0";
  if (n_chain > PEB_MAX_REJECTORS)
    return "rejector chain of " + std::to_string(n_chain) + " entries (at most " + std::to_string(PEB_MAX_REJECTORS) + ")";
  for (size_t s = 0; s < n_chain; ++s) {
    const peb_rejector& r = chain[s];
    const std::string at = "rejector " + std::to_string(s) + ": ";
    if (r.kind != PEB_REJECTOR_DISTANCE && r.kind != PEB_REJECTOR_MEDIAN_DISTANCE && r.kind != PEB_REJECTOR_ONE_TO_ONE &&
        r.kind != PEB_REJECTOR_TRIMMED)
      return at + "unknown kind " + std::to_string(r.kind);
    if (!std::isfinite(r.value)) return at + "non-finite value";
    if (r.min_correspondences < 0) return at + "negative min_correspondences";
  }
  return "";
}

static int check_chain(peb_ctx* ctx, const char* what, const peb_rejector* chain, size_t n_chain) {
  const std::string e = chain_error(chain, n_chain);
  return e.empty() ? PEB_OK : fail(ctx, PEB_E_INVALID_ARG, "%s: %s", what, e.c_str());
}
static int icp_align_batch_dev_impl(peb_ctx* ctx, const float* d_guesses, size_t n_guesses, const peb_icp_params* params,
                                    peb_icp_result* d_results) {
  if (!ctx || !params) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  if (n_guesses > 0 && !d_results) return fail(ctx, PEB_E_INVALID_ARG, "align_batch_dev: null results");
  return icp_align_device(ctx, d_guesses, n_guesses, params, d_results, false);
}

static int icp_align_dev_impl(peb_ctx* ctx, const float guess[16], const peb_icp_params* params, peb_icp_result* d_result) {
  if (!ctx || !params || !d_result) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  const float* d_g = nullptr;
  PEB_TRY(upload_guesses(ctx, guess, 1, &d_g));
  return icp_align_device(ctx, d_g, 1, params, d_result, true);
}

static int icp_align_impl(peb_ctx* ctx, const float guess[16], const peb_icp_params* params, peb_icp_result* result,
                          float* out_aligned_xyz4, int32_t* out_corr_idx, float* out_corr_d2,
                          const peb_rejector* chain = nullptr, size_t n_chain = 0) {
  if (!ctx || !params || !result) return PEB_E_INVALID_ARG;
  PEB_TRY(check_chain(ctx, "peb_icp_align_ex", chain, n_chain));
  DeviceGuard guard(ctx->device);
  const float* d_g = nullptr;
  PEB_TRY(upload_guesses(ctx, guess, 1, &d_g));
  PEB_CUDA(ctx, ctx->d_results.ensure(sizeof(peb_icp_result)));
  PEB_TRY(icp_align_device(ctx, d_g, 1, params, ctx->d_results.as<peb_icp_result>(), true, chain, static_cast<int>(n_chain)));
  const size_t n = ctx->n_src;
  PEB_CUDA(ctx, cudaMemcpyAsync(result, ctx->d_results.p, sizeof(peb_icp_result), cudaMemcpyDeviceToHost, ctx->stream));
  if (out_aligned_xyz4 && n) {
    PEB_CUDA(ctx, ctx->d_aligned.ensure(n * sizeof(float4)));
    PEB_TRY(icp_output_device(ctx, ctx->d_aligned.as<float4>()));
    PEB_CUDA(ctx, cudaMemcpyAsync(out_aligned_xyz4, ctx->d_aligned.p, n * sizeof(float4), cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (out_corr_idx && n)
    PEB_CUDA(ctx, cudaMemcpyAsync(out_corr_idx, ctx->corr_idx.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  if (out_corr_d2 && n)
    PEB_CUDA(ctx, cudaMemcpyAsync(out_corr_d2, ctx->corr_d2.p, n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  PEB_TRY(sync(ctx));
  ctx->last_iterations = result->iterations;
  return PEB_OK;
}

static int icp_align_batch_impl(peb_ctx* ctx, const float* guesses, size_t n_guesses, const peb_icp_params* params,
                                peb_icp_result* results, const peb_rejector* chain = nullptr, size_t n_chain = 0) {
  if (!ctx || !params) return PEB_E_INVALID_ARG;
  PEB_TRY(check_chain(ctx, "peb_icp_align_batch_ex", chain, n_chain));
  DeviceGuard guard(ctx->device);
  if (n_guesses == 0) return PEB_OK;
  if (!guesses || !results) return fail(ctx, PEB_E_INVALID_ARG, "align_batch: null guesses / results");
  const float* d_g = nullptr;
  PEB_TRY(upload_guesses(ctx, guesses, n_guesses, &d_g));
  PEB_CUDA(ctx, ctx->d_results.ensure(n_guesses * sizeof(peb_icp_result)));
  PEB_TRY(icp_align_device(ctx, d_g, n_guesses, params, ctx->d_results.as<peb_icp_result>(), false, chain,
                           static_cast<int>(n_chain)));
  PEB_CUDA(ctx, cudaMemcpyAsync(results, ctx->d_results.p, n_guesses * sizeof(peb_icp_result), cudaMemcpyDeviceToHost,
                                ctx->stream));
  // the error flag of the dependency waits is read AFTER every launch of the align has finished: a record written
  // before another hypothesis hit its bound does not carry the error
  int* h_flag = ctx->h_small.as<int>() + 64;
  *h_flag = 0;
  if (ctx->last_err_flag)
    PEB_CUDA(ctx, cudaMemcpyAsync(h_flag, ctx->last_err_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  PEB_TRY(sync(ctx));
  if (*h_flag != 0 || results[0].state == PEB_STATE_INTERNAL_ERROR)
    return fail(ctx, PEB_E_CUDA, "align_batch: a per-hypothesis dependency wait ran into its bound (internal error; "
                                 "peb_ctx_set_int(ctx, \"flag_deps\", 0) restores whole-grid dependencies)");
  return PEB_OK;
}

PEB_API int peb_fitness_score(peb_ctx* ctx, const float T[16], double max_range, double* out_fitness, int32_t* out_n_inliers) {
  if (!ctx || !T || !out_fitness) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  const float* d_g = nullptr;
  PEB_TRY(upload_guesses(ctx, T, 1, &d_g));
  PEB_CUDA(ctx, ctx->d_results.ensure(sizeof(peb_icp_result)));
  PEB_TRY(fitness_device(ctx, d_g, max_range, ctx->d_results.as<peb_icp_result>()));
  peb_icp_result* h = ctx->h_small.as<peb_icp_result>() + 8;
  PEB_CUDA(ctx, cudaMemcpyAsync(h, ctx->d_results.p, sizeof(peb_icp_result), cudaMemcpyDeviceToHost, ctx->stream));
  PEB_TRY(sync(ctx));
  *out_fitness = h->fitness;
  if (out_n_inliers) *out_n_inliers = h->n_correspondences;
  return PEB_OK;
}

// ---- introspection ----------------------------------------------------------------------------------
PEB_API int peb_target_grid_info(peb_ctx* ctx, peb_grid_info* out) {
  if (!ctx || !out) return PEB_E_INVALID_ARG;
  if (!ctx->tgt_grid.valid) return fail(ctx, PEB_E_NO_TARGET, "grid_info: no target set");
  const GridView& v = ctx->tgt_grid.view;
  out->origin[0] = v.ox;
  out->origin[1] = v.oy;
  out->origin[2] = v.oz;
  out->cell = v.h;
  out->dims[0] = v.dx;
  out->dims[1] = v.dy;
  out->dims[2] = v.dz;
  out->n_points = v.n;
  out->n_cells = ctx->tgt_grid.n_cells;
  return PEB_OK;
}

PEB_API int peb_profile_read(peb_ctx* ctx, float* out_ms, size_t cap, size_t* out_n) {
  if (!ctx || !out_n) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  PEB_TRY(sync(ctx));
  size_t cnt = static_cast<size_t>(ctx->prof_launches);
  if (cnt > cap) cnt = cap;
  *out_n = cnt;
  if (ctx->prof_chain_ends > 0 && cnt == 1 && out_ms) {  // chains: the slowest chain's iteration launches
    float span = 0.0f;
    for (int c = 0; c < ctx->prof_chain_ends; ++c) {
      float ms = 0.0f;
      PEB_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->prof_events[0], ctx->prof_events[2 + c]));
      span = std::max(span, ms);
    }
    out_ms[0] = span;
    return PEB_OK;
  }
  for (size_t i = 0; i < cnt && out_ms; ++i)
    PEB_CUDA(ctx, cudaEventElapsedTime(&out_ms[i], ctx->prof_events[2 * i], ctx->prof_events[2 * i + 1]));
  return PEB_OK;
}

// development aid (not in the public header): copies the phase time stamps of the last align
extern "C" PEB_API int peb_debug_timers_read(peb_ctx* ctx, unsigned long long* out, size_t cap_launches, size_t* out_n) {
  if (!ctx || !out_n) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  size_t n = static_cast<size_t>(ctx->dbg_launches);
  if (n > cap_launches) n = cap_launches;
  *out_n = n;
  if (n) {
    PEB_CUDA(ctx, cudaMemcpyAsync(out, ctx->dbg.p, n * 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    PEB_TRY(sync(ctx));
  }
  return PEB_OK;
}

// development aids (not in the public header): the radix sort and the scan on host arrays, for tests/test_gpu_sort_scan.py
extern "C" PEB_API int peb_debug_sort_pairs(peb_ctx* ctx, uint32_t* keys, uint32_t* vals, size_t n, int key_bits) {
  if (!ctx || (n && (!keys || !vals)) || n > (1u << 30)) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  DevBuf b[4];
  int rc = PEB_OK;
  for (DevBuf& x : b)
    if (x.ensure(std::max<size_t>(n, 1) * 4) != cudaSuccess) rc = fail(ctx, PEB_E_OOM, "debug_sort_pairs: out of device memory");
  uint32_t *ko = nullptr, *vo = nullptr;
  if (rc == PEB_OK && n) {
    cudaMemcpyAsync(b[0].p, keys, n * 4, cudaMemcpyHostToDevice, ctx->stream);
    cudaMemcpyAsync(b[1].p, vals, n * 4, cudaMemcpyHostToDevice, ctx->stream);
    rc = sort_pairs(ctx, b[0].as<uint32_t>(), b[1].as<uint32_t>(), b[2].as<uint32_t>(), b[3].as<uint32_t>(), static_cast<int>(n),
                    key_bits, &ko, &vo);
    if (rc == PEB_OK) {
      cudaMemcpyAsync(keys, ko, n * 4, cudaMemcpyDeviceToHost, ctx->stream);
      cudaMemcpyAsync(vals, vo, n * 4, cudaMemcpyDeviceToHost, ctx->stream);
      rc = sync(ctx);
    }
  }
  for (DevBuf& x : b) x.release();
  return rc;
}

extern "C" PEB_API int peb_debug_exclusive_scan(peb_ctx* ctx, const uint32_t* in, uint32_t* out, size_t n, uint32_t* out_total) {
  if (!ctx || (n && (!in || !out)) || n > (1u << 30)) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  DevBuf b;
  if (b.ensure(std::max<size_t>(n, 1) * 4 + 4) != cudaSuccess) return fail(ctx, PEB_E_OOM, "debug_exclusive_scan: out of device memory");
  uint32_t* d = b.as<uint32_t>();
  if (n) cudaMemcpyAsync(d, in, n * 4, cudaMemcpyHostToDevice, ctx->stream);
  int rc = exclusive_scan_u32(ctx, d, d, static_cast<int>(n), d + n);  // in place
  if (rc == PEB_OK) {
    if (n) cudaMemcpyAsync(out, d, n * 4, cudaMemcpyDeviceToHost, ctx->stream);
    if (out_total) cudaMemcpyAsync(out_total, d + n, 4, cudaMemcpyDeviceToHost, ctx->stream);
    rc = sync(ctx);
  }
  b.release();
  return rc;
}


// development aid (not in the public header): block_select_nth over host values, one result per rank in nths, for
// tests/test_gpu_block_select.py.  Every rank must be below the number of values taken (all m, or with skip_neg the
// ones whose sign bit is clear); a rank outside is refused here, before any launch.
extern "C" PEB_API int peb_debug_select_nth(peb_ctx* ctx, const float* values, size_t m, const int32_t* nths, size_t n_nth, int skip_neg,
                                            float* out) {
  if (!ctx || !values || !nths || !out || m == 0 || m > (1u << 30) || n_nth == 0 || n_nth > 65535) return PEB_E_INVALID_ARG;
  size_t taken = m;
  if (skip_neg) {
    taken = 0;
    for (size_t i = 0; i < m; ++i) taken += !std::signbit(values[i]);
  }
  for (size_t k = 0; k < n_nth; ++k)
    if (nths[k] < 0 || static_cast<size_t>(nths[k]) >= taken)
      return fail(ctx, PEB_E_INVALID_ARG, "debug_select_nth: rank %d outside the %zu values taken", nths[k], taken);
  DeviceGuard guard(ctx->device);
  DevBuf b;
  const size_t o_nth = (m * 4 + 255) & ~static_cast<size_t>(255), o_out = o_nth + ((n_nth * 4 + 255) & ~static_cast<size_t>(255));
  if (b.ensure(o_out + n_nth * 4) != cudaSuccess) return fail(ctx, PEB_E_OOM, "debug_select_nth: out of device memory");
  char* base = b.as<char>();
  float* d_v = reinterpret_cast<float*>(base);
  int32_t* d_nth = reinterpret_cast<int32_t*>(base + o_nth);
  float* d_out = reinterpret_cast<float*>(base + o_out);
  const int rc = [&]() -> int {
    PEB_CUDA(ctx, cudaMemcpyAsync(d_v, values, m * 4, cudaMemcpyHostToDevice, ctx->stream));
    PEB_CUDA(ctx, cudaMemcpyAsync(d_nth, nths, n_nth * 4, cudaMemcpyHostToDevice, ctx->stream));
    if (skip_neg)
      PEB_LAUNCH(ctx, debug_select_nth_kernel<true>, static_cast<int>(n_nth), 1024, 0, d_v, static_cast<int>(m), d_nth, d_out);
    else
      PEB_LAUNCH(ctx, debug_select_nth_kernel<false>, static_cast<int>(n_nth), 1024, 0, d_v, static_cast<int>(m), d_nth, d_out);
    PEB_CUDA(ctx, cudaMemcpyAsync(out, d_out, n_nth * 4, cudaMemcpyDeviceToHost, ctx->stream));
    return sync(ctx);
  }();
  b.release();
  return rc;
}

PEB_API int peb_icp_trace(peb_ctx* ctx, float* out_T, size_t cap, size_t* out_n) {
  if (!ctx || !out_n) return PEB_E_INVALID_ARG;
  DeviceGuard guard(ctx->device);
  size_t cnt = static_cast<size_t>(ctx->last_iterations > 0 ? ctx->last_iterations : 0);
  if (cnt > static_cast<size_t>(ctx->last_trace_cap)) cnt = ctx->last_trace_cap;
  if (cnt > cap) cnt = cap;
  *out_n = cnt;
  if (cnt && out_T) {
    PEB_CUDA(ctx, cudaMemcpyAsync(out_T, ctx->trace.p, cnt * 16 * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    PEB_TRY(sync(ctx));
  }
  return PEB_OK;
}

// ---- entry points behind the exception barrier ------------------------------------------------------------
PEB_API int peb_sac_plane_dev(peb_ctx* ctx, const void* d_xyz4, size_t n, const peb_sac_params* params, float out_coeff[4], int32_t* d_out_inliers, size_t* out_n_inliers, int32_t* out_iterations) {
  return guarded(ctx, "peb_sac_plane_dev", [&]() { return sac_plane_dev_impl(ctx, d_xyz4, n, params, out_coeff, d_out_inliers, out_n_inliers, out_iterations); });
}

PEB_API int peb_sac_plane(peb_ctx* ctx, const void* pts, size_t n, size_t stride, const peb_sac_params* params, float out_coeff[4], int32_t* out_inliers, size_t* out_n_inliers, int32_t* out_iterations) {
  return guarded(ctx, "peb_sac_plane", [&]() { return sac_plane_impl(ctx, pts, n, stride, params, out_coeff, out_inliers, out_n_inliers, out_iterations); });
}

PEB_API int peb_scene_prepare(peb_ctx* ctx, const void* pts, size_t n, size_t stride, const peb_prefilter_params* filter, int num_planes, const peb_sac_params* sac, float leaf, float* out_xyz4, size_t* out_n, float* out_planes) {
  return guarded(ctx, "peb_scene_prepare", [&]() { return scene_prepare_impl(ctx, pts, n, stride, filter, num_planes, sac, leaf, out_xyz4, out_n, out_planes); });
}

PEB_API int peb_cvicp_register(peb_ctx* ctx, const float* model_xyzn, size_t n_model, const float* scene_xyzn, size_t n_scene, const peb_cvicp_params* params, double* poses, size_t n_poses, double* out_residuals) {
  return guarded(ctx, "peb_cvicp_register", [&]() { return cvicp_register_impl(ctx, model_xyzn, n_model, scene_xyzn, n_scene, params, poses, n_poses, out_residuals); });
}

PEB_API int peb_icp_align_batch_dev(peb_ctx* ctx, const float* d_guesses, size_t n_guesses, const peb_icp_params* params, peb_icp_result* d_results) {
  return guarded(ctx, "peb_icp_align_batch_dev", [&]() { return icp_align_batch_dev_impl(ctx, d_guesses, n_guesses, params, d_results); });
}

PEB_API int peb_icp_align_dev(peb_ctx* ctx, const float guess[16], const peb_icp_params* params, peb_icp_result* d_result) {
  return guarded(ctx, "peb_icp_align_dev", [&]() { return icp_align_dev_impl(ctx, guess, params, d_result); });
}

PEB_API int peb_icp_align(peb_ctx* ctx, const float guess[16], const peb_icp_params* params, peb_icp_result* result, float* out_aligned_xyz4, int32_t* out_corr_idx, float* out_corr_d2) {
  return guarded(ctx, "peb_icp_align", [&]() { return icp_align_impl(ctx, guess, params, result, out_aligned_xyz4, out_corr_idx, out_corr_d2); });
}

PEB_API int peb_icp_align_batch(peb_ctx* ctx, const float* guesses, size_t n_guesses, const peb_icp_params* params, peb_icp_result* results) {
  return guarded(ctx, "peb_icp_align_batch", [&]() { return icp_align_batch_impl(ctx, guesses, n_guesses, params, results); });
}

PEB_API int peb_icp_align_ex(peb_ctx* ctx, const float guess[16], const peb_icp_params* params, const peb_rejector* chain,
                             size_t n_chain, peb_icp_result* result, float* out_aligned_xyz4, int32_t* out_corr_idx,
                             float* out_corr_d2) {
  return guarded(ctx, "peb_icp_align_ex", [&]() {
    return icp_align_impl(ctx, guess, params, result, out_aligned_xyz4, out_corr_idx, out_corr_d2, chain, n_chain);
  });
}

PEB_API int peb_icp_align_batch_ex(peb_ctx* ctx, const float* guesses, size_t n_guesses, const peb_icp_params* params,
                                   const peb_rejector* chain, size_t n_chain, peb_icp_result* results) {
  return guarded(ctx, "peb_icp_align_batch_ex",
                 [&]() { return icp_align_batch_impl(ctx, guesses, n_guesses, params, results, chain, n_chain); });
}

// (here rather than in multi.cu, which is also compiled against fake single-device entry points that have no _ex)
PEB_API int peb_multi_icp_align_batch_ex(peb_multi* m, const float* guesses, size_t n_guesses, const peb_icp_params* params,
                                         const peb_rejector* chain, size_t n_chain, peb_icp_result* results) {
  if (!m || !params) return PEB_E_INVALID_ARG;
  if (n_guesses == 0) return PEB_OK;
  if (!guesses || !results) return multi_set_error(m, PEB_E_INVALID_ARG, "peb_multi_icp_align_batch_ex: null guesses / results");
  try {
    const std::string e = chain_error(chain, n_chain);
    if (!e.empty()) return multi_set_error(m, PEB_E_INVALID_ARG, ("peb_multi_icp_align_batch_ex: " + e).c_str());
  } catch (...) {
    return multi_set_error(m, PEB_E_OOM, "peb_multi_icp_align_batch_ex: out of host memory");
  }
  struct Job {
    const float* guesses;
    const peb_icp_params* params;
    const peb_rejector* chain;
    size_t n_chain;
    peb_icp_result* results;
  } job{guesses, params, chain, n_chain, results};
  return multi_run_sharded(m, "peb_multi_icp_align_batch_ex", n_guesses, [](peb_ctx* c, size_t lo, size_t hi, void* user) {
    const Job* j = static_cast<const Job*>(user);
    return peb_icp_align_batch_ex(c, j->guesses + 16 * lo, hi - lo, j->params, j->chain, j->n_chain, j->results + lo);
  }, &job);
}

}  // extern "C"
