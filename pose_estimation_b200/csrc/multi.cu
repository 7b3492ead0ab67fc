// multi.cu — several B200s behind one handle: the peb_multi_* entry points (include/pe_b200.h,
// SURVEY.md 8b layer 2 / 8e).  The reference node is ONE process (a component container with a
// single-threaded executor, launch/pose_estimation.launch.py:17-35), so a drop-in that wants all the
// GPUs of the box cannot rely on one process per GPU: this file gives that process one context per
// device, a replica of the scene grid and of the model on each, and shards the H initial poses of
// registerModelToScene(model, scene, poses) (opencv_surface_match.cpp:94) into contiguous blocks,
// one per device — the same rule as pose_estimation_b200/multi.py : shard_range.  Hypotheses are
// independent: no collective; every device copies its block of result records straight into the
// caller's `results` array.
//
// Host code only (no kernel of its own):
//   * one PERSISTENT host thread per extra device (created with the handle, parked on a condition variable between
//     calls) drives the blocking single-device entry points of api.cu, so every device runs the tested path unchanged
//     and a call costs two wake-ups instead of thread creation;
//   * the scene and the model cross PCIe ONCE: device 0 stages the caller's host buffer (peb_target_stage), every other
//     device copies the staged cloud device-to-device (peb_target_clone: NVLink / NVSwitch between peers) while
//     device 0 already builds its grid; every device then runs the same deterministic grid build on the same bytes,
//     so the replicas are identical.
#include <algorithm>
#include <condition_variable>
#include <exception>
#include <functional>
#include <mutex>
#include <thread>

#include "common.cuh"

namespace {

// One parked host thread per extra device.  post() hands it a job, wait() collects the job's status.
class Worker {
 public:
  Worker() : thread_([this]() { run(); }) {}
  ~Worker() {
    {
      std::lock_guard<std::mutex> lk(mu_);
      quit_ = true;
    }
    cv_.notify_all();
    if (thread_.joinable()) thread_.join();
  }
  Worker(const Worker&) = delete;
  Worker& operator=(const Worker&) = delete;

  void post(const std::function<int()>* job) {
    {
      std::lock_guard<std::mutex> lk(mu_);
      job_ = job;
      done_ = false;
    }
    cv_.notify_all();
  }
  int wait() {
    std::unique_lock<std::mutex> lk(mu_);
    cv_.wait(lk, [this]() { return done_; });
    return rc_;
  }

 private:
  void run() {
    for (;;) {
      const std::function<int()>* job = nullptr;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [this]() { return quit_ || job_ != nullptr; });
        if (quit_) return;
        job = job_;
        job_ = nullptr;
      }
      int rc = PEB_E_CUDA;
      try {
        rc = (*job)();
      } catch (const std::bad_alloc&) {
        rc = PEB_E_OOM;
      } catch (...) {
      }
      {
        std::lock_guard<std::mutex> lk(mu_);
        rc_ = rc;
        done_ = true;
      }
      cv_.notify_all();
    }
  }

  std::mutex mu_;
  std::condition_variable cv_;
  const std::function<int()>* job_ = nullptr;
  bool done_ = true;
  bool quit_ = false;
  int rc_ = PEB_OK;
  std::thread thread_;  // last: starts when everything above exists
};

}  // namespace

struct peb_multi {
  std::vector<peb_ctx*> ctx;
  std::vector<Worker*> workers;  // workers[i - 1] drives ctx[i]; ctx[0] runs on the calling thread
  std::string err;
};

namespace {

thread_local std::string g_multi_create_error;

int multi_fail(peb_multi* m, int code, const std::string& msg) {
  if (m) m->err = msg;
  return code;
}

// fn(i) on every context, device 0's on the calling thread; the first failing device (lowest index) is reported
template <typename Fn>
int on_all_devices(peb_multi* m, const char* what, Fn fn) {
  const size_t n = m->ctx.size();
  std::vector<int> rc(n, PEB_OK);
  try {
    std::vector<std::function<int()>> jobs;
    jobs.reserve(n);
    for (size_t i = 0; i < n; ++i) jobs.emplace_back([&fn, i]() { return fn(i); });
    for (size_t i = 1; i < n; ++i) m->workers[i - 1]->post(&jobs[i]);
    try {
      rc[0] = jobs[0]();
    } catch (...) {
      for (size_t i = 1; i < n; ++i) m->workers[i - 1]->wait();  // the jobs reference this frame
      throw;
    }
    for (size_t i = 1; i < n; ++i) rc[i] = m->workers[i - 1]->wait();
  } catch (const std::exception& e) {
    return multi_fail(m, PEB_E_OOM, std::string(what) + ": " + e.what());
  } catch (...) {
    return multi_fail(m, PEB_E_OOM, std::string(what) + ": host-side failure");
  }
  for (size_t i = 0; i < n; ++i)
    if (rc[i] != PEB_OK)
      return multi_fail(m, rc[i], std::string(what) + " [context " + std::to_string(i) + ", device " +
                                      std::to_string(m->ctx[i]->device) + "]: " + peb_last_error(m->ctx[i]));
  return PEB_OK;
}

}  // namespace

extern "C" {

PEB_API int peb_multi_create(int ndev, const int* devices, peb_multi** out) {
  if (!out) return PEB_E_INVALID_ARG;
  *out = nullptr;
  if (ndev < 1 || ndev > 64) {
    g_multi_create_error = "peb_multi_create: ndev must be in [1, 64]";
    return PEB_E_INVALID_ARG;
  }
  peb_multi* m = nullptr;
  try {
    m = new peb_multi();
    m->ctx.reserve(static_cast<size_t>(ndev));
    m->workers.reserve(static_cast<size_t>(ndev));
  } catch (...) {
    delete m;
    g_multi_create_error = "peb_multi_create: out of host memory";
    return PEB_E_OOM;
  }
  for (int i = 0; i < ndev; ++i) {
    peb_ctx* c = nullptr;
    const int dev = devices ? devices[i] : i;
    const int rc = peb_ctx_create(dev, &c);
    if (rc != PEB_OK) {
      g_multi_create_error = std::string("peb_multi_create [context ") + std::to_string(i) + ", device " + std::to_string(dev) +
                             "]: " + peb_last_error(nullptr);
      peb_multi_destroy(m);
      return rc;
    }
    m->ctx.push_back(c);
  }
  try {
    for (int i = 1; i < ndev; ++i) m->workers.push_back(new Worker());
  } catch (...) {
    g_multi_create_error = "peb_multi_create: could not start the per-device host threads";
    peb_multi_destroy(m);
    return PEB_E_OOM;
  }
  // replicas are copied device to device from context 0 (peb_multi_target_set): direct where the hardware allows it
  for (int i = 1; i < ndev; ++i) {
    peb_ctx_enable_peer(m->ctx[static_cast<size_t>(i)], m->ctx[0]);
    peb_ctx_enable_peer(m->ctx[0], m->ctx[static_cast<size_t>(i)]);
  }
  *out = m;
  return PEB_OK;
}

PEB_API void peb_multi_destroy(peb_multi* m) {
  if (!m) return;
  for (Worker* w : m->workers) delete w;  // joins the parked thread
  for (peb_ctx* c : m->ctx) peb_ctx_destroy(c);
  delete m;
}

PEB_API const char* peb_multi_last_error(const peb_multi* m) { return m ? m->err.c_str() : g_multi_create_error.c_str(); }
PEB_API int peb_multi_size(const peb_multi* m) { return m ? static_cast<int>(m->ctx.size()) : 0; }
PEB_API peb_ctx* peb_multi_ctx(peb_multi* m, int i) {
  return (m && i >= 0 && static_cast<size_t>(i) < m->ctx.size()) ? m->ctx[static_cast<size_t>(i)] : nullptr;
}

PEB_API int peb_multi_set_int(peb_multi* m, const char* key, int value) {
  if (!m || !key) return PEB_E_INVALID_ARG;
  for (size_t i = 0; i < m->ctx.size(); ++i) {
    const int rc = peb_ctx_set_int(m->ctx[i], key, value);
    if (rc != PEB_OK) return multi_fail(m, rc, peb_last_error(m->ctx[i]));
  }
  return PEB_OK;
}

PEB_API void peb_multi_shard_range(size_t n_items, int ndev, int i, size_t* lo, size_t* hi) {
  size_t a = 0, b = 0;
  if (ndev >= 1 && i >= 0 && i < ndev) {
    const size_t per = (n_items + static_cast<size_t>(ndev) - 1) / static_cast<size_t>(ndev);
    a = std::min(static_cast<size_t>(i) * per, n_items);
    b = std::min((static_cast<size_t>(i) + 1) * per, n_items);
  }
  if (lo) *lo = a;
  if (hi) *hi = b;
}

// One host-to-device copy (context 0), device-to-device replicas, the same grid build on every device.
PEB_API int peb_multi_target_set(peb_multi* m, const void* pts, size_t n, size_t stride, const void* normals, size_t nstride) {
  if (!m) return PEB_E_INVALID_ARG;
  const int rc = peb_target_stage(m->ctx[0], pts, n, stride, normals, nstride);
  if (rc != PEB_OK)
    return multi_fail(m, rc, std::string("peb_multi_target_set [context 0, device ") + std::to_string(m->ctx[0]->device) +
                                 "]: " + peb_last_error(m->ctx[0]));
  return on_all_devices(m, "peb_multi_target_set", [&](size_t i) {
    return i == 0 ? peb_target_build(m->ctx[0]) : peb_target_clone(m->ctx[i], m->ctx[0]);
  });
}

PEB_API int peb_multi_source_set(peb_multi* m, const void* pts, size_t n, size_t stride) {
  if (!m) return PEB_E_INVALID_ARG;
  const int rc = peb_source_stage(m->ctx[0], pts, n, stride);
  if (rc != PEB_OK)
    return multi_fail(m, rc, std::string("peb_multi_source_set [context 0, device ") + std::to_string(m->ctx[0]->device) +
                                 "]: " + peb_last_error(m->ctx[0]));
  return on_all_devices(m, "peb_multi_source_set", [&](size_t i) {
    return i == 0 ? peb_source_build(m->ctx[0]) : peb_source_clone(m->ctx[i], m->ctx[0]);
  });
}

PEB_API int peb_multi_icp_align_batch(peb_multi* m, const float* guesses, size_t n_guesses, const peb_icp_params* params,
                                      peb_icp_result* results) {
  if (!m || !params) return PEB_E_INVALID_ARG;
  if (n_guesses == 0) return PEB_OK;
  if (!guesses || !results) return multi_fail(m, PEB_E_INVALID_ARG, "peb_multi_icp_align_batch: null guesses / results");
  const int ndev = static_cast<int>(m->ctx.size());
  return on_all_devices(m, "peb_multi_icp_align_batch", [&](size_t i) {
    size_t lo = 0, hi = 0;
    peb_multi_shard_range(n_guesses, ndev, static_cast<int>(i), &lo, &hi);
    if (hi == lo) return static_cast<int>(PEB_OK);  // more devices than hypotheses
    return peb_icp_align_batch(m->ctx[i], guesses + 16 * lo, hi - lo, params, results + lo);
  });
}

}  // extern "C"

namespace peb {

int multi_run_sharded(peb_multi* m, const char* what, size_t n_items, int (*fn)(peb_ctx*, size_t lo, size_t hi, void* user),
                      void* user) {
  const int ndev = static_cast<int>(m->ctx.size());
  return on_all_devices(m, what, [&](size_t i) {
    size_t lo = 0, hi = 0;
    peb_multi_shard_range(n_items, ndev, static_cast<int>(i), &lo, &hi);
    if (hi == lo) return static_cast<int>(PEB_OK);  // more devices than items
    return fn(m->ctx[i], lo, hi, user);
  });
}

int multi_set_error(peb_multi* m, int code, const char* msg) { return multi_fail(m, code, msg); }

}  // namespace peb

extern "C" {

PEB_API uint64_t peb_multi_launch_count(const peb_multi* m) {
  uint64_t total = 0;
  if (m)
    for (const peb_ctx* c : m->ctx) total += peb_ctx_launch_count(c);
  return total;
}

}  // extern "C"
