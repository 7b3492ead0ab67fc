// gicp_host.cu — TEST SHIM, not product code.  The scalar GICP arithmetic of pose_estimation_b200/csrc/gicp_math.cuh
// (covariance tail, Mahalanobis inverse, applyState, cost and gradient, the BFGS of bfgs.h) compiled for the CPU, with the
// pair sums taken sequentially in pair order.  tests/gicp_reference.py builds it into a temporary directory.
#include <cstring>

#include "../../pose_estimation_b200/csrc/gicp_math.cuh"

using namespace peb;

namespace {

// the pairs of one BFGS run: p = output[i], t = its target point, M its Mahalanobis matrix
struct PairEval {
  const float* p;
  const float* t;
  const double* M;
  int m;
  int evals = 0;
  void fdf(const double* x, double& f, double* g) {
    ++evals;
    const Mat4 T = gicp_apply_state(x);
    double acc[kGicpAcc] = {0};
    for (int i = 0; i < m; ++i)
      gicp_pair_add(acc, T.m, p[3 * i], p[3 * i + 1], p[3 * i + 2], t[3 * i], t[3 * i + 1], t[3 * i + 2], M + 9 * i);
    gicp_fg_finish(acc, m, x, f, g);
  }
};

typedef void (*FdfFn)(const double* x, double* f, double* g);
struct FnEval {
  FdfFn fn;
  int evals = 0;
  void fdf(const double* x, double& f, double* g) {
    ++evals;
    fn(x, &f, g);
  }
};

}  // namespace

#define GH_API extern "C" __attribute__((visibility("default")))

GH_API void gh_fg(const float* p, const float* t, const double* M, int m, const double* x, double* f, double* g) {
  PairEval ev{p, t, M, m};
  ev.fdf(x, *f, g);
}

// returns the inner iterations; *evals: evaluations of f / g
GH_API int gh_bfgs(const float* p, const float* t, const double* M, int m, double* x, int max_inner, int* evals) {
  PairEval ev{p, t, M, m};
  const int inner = gicp_bfgs_minimize(ev, x, max_inner);
  if (evals) *evals = ev.evals;
  return inner;
}

GH_API int gh_bfgs_fn(FdfFn fn, double* x, int max_inner, int* evals) {
  FnEval ev{fn};
  const int inner = gicp_bfgs_minimize(ev, x, max_inner);
  if (evals) *evals = ev.evals;
  return inner;
}

// the covariance of k neighbours given in list order (k x 3 floats)
GH_API void gh_cov(const float* nb, int k, double* out9) {
  double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int i = 0; i < k; ++i) gicp_cov_add(acc, nb[3 * i], nb[3 * i + 1], nb[3 * i + 2]);
  double out[9];
  gicp_cov_finish(acc, k, out);
  memcpy(out9, out, sizeof(out));
}

GH_API void gh_rotation_d(const float* T, const float* G, double* R9) {
  double R[9];
  gicp_rotation_d(T, G, R);
  memcpy(R9, R, sizeof(R));
}

GH_API void gh_mahalanobis(const double* R9, const double* C1, const double* C2, double* M) {
  double R[9];
  memcpy(R, R9, sizeof(R));
  gicp_mahalanobis(R, C1, C2, M);
}

GH_API void gh_apply_state(const double* x, float* T16) {
  const Mat4 T = gicp_apply_state(x);
  memcpy(T16, T.m, sizeof(T.m));
}

GH_API void gh_state_of(const float* T16, double* x) { gicp_state_of(T16, x); }
