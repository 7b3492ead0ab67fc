// cv_normals_host.cu — TEST SHIM, not product code.  Compiles the __host__ __device__ tail of the
// computeNormalsPC3d path (core_math.cuh : cv_eigen_sym3, cv_moments_add, cv_normal_from_moments) for the
// CPU, so that tests/test_cv_normals.py can compare the solver with the real cv2.eigen without a GPU.
// Built into a temporary directory by that test; the product never loads this library.
#include <cstddef>

#include "../../pose_estimation_b200/csrc/core_math.cuh"

using namespace peb;

extern "C" {

// A: m row-major 3 x 3 doubles (upper triangle read) -> W: m x 3 eigenvalues, V: m x 9 eigenvectors as rows
__attribute__((visibility("default"))) void hc_cv_eigen_sym3(const double* A, size_t m, double* W, double* V) {
  for (size_t i = 0; i < m; ++i) {
    double a[9], w[3], v[9];
    for (int j = 0; j < 9; ++j) a[j] = A[9 * i + j];
    cv_eigen_sym3(a, w, v);
    for (int j = 0; j < 3; ++j) W[3 * i + j] = w[j];
    for (int j = 0; j < 9; ++j) V[9 * i + j] = v[j];
  }
}

// one normal from k neighbours (xyz rows of 3 floats, in list order) of the point p
__attribute__((visibility("default"))) void hc_cv_normal(const float* nb, int k, const float* p, int flip, const float* vp,
                                                         float* out3) {
  double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int i = 0; i < k; ++i) cv_moments_add(acc, nb[3 * i], nb[3 * i + 1], nb[3 * i + 2]);
  float n[3];
  cv_normal_from_moments(acc, k, p[0], p[1], p[2], flip != 0, vp[0], vp[1], vp[2], n);
  for (int j = 0; j < 3; ++j) out3[j] = n[j];
}
}
