// cv_normals_oracle.cpp — TEST INFRASTRUCTURE: the CPU oracle of cv::ppf_match_3d::computeNormalsPC3d (DESIGN.md §13).
//
// oracle/pcl_oracle.cpp is included unchanged for its exact kd-tree k-NN (KdTree, here with FLANN's leaf size 8 of
// indexPCFlann's KDTreeSingleIndexParams(8)); this file adds OpenCV's tail, restated from recollection of
// opencv_contrib/modules/surface_matching/src/ppf_helpers.cpp and opencv/modules/core/src/lapack.cpp (4.x):
// meanCovLocalPCInd, cv::eigen = JacobiImpl_<double> in upstream's general-n form, and flipNormalViewpoint.
// The eigen solver is pinned: tests/test_cv_normals.py compares it with the real cv2.eigen bit for bit.  The rest is
// checked against an independent numpy + cv2.flann_Index + cv2.eigen witness.  tests/cv_normals_oracle.py compiles it,
// with the oracle's parity flags, into a temporary directory.
#include "../oracle/pcl_oracle.cpp"

namespace orc {

namespace cvn {

// [CV] core/src/lapack.cpp : hypot<double>
static double hypot_cv(double a, double b) {
  a = std::fabs(a);
  b = std::fabs(b);
  if (a > b) {
    b /= a;
    return a * std::sqrt(1 + b * b);
  }
  if (b > 0) {
    a /= b;
    return b * std::sqrt(1 + a * a);
  }
  return 0;
}

// [CV] core/src/lapack.cpp : JacobiImpl_<double> as cv::eigen calls it without Eigen (A: n x n row-major, overwritten;
// W: eigenvalues descending; V: eigenvectors as rows), in upstream's general-n form
static void jacobi(double* A, int n, double* W, double* V) {
  const double eps = DBL_EPSILON;
  for (int i = 0; i < n; ++i) {
    for (int j = 0; j < n; ++j) V[i * n + j] = 0;
    V[i * n + i] = 1;
  }
  std::vector<int> indR(n), indC(n);
  auto row_max = [&](int k) {  // indR[k]: argmax over m > k of |A[k][m]|, first maximum wins
    int m = k + 1;
    double mv = std::fabs(A[k * n + m]);
    for (int i = k + 2; i < n; ++i)
      if (mv < std::fabs(A[k * n + i])) mv = std::fabs(A[k * n + i]), m = i;
    return m;
  };
  auto col_max = [&](int k) {  // indC[k]: argmax over m < k of |A[m][k]|
    int m = 0;
    double mv = std::fabs(A[k]);
    for (int i = 1; i < k; ++i)
      if (mv < std::fabs(A[i * n + k])) mv = std::fabs(A[i * n + k]), m = i;
    return m;
  };
  for (int k = 0; k < n; ++k) {
    W[k] = A[(n + 1) * k];
    if (k < n - 1) indR[k] = row_max(k);
    if (k > 0) indC[k] = col_max(k);
  }
  if (n > 1)
    for (int iters = 0; iters < n * n * 30; ++iters) {
      int k = 0;
      double mv = std::fabs(A[indR[0]]);
      for (int i = 1; i < n - 1; ++i)
        if (mv < std::fabs(A[i * n + indR[i]])) mv = std::fabs(A[i * n + indR[i]]), k = i;
      int l = indR[k];
      for (int i = 1; i < n; ++i)
        if (mv < std::fabs(A[indC[i] * n + i])) mv = std::fabs(A[indC[i] * n + i]), k = indC[i], l = i;
      const double p = A[k * n + l];
      if (std::fabs(p) <= eps) break;
      const double y = (W[l] - W[k]) * 0.5;
      double t = std::fabs(y) + hypot_cv(p, y);
      double s = hypot_cv(p, t);
      const double c = t / s;
      s = p / s;
      t = (p / t) * p;
      if (y < 0) s = -s, t = -t;
      A[k * n + l] = 0;
      W[k] -= t;
      W[l] += t;
      auto rot = [&](double& v0, double& v1) {
        const double a0 = v0, b0 = v1;
        v0 = a0 * c - b0 * s;
        v1 = a0 * s + b0 * c;
      };
      for (int i = 0; i < k; ++i) rot(A[i * n + k], A[i * n + l]);
      for (int i = k + 1; i < l; ++i) rot(A[k * n + i], A[i * n + l]);
      for (int i = l + 1; i < n; ++i) rot(A[k * n + i], A[l * n + i]);
      for (int i = 0; i < n; ++i) rot(V[k * n + i], V[l * n + i]);
      for (int j = 0; j < 2; ++j) {
        const int idx = j == 0 ? k : l;
        if (idx < n - 1) indR[idx] = row_max(idx);
        if (idx > 0) indC[idx] = col_max(idx);
      }
    }
  for (int k = 0; k < n - 1; ++k) {
    int m = k;
    for (int i = k + 1; i < n; ++i)
      if (W[m] < W[i]) m = i;
    if (k != m) {
      std::swap(W[m], W[k]);
      for (int i = 0; i < n; ++i) std::swap(V[m * n + i], V[k * n + i]);
    }
  }
}

// meanCovLocalPCInd over the neighbour list, cv::eigen, row 2 -> float, flipNormalViewpoint
static void normal_of(const void* pts, size_t stride, const int32_t* nn, int k, const float* p, bool flip, const float* vp,
                      float* n3) {
  double C[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, mu[3] = {0, 0, 0};
  for (int i = 0; i < k; ++i) {
    const float* c = reinterpret_cast<const float*>(static_cast<const char*>(pts) + static_cast<size_t>(nn[i]) * stride);
    for (int j = 0; j < 3; ++j) {
      for (int l = 0; l < 3; ++l) C[j * 3 + l] += c[j] * c[l];  // the product in float, the sum in double
      mu[j] += c[j];
    }
  }
  const double inv = 1.0 / k;
  for (int j = 0; j < 3; ++j) mu[j] *= inv;
  for (int j = 0; j < 9; ++j) C[j] *= inv;
  for (int j = 0; j < 3; ++j)
    for (int l = 0; l < 3; ++l) C[j * 3 + l] -= mu[j] * mu[l];
  double W[3], V[9];
  jacobi(C, 3, W, V);
  for (int j = 0; j < 3; ++j) n3[j] = static_cast<float>(V[6 + j]);
  if (flip) {
    const float d[3] = {vp[0] - p[0], vp[1] - p[1], vp[2] - p[2]};
    float cos_theta = 0;
    for (int j = 0; j < 3; ++j) cos_theta += d[j] * n3[j];
    if (cos_theta < 0)
      for (int j = 0; j < 3; ++j) n3[j] *= -1;
  }
}

}  // namespace cvn

}  // namespace orc

extern "C" {

// computeNormalsPC3d: out6 = n rows x y z nx ny nz; out_nn (nullable) n x k.  Returns 0, or -1 (PEB_E_INVALID_ARG)
// for k < 1 or k > the number of finite points (nothing written).  Non-finite points: x y z copied, NaN normal.
ORC_API int orc_cv_normals(const void* pts, size_t n, size_t stride, int k, int flip, const float* vp, float* out6,
                           int32_t* out_nn, int threads) {
  orc::KdTree tree;
  tree.leaf_max = 8;
  tree.build(pts, n, stride);
  if (k < 1 || (n > 0 && k > tree.n)) return -1;
  const float qnan = std::numeric_limits<float>::quiet_NaN();
#ifdef _OPENMP
  if (threads <= 0) threads = omp_get_max_threads();
#pragma omp parallel for num_threads(threads) schedule(dynamic, 1024)
#endif
  for (int64_t i = 0; i < static_cast<int64_t>(n); ++i) {
    std::vector<int32_t> nn(k, -1);
    std::vector<float> d2(k);
    const float* p = orc::rec(pts, static_cast<size_t>(i), stride);
    float* o = out6 + 6 * i;
    o[0] = p[0];
    o[1] = p[1];
    o[2] = p[2];
    if (orc::finite3(p[0], p[1], p[2])) {
      tree.knn(p, k, nn.data(), d2.data());
      orc::cvn::normal_of(pts, stride, nn.data(), k, p, flip != 0, vp, o + 3);
    } else {
      o[3] = o[4] = o[5] = qnan;
    }
    if (out_nn) std::memcpy(out_nn + i * k, nn.data(), k * sizeof(int32_t));
  }
  (void)threads;
  return 0;
}

// cv::eigen of m symmetric 3 x 3 matrices (row-major) through the general-n restatement above
ORC_API void orc_cv_eigen3(const double* A, size_t m, double* W, double* V) {
  for (size_t i = 0; i < m; ++i) {
    double a[9];
    std::memcpy(a, A + 9 * i, sizeof(a));
    orc::cvn::jacobi(a, 3, W + 3 * i, V + 9 * i);
  }
}
}
