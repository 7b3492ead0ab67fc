// gicp_math.cuh — the scalar arithmetic of pcl::GeneralizedIterativeClosestPoint (DESIGN.md §15), written
// __host__ __device__ so that tests/host compiles the same code for the CPU.  [PCL] registration/include/pcl/registration/
// gicp.h, impl/gicp.hpp, bfgs.h (PCL 1.10; restated from recollection, unpinned — no PCL, Eigen or GSL source exists here).
//
//   gicp_cov_*            computeCovariances: the moments of a point's k neighbours (float products added to doubles, in
//                         list order), the JacobiSVD of the covariance (core_math.cuh : svd3) and the reconstitution with
//                         singular values (1, 1, gicp_epsilon)
//   gicp_mahalanobis      (R C1 R^T + C2)^-1 with Eigen's 3 x 3 cofactor inverse, all double
//   gicp_apply_state      applyState: AngleAxisf(x5, Z) * AngleAxisf(x4, Y) * AngleAxisf(x3, X) as float quaternion
//                         products, toRotationMatrix, translation (float) x0..2
//   gicp_pair_add         one pair's share of f and of the gradient moments (13 doubles)
//   gicp_fg_finish        f / m, the gradient with computeRDerivative
//   GicpBfgs              bfgs.h: GSL's vector_bfgs2 with Fletcher's line search; the evaluator is a template argument
//                         (the device's is a collective reduction over a thread-block cluster, tests/host's a callback)
#pragma once

#include <limits>

#include "core_math.cuh"

namespace peb {

constexpr double kGicpEpsilon = 0.001;  // gicp_epsilon_
constexpr int kGicpAcc = 13;            // f, g[0..2], Racc[9] (row-major, Racc(r, c) = sum p_r temp_c)

// ---- computeCovariances ------------------------------------------------------------------------------------------
// acc: mean[3], then cov (0,0) (1,0) (1,1) (2,0) (2,1) (2,2) — the lower triangle, as PCL fills it
PEB_HD void gicp_cov_add(double (&acc)[9], float x, float y, float z) {
  acc[0] += x;
  acc[1] += y;
  acc[2] += z;
  acc[3] += x * x;  // (float products, widened when added)
  acc[4] += y * x;
  acc[5] += y * y;
  acc[6] += z * x;
  acc[7] += z * y;
  acc[8] += z * z;
}

// out: the reconstituted covariance, row-major
PEB_HD void gicp_cov_finish(const double (&acc)[9], int k, double (&out)[9]) {
  const double kd = static_cast<double>(k);
  double mean[3] = {acc[0] / kd, acc[1] / kd, acc[2] / kd};
  double cov[9];
  const int lower[6][2] = {{0, 0}, {1, 0}, {1, 1}, {2, 0}, {2, 1}, {2, 2}};
#pragma unroll
  for (int e = 0; e < 6; ++e) {
    const int r = lower[e][0], c = lower[e][1];
    double v = acc[3 + e] / kd;
    v = v - mean[r] * mean[c];
    cov[r * 3 + c] = v;
    cov[c * 3 + r] = v;
  }
  double U[9], sv[3], V[9];
  svd3(cov, U, sv, V);
#pragma unroll
  for (int i = 0; i < 9; ++i) out[i] = 0.0;
#pragma unroll
  for (int col = 0; col < 3; ++col) {
    const double v = col == 2 ? kGicpEpsilon : 1.0;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) out[r * 3 + c] = out[r * 3 + c] + (v * U[r * 3 + col]) * U[c * 3 + col];
  }
}

// ---- the per-iteration rotation and the Mahalanobis matrices ------------------------------------------------------
// R = top-left 3 x 3 of transformation_ * guess in double (k over all four columns, ascending); both column-major floats
PEB_HD void gicp_rotation_d(const float* T, const float* G, double (&R)[9]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      double a = 0.0;
#pragma unroll
      for (int k = 0; k < 4; ++k) a += static_cast<double>(T[k * 4 + i]) * static_cast<double>(G[j * 4 + k]);
      R[i * 3 + j] = a;
    }
}

PEB_HD void mat3d_mul(const double* A, const double* B, double* C) {
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) C[r * 3 + c] = (A[r * 3 + 0] * B[0 * 3 + c] + A[r * 3 + 1] * B[1 * 3 + c]) + A[r * 3 + 2] * B[2 * 3 + c];
}

// M = (R C1 R^T + C2)^-1, row-major: M = R * C1; temp = M * R^T; temp += C2; M = temp.inverse() (Eigen's cofactors)
PEB_HD void gicp_mahalanobis(const double (&R)[9], const double* C1, const double* C2, double* M) {
  double RC[9], Rt[9], t[9];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) Rt[r * 3 + c] = R[c * 3 + r];
  mat3d_mul(R, C1, RC);
  mat3d_mul(RC, Rt, t);
#pragma unroll
  for (int i = 0; i < 9; ++i) t[i] = t[i] + C2[i];
  auto cof = [&](int i, int j) {
    const int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (j + 1) % 3, j2 = (j + 2) % 3;
    return t[i1 * 3 + j1] * t[i2 * 3 + j2] - t[i1 * 3 + j2] * t[i2 * 3 + j1];
  };
  const double c00 = cof(0, 0), c10 = cof(1, 0), c20 = cof(2, 0);
  const double det = (c00 * t[0] + c10 * t[3]) + c20 * t[6];
  const double inv = 1.0 / det;
  // inverse(r, c) = cofactor(c, r) / det
  M[0] = c00 * inv;
  M[1] = c10 * inv;
  M[2] = c20 * inv;
  M[3] = cof(0, 1) * inv;
  M[4] = cof(1, 1) * inv;
  M[5] = cof(2, 1) * inv;
  M[6] = cof(0, 2) * inv;
  M[7] = cof(1, 2) * inv;
  M[8] = cof(2, 2) * inv;
}

// ---- the state vector ------------------------------------------------------------------------------------------
PEB_HD float gicp_cosf(float a) {
#ifdef __CUDA_ARCH__
  return cosf(a);
#else
  return std::cos(a);
#endif
}
PEB_HD float gicp_sinf(float a) {
#ifdef __CUDA_ARCH__
  return sinf(a);
#else
  return std::sin(a);
#endif
}

struct Quatf {
  float w, x, y, z;
};

// [EIGEN] Quaternion product (generic path)
PEB_HD Quatf quatf_mul(const Quatf& a, const Quatf& b) {
  Quatf r;
  r.w = ((a.w * b.w - a.x * b.x) - a.y * b.y) - a.z * b.z;
  r.x = ((a.w * b.x + a.x * b.w) + a.y * b.z) - a.z * b.y;
  r.y = ((a.w * b.y + a.y * b.w) + a.z * b.x) - a.x * b.z;
  r.z = ((a.w * b.z + a.z * b.w) + a.x * b.y) - a.y * b.x;
  return r;
}

// T (column-major) = identity with applyState(T, x): R = (AngleAxisf(x5, Z) * AngleAxisf(x4, Y)) * AngleAxisf(x3, X),
// t = (float) x0..2.  R * I is written out like Eigen's product so that signed zeros come out the same.
PEB_HD Mat4 gicp_apply_state(const double* x) {
  const float hx = 0.5f * static_cast<float>(x[3]), hy = 0.5f * static_cast<float>(x[4]), hz = 0.5f * static_cast<float>(x[5]);
  const Quatf qz{gicp_cosf(hz), 0.0f * gicp_sinf(hz), 0.0f * gicp_sinf(hz), 1.0f * gicp_sinf(hz)};
  const Quatf qy{gicp_cosf(hy), 0.0f * gicp_sinf(hy), 1.0f * gicp_sinf(hy), 0.0f * gicp_sinf(hy)};
  const Quatf qx{gicp_cosf(hx), 1.0f * gicp_sinf(hx), 0.0f * gicp_sinf(hx), 0.0f * gicp_sinf(hx)};
  const Quatf q = quatf_mul(quatf_mul(qz, qy), qx);
  // [EIGEN] QuaternionBase::toRotationMatrix
  const float tx = 2.0f * q.x, ty = 2.0f * q.y, tz = 2.0f * q.z;
  const float twx = tx * q.w, twy = ty * q.w, twz = tz * q.w;
  const float txx = tx * q.x, txy = ty * q.x, txz = tz * q.x;
  const float tyy = ty * q.y, tyz = tz * q.y, tzz = tz * q.z;
  float R[9];  // row-major
  R[0] = 1.0f - (tyy + tzz);
  R[1] = txy - twz;
  R[2] = txz + twy;
  R[3] = txy + twz;
  R[4] = 1.0f - (txx + tzz);
  R[5] = tyz - twx;
  R[6] = txz - twy;
  R[7] = tyz + twx;
  R[8] = 1.0f - (txx + tyy);
  Mat4 T = mat4_identity();
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float I0 = c == 0 ? 1.0f : 0.0f, I1 = c == 1 ? 1.0f : 0.0f, I2 = c == 2 ? 1.0f : 0.0f;
      T.m[c * 4 + r] = (R[r * 3 + 0] * I0 + R[r * 3 + 1] * I1) + R[r * 3 + 2] * I2;
    }
  T.m[12] = 0.0f + static_cast<float>(x[0]);
  T.m[13] = 0.0f + static_cast<float>(x[1]);
  T.m[14] = 0.0f + static_cast<float>(x[2]);
  return T;
}

PEB_HD float gicp_atan2f(float y, float x) {
#ifdef __CUDA_ARCH__
  return atan2f(y, x);
#else
  return std::atan2(y, x);
#endif
}
PEB_HD float gicp_asinf(float v) {
#ifdef __CUDA_ARCH__
  return asinf(v);
#else
  return std::asin(v);
#endif
}

// x0 of estimateRigidTransformationBFGS from the float transformation_ (float atan2 / asin)
PEB_HD void gicp_state_of(const float* T, double* x) {
  x[0] = T[12];
  x[1] = T[13];
  x[2] = T[14];
  x[3] = gicp_atan2f(T[1 * 4 + 2], T[2 * 4 + 2]);
  x[4] = gicp_asinf(-T[0 * 4 + 2]);
  x[5] = gicp_atan2f(T[0 * 4 + 1], T[0 * 4 + 0]);
}

// ---- the cost and its gradient -------------------------------------------------------------------------------------
// One pair: p = output[i] (float), tq = its target point, M its Mahalanobis matrix (row-major), T = T(x)
PEB_HD void gicp_pair_add(double (&acc)[kGicpAcc], const float* T, float px, float py, float pz, float tx, float ty, float tz,
                          const double* M) {
  float ppx, ppy, ppz;
  transform_icp(T, px, py, pz, ppx, ppy, ppz);
  const double r0 = ppx - tx, r1 = ppy - ty, r2 = ppz - tz;
  const double t0 = (M[0] * r0 + M[1] * r1) + M[2] * r2;
  const double t1 = (M[3] * r0 + M[4] * r1) + M[5] * r2;
  const double t2 = (M[6] * r0 + M[7] * r1) + M[8] * r2;
  acc[0] += (r0 * t0 + r1 * t1) + r2 * t2;
  acc[1] += t0;
  acc[2] += t1;
  acc[3] += t2;
  const double p[3] = {px, py, pz}, t[3] = {t0, t1, t2};
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int c = 0; c < 3; ++c) acc[4 + r * 3 + c] += p[r] * t[c];
}

PEB_HD double gicp_cos(double a) {
#ifdef __CUDA_ARCH__
  return ::cos(a);
#else
  return std::cos(a);
#endif
}
PEB_HD double gicp_sin(double a) {
#ifdef __CUDA_ARCH__
  return ::sin(a);
#else
  return std::sin(a);
#endif
}

// matricesInnerProd(A, B) = sum_i sum_j A(j, i) B(i, j), both row-major here
PEB_HD double gicp_inner(const double (&A)[9], const double (&B)[9]) {
  double r = 0.0;
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) r += A[j * 3 + i] * B[i * 3 + j];
  return r;
}

// sums over the m pairs -> f and g (fdf: f / m, g[0..2] * (2 / m), Racc * (2 / m), computeRDerivative)
PEB_HD void gicp_fg_finish(const double (&acc)[kGicpAcc], int m, const double* x, double& f, double* g) {
  const double md = static_cast<double>(m);
  const double s = 2.0 / md;
  f = acc[0] / md;
  g[0] = acc[1] * s;
  g[1] = acc[2] * s;
  g[2] = acc[3] * s;
  double R[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) R[i] = acc[4 + i] * s;
  const double cphi = gicp_cos(x[3]), sphi = gicp_sin(x[3]);
  const double ctheta = gicp_cos(x[4]), stheta = gicp_sin(x[4]);
  const double cpsi = gicp_cos(x[5]), spsi = gicp_sin(x[5]);
  const double dphi[9] = {0.,
                          sphi * spsi + cphi * cpsi * stheta,
                          cphi * spsi - cpsi * sphi * stheta,
                          0.,
                          -cpsi * sphi + cphi * spsi * stheta,
                          -cphi * cpsi - sphi * spsi * stheta,
                          0.,
                          cphi * ctheta,
                          -ctheta * sphi};
  const double dtheta[9] = {-cpsi * stheta,         cpsi * ctheta * sphi, cphi * cpsi * ctheta,
                            -spsi * stheta,         ctheta * sphi * spsi, cphi * ctheta * spsi,
                            -ctheta,                -sphi * stheta,       -cphi * stheta};
  const double dpsi[9] = {-ctheta * spsi, -cphi * cpsi - sphi * spsi * stheta, cpsi * sphi - cphi * spsi * stheta,
                          cpsi * ctheta,  -cphi * spsi + cpsi * sphi * stheta, sphi * spsi + cphi * cpsi * stheta,
                          0.,             0.,                                  0.};
  g[3] = gicp_inner(dphi, R);
  g[4] = gicp_inner(dtheta, R);
  g[5] = gicp_inner(dpsi, R);
}

// ---- bfgs.h -------------------------------------------------------------------------------------------------------
// BFGSSpace::Status
enum GicpBfgsStatus { kBfgsNegativeGradientEpsilon = -3, kBfgsNotStarted = -2, kBfgsRunning = -1, kBfgsSuccess = 0, kBfgsNoProgress = 1 };

PEB_HD double v6_dot(const double* a, const double* b) {
  double r = a[0] * b[0];
#pragma unroll
  for (int i = 1; i < 6; ++i) r += a[i] * b[i];
  return r;
}
PEB_HD double v6_norm(const double* a) { return sqrt(v6_dot(a, a)); }
PEB_HD bool isfinite_d(double v) { return v - v == 0.0; }
PEB_HD double qnan_d() {
#ifdef __CUDA_ARCH__
  return __longlong_as_double(0x7ff8000000000000ll);
#else
  return std::numeric_limits<double>::quiet_NaN();
#endif
}

// gsl_poly_solve_quadratic: the closed form PCL's PolynomialSolver call stands in for (a documented difference in the last bits)
PEB_HD int gicp_solve_quadratic(double a, double b, double c, double& x0, double& x1) {
  if (a == 0.0) {
    if (b == 0.0) return 0;
    x0 = -c / b;
    return 1;
  }
  const double disc = b * b - 4.0 * a * c;
  if (disc > 0.0) {
    if (b == 0.0) {
      const double r = sqrt(-c / a);
      x0 = -r;
      x1 = r;
    } else {
      const double sgnb = b > 0.0 ? 1.0 : -1.0;
      const double temp = -0.5 * (b + sgnb * sqrt(disc));
      const double r1 = temp / a, r2 = c / temp;
      if (r1 < r2) {
        x0 = r1;
        x1 = r2;
      } else {
        x0 = r2;
        x1 = r1;
      }
    }
    return 2;
  }
  if (disc == 0.0) {
    x0 = -0.5 * b / a;
    x1 = -0.5 * b / a;
    return 2;
  }
  return 0;
}

PEB_HD double bfgs_cubic(double c0, double c1, double c2, double c3, double z) { return c0 + z * (c1 + z * (c2 + z * c3)); }

PEB_HD void bfgs_check_extremum(double c0, double c1, double c2, double c3, double z, double& zmin, double& fmin) {
  const double y = bfgs_cubic(c0, c1, c2, c3, z);
  if (y < fmin) {
    zmin = z;
    fmin = y;
  }
}

PEB_HD double bfgs_cubicmin(double f0, double fp0, double f1, double fp1, double zl, double zh) {
  const double eta = 3.0 * (f1 - f0) - 2.0 * fp0 - fp1;
  const double xi = fp0 + fp1 - 2.0 * (f1 - f0);
  const double c0 = f0, c1 = fp0, c2 = eta, c3 = xi;
  double zmin = zl, fmin = bfgs_cubic(c0, c1, c2, c3, zl);
  bfgs_check_extremum(c0, c1, c2, c3, zh, zmin, fmin);
  double z0 = 0.0, z1 = 0.0;
  const int n = gicp_solve_quadratic(3.0 * c3, 2.0 * c2, c1, z0, z1);
  if (n == 2) {
    if (z0 > zl && z0 < zh) bfgs_check_extremum(c0, c1, c2, c3, z0, zmin, fmin);
    if (z1 > zl && z1 < zh) bfgs_check_extremum(c0, c1, c2, c3, z1, zmin, fmin);
  } else if (n == 1) {
    if (z0 > zl && z0 < zh) bfgs_check_extremum(c0, c1, c2, c3, z0, zmin, fmin);
  }
  return zmin;
}

PEB_HD double bfgs_interp_quad(double f0, double fp0, double f1, double zl, double zh) {
  const double fl = f0 + zl * (fp0 + zl * (f1 - f0 - fp0));
  const double fh = f0 + zh * (fp0 + zh * (f1 - f0 - fp0));
  const double c = 2.0 * (f1 - f0 - fp0);
  double zmin = zl, fmin = fl;
  if (fh < fmin) {
    zmin = zh;
    fmin = fh;
  }
  if (c > 0.0) {
    const double z = -fp0 / c;
    if (z > zl && z < zh) {
      const double f = f0 + z * (fp0 + z * (f1 - f0 - fp0));
      if (f < fmin) zmin = z;
    }
  }
  return zmin;
}

// order 3: cubic when fpb is known, quadratic otherwise
PEB_HD double bfgs_interpolate(double a, double fa, double fpa, double b, double fb, double fpb, double xmin, double xmax) {
  double zmin = (xmin - a) / (b - a), zmax = (xmax - a) / (b - a);
  if (zmin > zmax) {
    const double t = zmin;
    zmin = zmax;
    zmax = t;
  }
  double z;
  if (isfinite_d(fpb))  // GSL_IS_REAL
    z = bfgs_cubicmin(fa, fpa * (b - a), fb, fpb * (b - a), zmin, zmax);
  else
    z = bfgs_interp_quad(fa, fpa * (b - a), fb, zmin, zmax);
  return a + z * (b - a);
}

// The minimiser.  Eval: a functor with fdf(const double x[6], double& f, double g[6]); every f / df / fdf of bfgs.h is
// served by it (PCL's three functor calls compute the same sums in the same order, so one evaluation answers all three;
// the caches below decide, as in bfgs.h, which alphas are evaluated at all).
template <typename Eval>
struct GicpBfgs {
  Eval& ev;
  double x0[6], g0[6], p[6], dx[6];
  double x_alpha[6], g_alpha[6];
  double f, gradient[6];
  double f_alpha, df_alpha;
  double x_cache_key, f_cache_key, df_cache_key, g_cache_key;
  double g0norm, pnorm, fp0, delta_f;
  // parameters (estimateRigidTransformationBFGS)
  static constexpr double kRho = 0.01, kSigma = 0.01, kTau1 = 9.0, kTau2 = 0.05, kTau3 = 0.5, kStep = 1.0;
  static constexpr int kBracketIters = 100, kSectionIters = 100;

  PEB_HD explicit GicpBfgs(Eval& e) : ev(e) {}

  PEB_HD double slope() const { return v6_dot(g_alpha, p); }
  PEB_HD void move_to(double alpha) {
    if (alpha == x_cache_key) return;
#pragma unroll
    for (int i = 0; i < 6; ++i) x_alpha[i] = x0[i] + alpha * p[i];
    x_cache_key = alpha;
  }
  PEB_HD double apply_f(double alpha) {
    if (alpha == f_cache_key) return f_alpha;
    move_to(alpha);
    double g[6];
    ev.fdf(x_alpha, f_alpha, g);
    f_cache_key = alpha;
    return f_alpha;
  }
  PEB_HD double apply_df(double alpha) {
    if (alpha == df_cache_key) return df_alpha;
    move_to(alpha);
    if (alpha != g_cache_key) {
      double fx;
      ev.fdf(x_alpha, fx, g_alpha);
      g_cache_key = alpha;
    }
    df_alpha = slope();
    df_cache_key = alpha;
    return df_alpha;
  }
  PEB_HD void apply_fdf(double alpha, double& fo, double& dfo) {
    if (alpha == f_cache_key && alpha == df_cache_key) {
      fo = f_alpha;
      dfo = df_alpha;
      return;
    }
    if (alpha == f_cache_key || alpha == df_cache_key) {
      fo = apply_f(alpha);
      dfo = apply_df(alpha);
      return;
    }
    move_to(alpha);
    ev.fdf(x_alpha, f_alpha, g_alpha);
    f_cache_key = alpha;
    g_cache_key = alpha;
    df_alpha = slope();
    df_cache_key = alpha;
    fo = f_alpha;
    dfo = df_alpha;
  }
  PEB_HD void change_direction() {
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      x_alpha[i] = x0[i];
      g_alpha[i] = g0[i];
    }
    x_cache_key = 0.0;
    f_cache_key = 0.0;
    g_cache_key = 0.0;
    df_alpha = slope();
    df_cache_key = 0.0;
  }

  PEB_HD int minimize_init(const double* x) {
    delta_f = 0.0;
#pragma unroll
    for (int i = 0; i < 6; ++i) dx[i] = 0.0;
    ev.fdf(x, f, gradient);
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      x0[i] = x[i];
      g0[i] = gradient[i];
    }
    g0norm = v6_norm(g0);
#pragma unroll
    for (int i = 0; i < 6; ++i) p[i] = gradient[i] * -1.0 / g0norm;
    pnorm = v6_norm(p);
    fp0 = -g0norm;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      x_alpha[i] = x0[i];
      g_alpha[i] = g0[i];
    }
    x_cache_key = 0.0;
    f_alpha = f;
    f_cache_key = 0.0;
    g_cache_key = 0.0;
    df_alpha = slope();
    df_cache_key = 0.0;
    return kBfgsNotStarted;
  }

  // linear_minimize (Fletcher); one step counter for bracketing and sectioning, as in GSL
  PEB_HD int line_search(double alpha1, double& alpha_new) {
    double falpha, fpalpha, delta, alpha_next;
    double alpha = alpha1, alpha_prev = 0.0;
    int i = 0;
    const double f0 = apply_f(0.0);
    const double fp0l = apply_df(0.0);
    double falpha_prev = f0, fpalpha_prev = fp0l;
    double a = 0.0, b = alpha, fa = f0, fb = 0.0, fpa = fp0l, fpb = 0.0;
    while (i++ < kBracketIters) {
      falpha = apply_f(alpha);
      if (falpha > f0 + alpha * kRho * fp0l || falpha >= falpha_prev) {
        a = alpha_prev;
        fa = falpha_prev;
        fpa = fpalpha_prev;
        b = alpha;
        fb = falpha;
        fpb = qnan_d();
        break;
      }
      fpalpha = apply_df(alpha);
      if (fabs(fpalpha) <= -kSigma * fp0l) {
        alpha_new = alpha;
        return kBfgsSuccess;
      }
      if (fpalpha >= 0.0) {
        a = alpha;
        fa = falpha;
        fpa = fpalpha;
        b = alpha_prev;
        fb = falpha_prev;
        fpb = fpalpha_prev;
        break;
      }
      delta = alpha - alpha_prev;
      {
        const double lower = alpha + delta, upper = alpha + kTau1 * delta;
        alpha_next = bfgs_interpolate(alpha_prev, falpha_prev, fpalpha_prev, alpha, falpha, fpalpha, lower, upper);
      }
      alpha_prev = alpha;
      falpha_prev = falpha;
      fpalpha_prev = fpalpha;
      alpha = alpha_next;
    }
    while (i++ < kSectionIters) {
      delta = b - a;
      {
        const double lower = a + kTau2 * delta, upper = b - kTau3 * delta;
        alpha = bfgs_interpolate(a, fa, fpa, b, fb, fpb, lower, upper);
      }
      falpha = apply_f(alpha);
      if ((a - alpha) * fpa <= DBL_EPSILON) return kBfgsNoProgress;  // round-off prevents progress
      if (falpha > f0 + kRho * alpha * fp0l || falpha >= fa) {
        b = alpha;
        fb = falpha;
        fpb = qnan_d();
      } else {
        fpalpha = apply_df(alpha);
        if (fabs(fpalpha) <= -kSigma * fp0l) {
          alpha_new = alpha;
          return kBfgsSuccess;
        }
        if (((b - a) >= 0.0 && fpalpha >= 0.0) || ((b - a) <= 0.0 && fpalpha <= 0.0)) {
          b = a;
          fb = fa;
          fpb = fpa;
          a = alpha;
          fa = falpha;
          fpa = fpalpha;
        } else {
          a = alpha;
          fa = falpha;
          fpa = fpalpha;
        }
      }
    }
    return kBfgsSuccess;
  }

  PEB_HD int minimize_one_step(double* x) {
    double alpha = 0.0, alpha1;
    const double f0 = f;
    if (pnorm == 0.0 || g0norm == 0.0 || fp0 == 0.0) {
#pragma unroll
      for (int i = 0; i < 6; ++i) dx[i] = 0.0;
      return kBfgsNoProgress;
    }
    if (delta_f < 0.0) {
      const double del = fmax(-delta_f, 10.0 * DBL_EPSILON * fabs(f0));
      alpha1 = fmin(1.0, 2.0 * del / (-fp0));
    } else {
      alpha1 = fabs(kStep);
    }
    const int status = line_search(alpha1, alpha);
    if (status != kBfgsSuccess) return status;
    {  // updatePosition
      double fa, dfa;
      apply_fdf(alpha, fa, dfa);
      f = f_alpha;
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        x[i] = x_alpha[i];
        gradient[i] = g_alpha[i];
      }
    }
    delta_f = f - f0;
    {  // p' = g1 - A dx - B dg
      double dx0[6], dg0[6];
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        dx0[i] = x[i] - x0[i];
        dx[i] = dx0[i];
        dg0[i] = gradient[i] - g0[i];
      }
      const double dxg = v6_dot(dx0, gradient), dgg = v6_dot(dg0, gradient), dxdg = v6_dot(dx0, dg0);
      const double dgnorm = v6_norm(dg0);
      double A, B;
      if (dxdg != 0.0) {
        B = dxg / dxdg;
        A = -(1.0 + dgnorm * dgnorm / dxdg) * B + dgg / dxdg;
      } else {
        B = 0.0;
        A = 0.0;
      }
#pragma unroll
      for (int i = 0; i < 6; ++i) p[i] = (gradient[i] - A * dx0[i]) - B * dg0[i];  // Eigen: gradient - A * dx0 - B * dg0
    }
#pragma unroll
    for (int i = 0; i < 6; ++i) {
      g0[i] = gradient[i];
      x0[i] = x[i];
    }
    g0norm = v6_norm(g0);
    pnorm = v6_norm(p);
    const double dir = v6_dot(p, gradient) >= 0.0 ? -1.0 : 1.0;  // (GSL: pg >= 0)
#pragma unroll
    for (int i = 0; i < 6; ++i) p[i] = p[i] * (dir / pnorm);
    pnorm = v6_norm(p);
    fp0 = v6_dot(p, g0);
    change_direction();
    return kBfgsSuccess;
  }

  PEB_HD int test_gradient(double eps) const {
    if (eps < 0.0) return kBfgsNegativeGradientEpsilon;
    return v6_norm(gradient) < eps ? kBfgsSuccess : kBfgsRunning;
  }
};

// estimateRigidTransformationBFGS's driver: x in / out; returns the inner iterations run
template <typename Eval>
PEB_HD int gicp_bfgs_minimize(Eval& ev, double* x, int max_inner) {
  GicpBfgs<Eval> bfgs(ev);
  bfgs.minimize_init(x);
  int inner = 0, result;
  do {
    ++inner;
    result = bfgs.minimize_one_step(x);
    if (result) break;
    result = bfgs.test_gradient(1e-2);
  } while (result == kBfgsRunning && inner < max_inner);
  return inner;
}

}  // namespace peb
