// gicp_oracle.cpp — CPU ORACLE of pcl::GeneralizedIterativeClosestPoint<PointXYZ, PointXYZ>.  TEST INFRASTRUCTURE ONLY.
//
// oracle/pcl_oracle.cpp is included unchanged for its kd-tree (exact nearestKSearch), Eigen's JacobiSVD and the float
// transforms.  On top of it this file restates, sequentially and independently of the library's gicp_math.cuh:
//   [PCL] registration/impl/gicp.hpp : computeCovariances, computeTransformation, estimateRigidTransformationBFGS,
//                                      OptimizationFunctorWithIndices (operator(), df, fdf), applyState, computeRDerivative
//   [PCL] registration/bfgs.h        : BFGS<FunctorType> — minimizeInit, minimizeOneStep, lineSearch (GSL's Fletcher line
//                                      search), interpolate, cubicmin, interp_quad, the alpha caches, testGradient
// (PCL 1.10, restated from recollection; no PCL, Eigen or GSL source exists here).  Double sums run in index order.  The
// quadratic of cubicmin is solved with gsl_poly_solve_quadratic's closed form where PCL calls Eigen's PolynomialSolver.
#include "../oracle/pcl_oracle.cpp"

#include <array>

namespace orc_gicp {

using V6 = std::array<double, 6>;
using M3 = std::array<double, 9>;  // row-major

static double dot(const V6& a, const V6& b) {
  double r = a[0] * b[0];
  for (int i = 1; i < 6; ++i) r += a[i] * b[i];
  return r;
}
static double norm(const V6& a) { return std::sqrt(dot(a, a)); }

// ---- computeCovariances ---------------------------------------------------------------------------------------------
static void covariance(const float* nb /*k x 3*/, int k, double* out9) {
  double mean[3] = {0, 0, 0};
  double cov[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  for (int j = 0; j < k; ++j) {
    const float x = nb[3 * j], y = nb[3 * j + 1], z = nb[3 * j + 2];
    mean[0] += x;
    mean[1] += y;
    mean[2] += z;
    cov[0] += x * x;      // cov(0,0) += pt.x * pt.x  (float product)
    cov[3] += y * x;      // cov(1,0)
    cov[4] += y * y;      // cov(1,1)
    cov[6] += z * x;      // cov(2,0)
    cov[7] += z * y;      // cov(2,1)
    cov[8] += z * z;      // cov(2,2)
  }
  for (int a = 0; a < 3; ++a) mean[a] /= static_cast<double>(k);
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c <= r; ++c) {
      cov[r * 3 + c] /= static_cast<double>(k);
      cov[r * 3 + c] -= mean[r] * mean[c];
      cov[c * 3 + r] = cov[r * 3 + c];
    }
  double U[9], S[3], V[9];
  orc::jacobi_svd3<double>(cov, U, S, V);
  for (int i = 0; i < 9; ++i) out9[i] = 0.0;
  for (int col = 0; col < 3; ++col) {
    const double v = col == 2 ? 0.001 : 1.0;  // gicp_epsilon_
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 3; ++c) out9[r * 3 + c] += (v * U[r * 3 + col]) * U[c * 3 + col];
  }
}

// ---- applyState ------------------------------------------------------------------------------------------------------
struct Qf {
  float w, x, y, z;
};
static Qf qmul(const Qf& a, const Qf& b) {  // Eigen's generic quaternion product
  return Qf{a.w * b.w - a.x * b.x - a.y * b.y - a.z * b.z, a.w * b.x + a.x * b.w + a.y * b.z - a.z * b.y,
            a.w * b.y + a.y * b.w + a.z * b.x - a.x * b.z, a.w * b.z + a.z * b.w + a.x * b.y - a.y * b.x};
}
static Qf angle_axis(float angle, int axis) {  // AngleAxisf -> Quaternionf: w = cos(a / 2), vec = sin(a / 2) * axis
  const float ha = 0.5f * angle;
  const float c = std::cos(ha), s = std::sin(ha);
  return Qf{c, s * (axis == 0 ? 1.0f : 0.0f), s * (axis == 1 ? 1.0f : 0.0f), s * (axis == 2 ? 1.0f : 0.0f)};
}
// t = I; applyState(t, x)
static orc::M4 apply_state(const V6& x) {
  const Qf q = qmul(qmul(angle_axis(static_cast<float>(x[5]), 2), angle_axis(static_cast<float>(x[4]), 1)),
                    angle_axis(static_cast<float>(x[3]), 0));
  const float tx = 2.0f * q.x, ty = 2.0f * q.y, tz = 2.0f * q.z;
  const float twx = tx * q.w, twy = ty * q.w, twz = tz * q.w, txx = tx * q.x, txy = ty * q.x, txz = tz * q.x;
  const float tyy = ty * q.y, tyz = tz * q.y, tzz = tz * q.z;
  float R[3][3] = {{1.0f - (tyy + tzz), txy - twz, txz + twy}, {txy + twz, 1.0f - (txx + tzz), tyz - twx},
                   {txz - twy, tyz + twx, 1.0f - (txx + tyy)}};
  orc::M4 t = orc::M4::identity();
  orc::M4 r3 = orc::M4::identity();
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) r3(i, j) = R[i][j];
  // t.topLeftCorner<3,3>() = R * t.topLeftCorner<3,3>()
  orc::M4 out = t;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) {
      float acc = r3(i, 0) * t(0, j);
      acc = acc + r3(i, 1) * t(1, j);
      acc = acc + r3(i, 2) * t(2, j);
      out(i, j) = acc;
    }
  out(0, 3) = t(0, 3) + static_cast<float>(x[0]);
  out(1, 3) = t(1, 3) + static_cast<float>(x[1]);
  out(2, 3) = t(2, 3) + static_cast<float>(x[2]);
  return out;
}

// ---- OptimizationFunctorWithIndices ------------------------------------------------------------------------------------
struct Pairs {
  const float* p;   // m x 3: output[source index]
  const float* t;   // m x 3: target point
  const double* M;  // m x 9: mahalanobis(source index), row-major
  int m;
};

struct Functor {
  const Pairs* pr = nullptr;
  void (*cb)(const double*, double*, double*) = nullptr;  // a plain objective instead of pairs (optimizer tests)
  int evals = 0;

  // one pass: f and g, exactly the sums of fdf (operator() and df take the same sums in the same order)
  void pass(const V6& x, double& f, V6* g) {
    ++evals;
    if (cb) {
      double gg[6];
      cb(x.data(), &f, gg);
      if (g)
        for (int i = 0; i < 6; ++i) (*g)[i] = gg[i];
      return;
    }
    const orc::M4 T = apply_state(x);
    f = 0;
    double gt[3] = {0, 0, 0};
    double R[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = 0; i < pr->m; ++i) {
      const float* ps = pr->p + 3 * i;
      const float* pt = pr->t + 3 * i;
      float pp[3];
      orc::transform_icp(T, ps, pp);
      const double res[3] = {static_cast<double>(pp[0] - pt[0]), static_cast<double>(pp[1] - pt[1]),
                             static_cast<double>(pp[2] - pt[2])};
      const double* M = pr->M + 9 * i;
      double temp[3];
      for (int r = 0; r < 3; ++r) temp[r] = M[3 * r] * res[0] + M[3 * r + 1] * res[1] + M[3 * r + 2] * res[2];
      f += res[0] * temp[0] + res[1] * temp[1] + res[2] * temp[2];
      for (int r = 0; r < 3; ++r) gt[r] += temp[r];
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) R[3 * r + c] += static_cast<double>(ps[r]) * temp[c];
    }
    const double m = static_cast<double>(pr->m);
    f /= m;
    if (!g) return;
    for (int r = 0; r < 3; ++r) (*g)[r] = gt[r] * (2.0 / m);
    for (int i = 0; i < 9; ++i) R[i] *= 2.0 / m;
    r_derivative(x, R, *g);
  }
  double operator()(const V6& x) {
    double f;
    pass(x, f, nullptr);
    return f;
  }
  void df(const V6& x, V6& g) {
    double f;
    pass(x, f, &g);
  }
  void fdf(const V6& x, double& f, V6& g) { pass(x, f, &g); }

  // computeRDerivative: g[3..5] = matricesInnerProd(dR/dphi, R), ... with matricesInnerProd(A, B) = sum_i sum_j A(j,i) B(i,j)
  static void r_derivative(const V6& x, const double* R, V6& g) {
    const double cphi = std::cos(x[3]), sphi = std::sin(x[3]);
    const double ctheta = std::cos(x[4]), stheta = std::sin(x[4]);
    const double cpsi = std::cos(x[5]), spsi = std::sin(x[5]);
    double a[9], b[9], c[9];  // row-major dR_dPhi, dR_dTheta, dR_dPsi
    a[0] = 0.;
    a[3] = 0.;
    a[6] = 0.;
    a[1] = sphi * spsi + cphi * cpsi * stheta;
    a[4] = -cpsi * sphi + cphi * spsi * stheta;
    a[7] = cphi * ctheta;
    a[2] = cphi * spsi - cpsi * sphi * stheta;
    a[5] = -cphi * cpsi - sphi * spsi * stheta;
    a[8] = -ctheta * sphi;
    b[0] = -cpsi * stheta;
    b[3] = -spsi * stheta;
    b[6] = -ctheta;
    b[1] = cpsi * ctheta * sphi;
    b[4] = ctheta * sphi * spsi;
    b[7] = -sphi * stheta;
    b[2] = cphi * cpsi * ctheta;
    b[5] = cphi * ctheta * spsi;
    b[8] = -cphi * stheta;
    c[0] = -ctheta * spsi;
    c[3] = cpsi * ctheta;
    c[6] = 0.;
    c[1] = -cphi * cpsi - sphi * spsi * stheta;
    c[4] = -cphi * spsi + cpsi * sphi * stheta;
    c[7] = 0.;
    c[2] = cpsi * sphi - cphi * spsi * stheta;
    c[5] = sphi * spsi + cphi * cpsi * stheta;
    c[8] = 0.;
    auto inner = [&](const double* A) {
      double r = 0.;
      for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) r += A[3 * j + i] * R[3 * i + j];
      return r;
    };
    g[3] = inner(a);
    g[4] = inner(b);
    g[5] = inner(c);
  }
};

// ---- bfgs.h -------------------------------------------------------------------------------------------------------------
enum Status { NegativeGradientEpsilon = -3, NotStarted = -2, Running = -1, Success = 0, NoProgress = 1 };

struct BFGS {
  Functor& functor;
  double rho = 0.01, sigma = 0.01, tau1 = 9, tau2 = 0.05, tau3 = 0.5, step_size = 1;
  int order = 3, bracket_iters = 100, section_iters = 100;
  V6 x0{}, g0{}, p{}, dx{}, gradient{}, x_alpha{}, g_alpha{};
  double f = 0, delta_f = 0, g0norm = 0, pnorm = 0, fp0 = 0, f_alpha = 0, df_alpha = 0;
  double x_cache_key = 0, f_cache_key = 0, df_cache_key = 0, g_cache_key = 0;

  explicit BFGS(Functor& fn) : functor(fn) {}

  double slope() { return dot(g_alpha, p); }
  void moveTo(double alpha) {
    if (alpha == x_cache_key) return;
    for (int i = 0; i < 6; ++i) x_alpha[i] = x0[i] + alpha * p[i];
    x_cache_key = alpha;
  }
  double applyF(double alpha) {
    if (alpha == f_cache_key) return f_alpha;
    moveTo(alpha);
    f_alpha = functor(x_alpha);
    f_cache_key = alpha;
    return f_alpha;
  }
  double applyDF(double alpha) {
    if (alpha == df_cache_key) return df_alpha;
    moveTo(alpha);
    if (alpha != g_cache_key) {
      functor.df(x_alpha, g_alpha);
      g_cache_key = alpha;
    }
    df_alpha = slope();
    df_cache_key = alpha;
    return df_alpha;
  }
  void applyFDF(double alpha, double& fo, double& dfo) {
    if (alpha == f_cache_key && alpha == df_cache_key) {
      fo = f_alpha;
      dfo = df_alpha;
      return;
    }
    if (alpha == f_cache_key || alpha == df_cache_key) {
      fo = applyF(alpha);
      dfo = applyDF(alpha);
      return;
    }
    moveTo(alpha);
    functor.fdf(x_alpha, f_alpha, g_alpha);
    f_cache_key = alpha;
    g_cache_key = alpha;
    df_alpha = slope();
    df_cache_key = alpha;
    fo = f_alpha;
    dfo = df_alpha;
  }
  void changeDirection() {
    x_alpha = x0;
    x_cache_key = 0.0;
    f_cache_key = 0.0;
    g_alpha = g0;
    g_cache_key = 0.0;
    df_alpha = slope();
    df_cache_key = 0.0;
  }

  static double interp_quad(double f0, double fp0, double f1, double zl, double zh) {
    const double fl = f0 + zl * (fp0 + zl * (f1 - f0 - fp0));
    const double fh = f0 + zh * (fp0 + zh * (f1 - f0 - fp0));
    const double c = 2 * (f1 - f0 - fp0);
    double zmin = zl, fmin = fl;
    if (fh < fmin) {
      zmin = zh;
      fmin = fh;
    }
    if (c > 0) {
      const double z = -fp0 / c;
      if (z > zl && z < zh) {
        const double fz = f0 + z * (fp0 + z * (f1 - f0 - fp0));
        if (fz < fmin) {
          zmin = z;
          fmin = fz;
        }
      }
    }
    return zmin;
  }
  static double cubic(double c0, double c1, double c2, double c3, double z) { return c0 + z * (c1 + z * (c2 + z * c3)); }
  static void check_extremum(double c0, double c1, double c2, double c3, double z, double& zmin, double& fmin) {
    const double y = cubic(c0, c1, c2, c3, z);
    if (y < fmin) {
      zmin = z;
      fmin = y;
    }
  }
  static int solve_quadratic(double a, double b, double c, double* x0, double* x1) {  // gsl_poly_solve_quadratic
    if (a == 0) {
      if (b == 0) return 0;
      *x0 = -c / b;
      return 1;
    }
    const double disc = b * b - 4 * a * c;
    if (disc > 0) {
      if (b == 0) {
        const double r = std::sqrt(-c / a);
        *x0 = -r;
        *x1 = r;
      } else {
        const double sgnb = (b > 0 ? 1 : -1);
        const double temp = -0.5 * (b + sgnb * std::sqrt(disc));
        const double r1 = temp / a, r2 = c / temp;
        if (r1 < r2) {
          *x0 = r1;
          *x1 = r2;
        } else {
          *x0 = r2;
          *x1 = r1;
        }
      }
      return 2;
    } else if (disc == 0) {
      *x0 = -0.5 * b / a;
      *x1 = -0.5 * b / a;
      return 2;
    }
    return 0;
  }
  static double cubicmin(double f0, double fp0, double f1, double fp1, double zl, double zh) {
    const double eta = 3 * (f1 - f0) - 2 * fp0 - fp1;
    const double xi = fp0 + fp1 - 2 * (f1 - f0);
    const double c0 = f0, c1 = fp0, c2 = eta, c3 = xi;
    double zmin = zl, fmin = cubic(c0, c1, c2, c3, zl);
    check_extremum(c0, c1, c2, c3, zh, zmin, fmin);
    double z0 = 0, z1 = 0;
    const int n = solve_quadratic(3 * c3, 2 * c2, c1, &z0, &z1);
    if (n == 2) {
      if (z0 > zl && z0 < zh) check_extremum(c0, c1, c2, c3, z0, zmin, fmin);
      if (z1 > zl && z1 < zh) check_extremum(c0, c1, c2, c3, z1, zmin, fmin);
    } else if (n == 1) {
      if (z0 > zl && z0 < zh) check_extremum(c0, c1, c2, c3, z0, zmin, fmin);
    }
    return zmin;
  }
  double interpolate(double a, double fa, double fpa, double b, double fb, double fpb, double xmin, double xmax) const {
    double zmin = (xmin - a) / (b - a), zmax = (xmax - a) / (b - a);
    if (zmin > zmax) std::swap(zmin, zmax);
    double z;
    if (order > 2 && std::isfinite(fpb))
      z = cubicmin(fa, fpa * (b - a), fb, fpb * (b - a), zmin, zmax);
    else
      z = interp_quad(fa, fpa * (b - a), fb, zmin, zmax);
    return a + z * (b - a);
  }

  Status lineSearch(double alpha1, double& alpha_new) {
    double falpha, fpalpha, delta, alpha_next;
    double alpha = alpha1, alpha_prev = 0.0;
    int i = 0;
    const double f0 = applyF(0.0);
    const double fp0l = applyDF(0.0);
    double falpha_prev = f0, fpalpha_prev = fp0l;
    double a = 0.0, b = alpha, fa = f0, fb = 0.0, fpa = fp0l, fpb = 0.0;
    const double nan = std::numeric_limits<double>::quiet_NaN();
    while (i++ < bracket_iters) {
      falpha = applyF(alpha);
      if (falpha > f0 + alpha * rho * fp0l || falpha >= falpha_prev) {
        a = alpha_prev;
        fa = falpha_prev;
        fpa = fpalpha_prev;
        b = alpha;
        fb = falpha;
        fpb = nan;
        break;
      }
      fpalpha = applyDF(alpha);
      if (std::fabs(fpalpha) <= -sigma * fp0l) {
        alpha_new = alpha;
        return Success;
      }
      if (fpalpha >= 0) {
        a = alpha;
        fa = falpha;
        fpa = fpalpha;
        b = alpha_prev;
        fb = falpha_prev;
        fpb = fpalpha_prev;
        break;
      }
      delta = alpha - alpha_prev;
      alpha_next = interpolate(alpha_prev, falpha_prev, fpalpha_prev, alpha, falpha, fpalpha, alpha + delta, alpha + tau1 * delta);
      alpha_prev = alpha;
      falpha_prev = falpha;
      fpalpha_prev = fpalpha;
      alpha = alpha_next;
    }
    while (i++ < section_iters) {
      delta = b - a;
      alpha = interpolate(a, fa, fpa, b, fb, fpb, a + tau2 * delta, b - tau3 * delta);
      falpha = applyF(alpha);
      if ((a - alpha) * fpa <= std::numeric_limits<double>::epsilon()) return NoProgress;
      if (falpha > f0 + rho * alpha * fp0l || falpha >= fa) {
        b = alpha;
        fb = falpha;
        fpb = nan;
      } else {
        fpalpha = applyDF(alpha);
        if (std::fabs(fpalpha) <= -sigma * fp0l) {
          alpha_new = alpha;
          return Success;
        }
        if (((b - a) >= 0 && fpalpha >= 0) || ((b - a) <= 0 && fpalpha <= 0)) {
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
    return Success;
  }

  Status minimizeInit(const V6& x) {
    delta_f = 0;
    dx.fill(0.0);
    functor.fdf(x, f, gradient);
    x0 = x;
    g0 = gradient;
    g0norm = norm(g0);
    for (int i = 0; i < 6; ++i) p[i] = gradient[i] * -1 / g0norm;
    pnorm = norm(p);
    fp0 = -g0norm;
    x_alpha = x0;
    x_cache_key = 0;
    f_alpha = f;
    f_cache_key = 0;
    g_alpha = g0;
    g_cache_key = 0;
    df_alpha = slope();
    df_cache_key = 0;
    return NotStarted;
  }

  Status minimizeOneStep(V6& x) {
    double alpha = 0.0, alpha1;
    const double f0 = f;
    if (pnorm == 0.0 || g0norm == 0.0 || fp0 == 0) {
      dx.fill(0.0);
      return NoProgress;
    }
    if (delta_f < 0) {
      const double del = std::max(-delta_f, 10 * std::numeric_limits<double>::epsilon() * std::fabs(f0));
      alpha1 = std::min(1.0, 2.0 * del / (-fp0));
    } else {
      alpha1 = std::fabs(step_size);
    }
    const Status status = lineSearch(alpha1, alpha);
    if (status != Success) return status;
    {  // updatePosition
      double fa, dfa;
      applyFDF(alpha, fa, dfa);
    }
    f = f_alpha;
    x = x_alpha;
    gradient = g_alpha;
    delta_f = f - f0;
    {
      V6 dx0, dg0;
      for (int i = 0; i < 6; ++i) {
        dx0[i] = x[i] - x0[i];
        dg0[i] = gradient[i] - g0[i];
      }
      dx = dx0;
      const double dxg = dot(dx0, gradient), dgg = dot(dg0, gradient), dxdg = dot(dx0, dg0);
      const double dgnorm = norm(dg0);
      double A, B;
      if (dxdg != 0) {
        B = dxg / dxdg;
        A = -(1.0 + dgnorm * dgnorm / dxdg) * B + dgg / dxdg;
      } else {
        B = 0;
        A = 0;
      }
      for (int i = 0; i < 6; ++i) p[i] = gradient[i] - A * dx0[i] - B * dg0[i];
    }
    g0 = gradient;
    x0 = x;
    g0norm = norm(g0);
    pnorm = norm(p);
    const double dir = (dot(p, gradient) >= 0) ? -1.0 : 1.0;
    for (int i = 0; i < 6; ++i) p[i] *= dir / pnorm;
    pnorm = norm(p);
    fp0 = dot(p, g0);
    changeDirection();
    return Success;
  }

  Status testGradient(double epsilon) {
    if (epsilon < 0) return NegativeGradientEpsilon;
    return norm(gradient) < epsilon ? Success : Running;
  }
};

// estimateRigidTransformationBFGS's loop; returns the inner iterations
static int minimize(Functor& fn, V6& x, int max_inner) {
  BFGS bfgs(fn);
  int inner = 0;
  int result = bfgs.minimizeInit(x);
  result = Running;
  do {
    inner++;
    result = bfgs.minimizeOneStep(x);
    if (result) break;
    result = bfgs.testGradient(1e-2);
  } while (result == Running && inner < max_inner);
  return inner;
}

}  // namespace orc_gicp

extern "C" {

ORC_API void orc_gicp_covariances(const void* pts, size_t n, size_t stride, int k, double* out9) {
  orc::KdTree tree;
  tree.build(pts, n, stride);
  std::vector<int> idx(k);
  std::vector<float> d2(k), nb(3 * k);
  for (size_t i = 0; i < n; ++i) {
    const float* p = orc::rec(pts, i, stride);
    if (!orc::finite3(p[0], p[1], p[2])) {
      for (int e = 0; e < 9; ++e) out9[9 * i + e] = std::numeric_limits<double>::quiet_NaN();
      continue;
    }
    const int cnt = tree.knn(p, k, idx.data(), d2.data());
    for (int j = 0; j < cnt; ++j) {
      const float* q = orc::rec(pts, idx[j], stride);
      nb[3 * j] = q[0];
      nb[3 * j + 1] = q[1];
      nb[3 * j + 2] = q[2];
    }
    orc_gicp::covariance(nb.data(), cnt, out9 + 9 * i);
  }
}

ORC_API void orc_gicp_fg(const float* p3, const float* t3, const double* M9, int m, const double* x6, double* f, double* g6) {
  orc_gicp::Pairs pr{p3, t3, M9, m};
  orc_gicp::Functor fn;
  fn.pr = &pr;
  orc_gicp::V6 x, g;
  for (int i = 0; i < 6; ++i) x[i] = x6[i];
  fn.fdf(x, *f, g);
  for (int i = 0; i < 6; ++i) g6[i] = g[i];
}

ORC_API void orc_gicp_apply_state(const double* x6, float* T16) {
  orc_gicp::V6 x;
  for (int i = 0; i < 6; ++i) x[i] = x6[i];
  const orc::M4 T = orc_gicp::apply_state(x);
  std::memcpy(T16, T.m, sizeof(T.m));
}

// pairs, or (p3 == NULL) the objective cb; x6 in / out; returns the inner iterations
ORC_API int orc_gicp_bfgs(const float* p3, const float* t3, const double* M9, int m, void (*cb)(const double*, double*, double*),
                          double* x6, int max_inner, int* evals) {
  orc_gicp::Pairs pr{p3, t3, M9, m};
  orc_gicp::Functor fn;
  if (p3) fn.pr = &pr;
  else fn.cb = cb;
  orc_gicp::V6 x;
  for (int i = 0; i < 6; ++i) x[i] = x6[i];
  const int inner = orc_gicp::minimize(fn, x, max_inner);
  for (int i = 0; i < 6; ++i) x6[i] = x[i];
  if (evals) *evals = fn.evals;
  return inner;
}

// computeTransformation + getFitnessScore(params->fitness_max_range); guess16: column-major (NULL: identity)
ORC_API void orc_gicp_align(const void* src, size_t ns, size_t sstride, const void* tgt, size_t nt, size_t tstride,
                            const float* guess16, const peb_gicp_params* prm, peb_icp_result* out) {
  const int k = prm->k_correspondences;
  std::vector<double> Cs(9 * ns), Ct(9 * nt);
  orc_gicp_covariances(src, ns, sstride, k, Cs.data());
  orc_gicp_covariances(tgt, nt, tstride, k, Ct.data());
  orc::KdTree tree;
  tree.build(tgt, nt, tstride);
  orc::M4 guess = orc::M4::identity();
  if (guess16) std::memcpy(guess.m, guess16, sizeof(guess.m));
  // output = transformPointCloud(input, guess); non-finite points are no queries
  std::vector<int> sidx;
  std::vector<float> output;
  for (size_t i = 0; i < ns; ++i) {
    const float* p = orc::rec(src, i, sstride);
    if (!orc::finite3(p[0], p[1], p[2])) continue;
    float o[3];
    orc::transform_tpc(guess, p, o);
    sidx.push_back(static_cast<int>(i));
    output.insert(output.end(), o, o + 3);
  }
  orc::M4 transformation = orc::M4::identity(), previous = transformation;
  const double dist_threshold = prm->max_corr_dist * prm->max_corr_dist;
  int nr_iterations = 0, converged = 0, state = PEB_NOT_CONVERGED, m = 0;
  double last_mse = DBL_MAX;
  for (;;) {
    double R[9];
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) {
        double a = 0;
        for (int kk = 0; kk < 4; ++kk) a += static_cast<double>(transformation(i, kk)) * static_cast<double>(guess(kk, j));
        R[3 * i + j] = a;
      }
    std::vector<float> pp, tp;
    std::vector<double> Ms;
    double sum_d2 = 0;
    for (size_t q = 0; q < sidx.size(); ++q) {
      float query[3];
      orc::transform_icp(transformation, &output[3 * q], query);
      int j;
      float d2;
      if (tree.knn(query, 1, &j, &d2) == 0) continue;
      if (!(static_cast<double>(d2) < dist_threshold)) continue;
      const double* C1 = &Cs[9 * sidx[q]];
      const double* C2 = &Ct[9 * j];
      double RC[9], tmp[9];
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) RC[3 * r + c] = R[3 * r] * C1[c] + R[3 * r + 1] * C1[3 + c] + R[3 * r + 2] * C1[6 + c];
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) tmp[3 * r + c] = RC[3 * r] * R[3 * c] + RC[3 * r + 1] * R[3 * c + 1] + RC[3 * r + 2] * R[3 * c + 2];
      for (int e = 0; e < 9; ++e) tmp[e] += C2[e];
      auto cof = [&](int i, int jj) {
        const int i1 = (i + 1) % 3, i2 = (i + 2) % 3, j1 = (jj + 1) % 3, j2 = (jj + 2) % 3;
        return tmp[3 * i1 + j1] * tmp[3 * i2 + j2] - tmp[3 * i1 + j2] * tmp[3 * i2 + j1];
      };
      const double det = cof(0, 0) * tmp[0] + cof(1, 0) * tmp[3] + cof(2, 0) * tmp[6];
      const double invdet = 1.0 / det;
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) Ms.push_back(cof(c, r) * invdet);
      pp.insert(pp.end(), &output[3 * q], &output[3 * q] + 3);
      const float* t = orc::rec(tgt, j, tstride);
      tp.insert(tp.end(), t, t + 3);
      sum_d2 += static_cast<double>(d2);
    }
    m = static_cast<int>(pp.size() / 3);
    last_mse = m > 0 ? sum_d2 / m : DBL_MAX;
    previous = transformation;
    if (m < 4) {  // NotEnoughPointsException: the loop ends, converged_ stays false
      state = PEB_NO_CORRESPONDENCES;
      break;
    }
    orc_gicp::V6 x;
    x[0] = transformation(0, 3);
    x[1] = transformation(1, 3);
    x[2] = transformation(2, 3);
    x[3] = std::atan2(transformation(2, 1), transformation(2, 2));
    x[4] = std::asin(-transformation(2, 0));
    x[5] = std::atan2(transformation(1, 0), transformation(0, 0));
    orc_gicp::Pairs pr{pp.data(), tp.data(), Ms.data(), m};
    orc_gicp::Functor fn;
    fn.pr = &pr;
    orc_gicp::minimize(fn, x, prm->max_inner_iterations);
    transformation = orc_gicp::apply_state(x);
    double delta = 0.;
    for (int kk = 0; kk < 4; kk++)
      for (int l = 0; l < 4; l++) {
        const double ratio = (kk < 3 && l < 3) ? 1. / prm->rotation_epsilon : 1. / prm->transformation_epsilon;
        const double c_delta = ratio * std::fabs(previous(kk, l) - transformation(kk, l));
        if (c_delta > delta) delta = c_delta;
      }
    nr_iterations++;
    if (nr_iterations >= prm->max_iterations || delta < 1) {
      converged = 1;
      state = delta < 1 ? PEB_TRANSFORM : PEB_ITERATIONS;
      previous = transformation;
      break;
    }
  }
  const orc::M4 final_t = orc::mul(previous, guess);
  // getFitnessScore(max_range): transformPointCloud(input, final), nearest target point, mean of d2 <= max_range
  double fit = 0;
  int nfit = 0;
  for (size_t i = 0; i < ns; ++i) {
    const float* p = orc::rec(src, i, sstride);
    if (!orc::finite3(p[0], p[1], p[2])) continue;
    float o[3];
    orc::transform_tpc(final_t, p, o);
    int j;
    float d2;
    if (tree.knn(o, 1, &j, &d2) == 0) continue;
    if (static_cast<double>(d2) <= prm->fitness_max_range) {
      fit += d2;
      ++nfit;
    }
  }
  std::memcpy(out->T, final_t.m, sizeof(out->T));
  out->fitness = nfit > 0 ? fit / nfit : DBL_MAX;
  out->last_mse = last_mse;
  out->iterations = nr_iterations;
  out->converged = converged;
  out->state = state;
  out->n_correspondences = m;
}

}  // extern "C"
