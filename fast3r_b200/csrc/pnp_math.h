// Host/device fp64 math of the PnP-RANSAC pipeline (pnp.cu): the hypothesis sampler, the P3P minimal solver, the 6x6
// Cholesky solve of the Levenberg-Marquardt refit and pose helpers.  Plain C++ as well, so the CPU test suite runs
// exactly this code (tests/pnp_math_host.cpp) against the numpy oracle (tests/pnp_oracle.py).
#pragma once
#include <math.h>
#include <stdint.h>

#ifndef F3R_HD
#if defined(__CUDACC__)
#define F3R_HD __host__ __device__
#else
#define F3R_HD
#endif
#endif

namespace f3r {

// Fixed seed of the hypothesis sampler: results are a pure function of the inputs.
constexpr uint64_t PNP_SEED = 0x3f3a2b1c0d0e0f10ull;
constexpr int PNP_MAX_DRAWS = 64;  // draws allowed to find 4 distinct entries (then the hypothesis is invalid)

F3R_HD inline uint64_t splitmix64(uint64_t x) {
  uint64_t z = x + 0x9e3779b97f4a7c15ull;
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}

// Draw d of hypothesis (k, i): an entry of a list of m, by multiply-high of the hash's top 32 bits.  The view is not part
// of the key, so a view gets the same samples whichever call (and position in it) it is processed in.
F3R_HD inline uint32_t pnp_draw(uint32_t m, uint32_t k, uint32_t i, uint32_t d) {
  const uint64_t h = splitmix64(splitmix64(splitmix64(PNP_SEED ^ k) ^ i) ^ d);
  return static_cast<uint32_t>(((h >> 32) * static_cast<uint64_t>(m)) >> 32);
}

// 4 distinct entries of [0, m) for hypothesis (k, i); false when m < 4 or the draws run out.
F3R_HD inline bool pnp_sample4(uint32_t m, uint32_t k, uint32_t i, uint32_t out[4]) {
  if (m < 4) return false;
  int n = 0;
  for (uint32_t d = 0; d < static_cast<uint32_t>(PNP_MAX_DRAWS) && n < 4; ++d) {
    const uint32_t e = pnp_draw(m, k, i, d);
    bool dup = false;
    for (int j = 0; j < n; ++j) dup |= out[j] == e;
    if (!dup) out[n++] = e;
  }
  return n == 4;
}

F3R_HD inline double poly_eval(const double* c, int deg, double x) {  // c[0] x^deg + ... + c[deg]
  double r = c[0];
  for (int j = 1; j <= deg; ++j) r = r * x + c[j];
  return r;
}

// Real roots of a monic polynomial of degree deg in [lo0, hi0] given its sorted critical points: one bisection per
// monotone interval with a sign change, down to adjacent doubles.
F3R_HD inline int roots_between(const double* c, int deg, const double* crit, int ncrit, double lo0, double hi0, double* out) {
  int n = 0;
  double a = lo0;
  for (int s = 0; s <= ncrit; ++s) {
    const double b = (s < ncrit) ? crit[s] : hi0;
    if (b > a) {
      double lo = a, hi = b, flo = poly_eval(c, deg, lo), fhi = poly_eval(c, deg, hi);
      if (flo == 0.0) {
        if (n == 0 || out[n - 1] != lo) out[n++] = lo;
      } else if (fhi != 0.0 && (flo < 0.0) != (fhi < 0.0)) {
        for (int it = 0; it < 200; ++it) {
          const double mid = 0.5 * (lo + hi);
          if (!(mid > lo && mid < hi)) break;
          const double fm = poly_eval(c, deg, mid);
          if (fm == 0.0) { lo = hi = mid; break; }
          if ((fm < 0.0) == (flo < 0.0)) { lo = mid; flo = fm; } else { hi = mid; }
        }
        out[n++] = 0.5 * (lo + hi);
      }
    }
    a = (s < ncrit) ? crit[s] : a;
  }
  if (poly_eval(c, deg, hi0) == 0.0 && (n == 0 || out[n - 1] != hi0)) out[n++] = hi0;
  return n;
}

// Real roots (ascending) of a4 x^4 + a3 x^3 + a2 x^2 + a1 x + a0 with a4 != 0: the roots of each derivative bracket
// those of the polynomial above it (quadratic -> cubic -> quartic), inside the Cauchy bound.
F3R_HD inline int quartic_real_roots(const double a[5], double out[4]) {
  if (!(a[0] != 0.0) || !isfinite(a[0])) return 0;
  double c4[5];
  double bound = 0.0;
  for (int j = 0; j < 5; ++j) c4[j] = a[j] / a[0];
  for (int j = 1; j < 5; ++j) bound = fmax(bound, fabs(c4[j]));
  if (!isfinite(bound)) return 0;
  bound += 1.0;
  const double c3[4] = {1.0, 0.75 * c4[1], 0.5 * c4[2], 0.25 * c4[3]};  // p'/4
  const double c2[3] = {1.0, 2.0 * c3[1] / 3.0, c3[2] / 3.0};          // (p'/4)'/3
  double r2[2];
  int n2 = 0;
  const double disc = c2[1] * c2[1] - 4.0 * c2[2];
  if (disc >= 0.0) {
    const double sq = sqrt(disc);
    r2[0] = 0.5 * (-c2[1] - sq);
    r2[1] = 0.5 * (-c2[1] + sq);
    n2 = 2;
  }
  double r3[3];
  const int n3 = roots_between(c3, 3, r2, n2, -bound, bound, r3);
  return roots_between(c4, 4, r3, n3, -bound, bound, out);
}

F3R_HD inline void cross3d(const double* a, const double* b, double* c) {
  c[0] = a[1] * b[2] - a[2] * b[1];
  c[1] = a[2] * b[0] - a[0] * b[2];
  c[2] = a[0] * b[1] - a[1] * b[0];
}
F3R_HD inline double dot3d(const double* a, const double* b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }

constexpr double PNP_MIN_SINE = 1e-5;  // point triples closer than this (sine of the angle at p0) to collinear are rejected

// Orthonormal frame (columns e1 e2 e3) of a point triple: e1 along p1 - p0, e3 normal to the triangle.  false for a
// (numerically) collinear triple.
F3R_HD inline bool triad(const double* p0, const double* p1, const double* p2, double f[9]) {
  double e1[3] = {p1[0] - p0[0], p1[1] - p0[1], p1[2] - p0[2]}, d2[3] = {p2[0] - p0[0], p2[1] - p0[1], p2[2] - p0[2]};
  double e3[3], e2[3];
  cross3d(e1, d2, e3);
  const double l1 = sqrt(dot3d(e1, e1)), l2 = sqrt(dot3d(d2, d2)), l3 = sqrt(dot3d(e3, e3));
  if (!(l1 > 0.0) || !(l3 > PNP_MIN_SINE * l1 * l2)) return false;
  for (int j = 0; j < 3; ++j) { e1[j] /= l1; e3[j] /= l3; }
  cross3d(e3, e1, e2);
  for (int r = 0; r < 3; ++r) { f[3 * r] = e1[r]; f[3 * r + 1] = e2[r]; f[3 * r + 2] = e3[r]; }
  return true;
}

// P3P after Grunert (1841), in the form of Haralick et al. (IJCV 1994): with s_j the depths along the unit bearings b_j
// and s2 = u s1, s3 = v s1, the three laws of cosines reduce to a quartic in v.  For each real root with positive
// depths, the camera-frame points s_j b_j and the world points X_j give (R, t) with Xc = R X + t by aligning the two
// triangles' frames.  R row-major [9], t [3]; returns the number of solutions (<= 4).
F3R_HD inline int p3p_grunert(const double b[3][3], const double X[3][3], double R[4][9], double t[4][3]) {
  const double ca = dot3d(b[1], b[2]), cb = dot3d(b[0], b[2]), cg = dot3d(b[0], b[1]);
  double d[3];
  for (int j = 0; j < 3; ++j) d[j] = X[1][j] - X[2][j];
  const double a2 = dot3d(d, d);
  for (int j = 0; j < 3; ++j) d[j] = X[0][j] - X[2][j];
  const double b2 = dot3d(d, d);
  for (int j = 0; j < 3; ++j) d[j] = X[0][j] - X[1][j];
  const double c2 = dot3d(d, d);
  if (!(b2 > 0.0) || !(a2 > 0.0) || !(c2 > 0.0)) return 0;
  const double p = (a2 - c2) / b2, q = (a2 + c2) / b2;
  double A[5];
  A[0] = (p - 1.0) * (p - 1.0) - 4.0 * c2 / b2 * ca * ca;
  A[1] = 4.0 * (p * (1.0 - p) * cb - (1.0 - q) * ca * cg + 2.0 * c2 / b2 * ca * ca * cb);
  A[2] = 2.0 * (p * p - 1.0 + 2.0 * p * p * cb * cb + 2.0 * (b2 - c2) / b2 * ca * ca - 4.0 * q * ca * cb * cg +
                2.0 * (b2 - a2) / b2 * cg * cg);
  A[3] = 4.0 * (-p * (1.0 + p) * cb + 2.0 * a2 / b2 * cg * cg * cb - (1.0 - q) * ca * cg);
  A[4] = (1.0 + p) * (1.0 + p) - 4.0 * a2 / b2 * cg * cg;
  double roots[4];
  const int nr = quartic_real_roots(A, roots);
  double fw[9];
  if (!triad(X[0], X[1], X[2], fw)) return 0;
  int ns = 0;
  for (int r = 0; r < nr; ++r) {
    const double v = roots[r];
    const double den = 2.0 * (cg - v * ca);
    const double s1sq = b2 / (1.0 + v * v - 2.0 * v * cb);
    if (den == 0.0 || !(s1sq > 0.0)) continue;
    const double u = ((p - 1.0) * v * v - 2.0 * p * cb * v + 1.0 + p) / den;
    const double s1 = sqrt(s1sq), s[3] = {s1, u * s1, v * s1};
    if (!(s[1] > 0.0) || !(s[2] > 0.0) || !isfinite(s[1]) || !isfinite(s[2])) continue;
    double pc[3][3];
    for (int i = 0; i < 3; ++i)
      for (int j = 0; j < 3; ++j) pc[i][j] = s[i] * b[i][j];
    double fc[9];
    if (!triad(pc[0], pc[1], pc[2], fc)) continue;
    double* Ri = R[ns];
    for (int i = 0; i < 3; ++i)  // R = Fc Fw^T
      for (int j = 0; j < 3; ++j) Ri[3 * i + j] = fc[3 * i] * fw[3 * j] + fc[3 * i + 1] * fw[3 * j + 1] + fc[3 * i + 2] * fw[3 * j + 2];
    for (int i = 0; i < 3; ++i) t[ns][i] = pc[0][i] - (Ri[3 * i] * X[0][0] + Ri[3 * i + 1] * X[0][1] + Ri[3 * i + 2] * X[0][2]);
    ++ns;
  }
  return ns;
}

// Squared pixel error of world point X under (R, t) and the pinhole (f, cx, cy); +inf when the point is not in front.
F3R_HD inline double reproj_err2(const double* R, const double* t, double f, double cx, double cy, const double* X,
                                 double u, double v) {
  const double xc = R[0] * X[0] + R[1] * X[1] + R[2] * X[2] + t[0];
  const double yc = R[3] * X[0] + R[4] * X[1] + R[5] * X[2] + t[1];
  const double zc = R[6] * X[0] + R[7] * X[1] + R[8] * X[2] + t[2];
  if (!(zc > 0.0)) return INFINITY;
  const double du = f * xc / zc + cx - u, dv = f * yc / zc + cy - v;
  return du * du + dv * dv;
}

// One hypothesis from 4 correspondences (world X[4], pixels uv[4]): P3P on the first three, the solution that
// reprojects the fourth best.  pose = R row-major (9) | t (3).  false when no solution puts the fourth point in front.
F3R_HD inline bool p3p_hypothesis(const double X[4][3], const double uv[4][2], double f, double cx, double cy, double pose[12]) {
  double b[3][3];
  for (int j = 0; j < 3; ++j) {
    const double x = (uv[j][0] - cx) / f, y = (uv[j][1] - cy) / f, n = sqrt(x * x + y * y + 1.0);
    b[j][0] = x / n; b[j][1] = y / n; b[j][2] = 1.0 / n;
  }
  double R[4][9], t[4][3];
  const int ns = p3p_grunert(b, X, R, t);
  int best = -1;
  double best_e = INFINITY;
  for (int s = 0; s < ns; ++s) {
    const double e = reproj_err2(R[s], t[s], f, cx, cy, X[3], uv[3][0], uv[3][1]);
    if (e < best_e) { best_e = e; best = s; }
  }
  if (best < 0) return false;
  for (int j = 0; j < 9; ++j) pose[j] = R[best][j];
  for (int j = 0; j < 3; ++j) pose[9 + j] = t[best][j];
  return true;
}

// P = K [R | t] (row-major 3x4) for K = [[f, 0, cx], [0, f, cy], [0, 0, 1]]
F3R_HD inline void projection_matrix(const double pose[12], double f, double cx, double cy, double P[12]) {
  const double* R = pose;
  const double* t = pose + 9;
  for (int j = 0; j < 3; ++j) {
    P[j] = f * R[j] + cx * R[6 + j];
    P[4 + j] = f * R[3 + j] + cy * R[6 + j];
    P[8 + j] = R[6 + j];
  }
  P[3] = f * t[0] + cx * t[2];
  P[7] = f * t[1] + cy * t[2];
  P[11] = t[2];
}

// Solves (A) x = b for a symmetric positive definite 6x6 A given as its upper triangle, row by row (21 values);
// false when A is not numerically positive definite.
F3R_HD inline bool chol6_solve(const double* upper, const double* rhs, double* x) {
  double L[6][6];
  int k = 0;
  double A[6][6];
  for (int i = 0; i < 6; ++i)
    for (int j = i; j < 6; ++j) A[i][j] = A[j][i] = upper[k++];
  for (int j = 0; j < 6; ++j) {
    double s = A[j][j];
    for (int p = 0; p < j; ++p) s -= L[j][p] * L[j][p];
    if (!(s > 0.0)) return false;
    L[j][j] = sqrt(s);
    for (int i = j + 1; i < 6; ++i) {
      double v = A[i][j];
      for (int p = 0; p < j; ++p) v -= L[i][p] * L[j][p];
      L[i][j] = v / L[j][j];
    }
  }
  double y[6];
  for (int i = 0; i < 6; ++i) {
    double v = rhs[i];
    for (int p = 0; p < i; ++p) v -= L[i][p] * y[p];
    y[i] = v / L[i][i];
  }
  for (int i = 5; i >= 0; --i) {
    double v = y[i];
    for (int p = i + 1; p < 6; ++p) v -= L[p][i] * x[p];
    x[i] = v / L[i][i];
  }
  return true;
}

// pose' = (exp([w]x) R, t + dt) for the increment d = (w, dt): the left-multiplied rotation update of the refit
F3R_HD inline void pose_update(const double pose[12], const double d[6], double out[12]) {
  const double th = sqrt(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
  double E[9];
  const double kx = th > 0.0 ? d[0] / th : 0.0, ky = th > 0.0 ? d[1] / th : 0.0, kz = th > 0.0 ? d[2] / th : 0.0;
  const double c = cos(th), s = sin(th), v = 1.0 - c;
  E[0] = c + kx * kx * v;      E[1] = kx * ky * v - kz * s; E[2] = kx * kz * v + ky * s;
  E[3] = ky * kx * v + kz * s; E[4] = c + ky * ky * v;      E[5] = ky * kz * v - kx * s;
  E[6] = kz * kx * v - ky * s; E[7] = kz * ky * v + kx * s; E[8] = c + kz * kz * v;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) out[3 * i + j] = E[3 * i] * pose[j] + E[3 * i + 1] * pose[3 + j] + E[3 * i + 2] * pose[6 + j];
  for (int j = 0; j < 3; ++j) out[9 + j] = pose[9 + j] + d[3 + j];
}

// camera-to-world [R^T | -R^T t] (3x4 row-major) of the world-to-camera pose (R | t)
F3R_HD inline void pose_inverse(const double pose[12], double c2w[12]) {
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) c2w[4 * i + j] = pose[3 * j + i];
    c2w[4 * i + 3] = -(pose[i] * pose[9] + pose[3 + i] * pose[10] + pose[6 + i] * pose[11]);
  }
}

}  // namespace f3r
