// Host build of fast3r_b200/csrc/pnp_math.h for tests/test_pnp_cpu.py (C entry points for ctypes).
#include "pnp_math.h"

extern "C" {

int f3r_test_pnp_sample4(uint32_t m, uint32_t k, uint32_t i, uint32_t* out) { return f3r::pnp_sample4(m, k, i, out) ? 1 : 0; }

int f3r_test_p3p(const double* b, const double* X, double* R, double* t) {
  double bb[3][3], xx[3][3], r[4][9], tt[4][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) { bb[i][j] = b[3 * i + j]; xx[i][j] = X[3 * i + j]; }
  const int n = f3r::p3p_grunert(bb, xx, r, tt);
  for (int s = 0; s < n; ++s) {
    for (int j = 0; j < 9; ++j) R[9 * s + j] = r[s][j];
    for (int j = 0; j < 3; ++j) t[3 * s + j] = tt[s][j];
  }
  return n;
}

int f3r_test_hypothesis(const double* X, const double* uv, double f, double cx, double cy, double* pose) {
  double xx[4][3], u[4][2];
  for (int i = 0; i < 4; ++i) {
    for (int j = 0; j < 3; ++j) xx[i][j] = X[3 * i + j];
    u[i][0] = uv[2 * i]; u[i][1] = uv[2 * i + 1];
  }
  return f3r::p3p_hypothesis(xx, u, f, cx, cy, pose) ? 1 : 0;
}

int f3r_test_chol6(const double* upper, const double* rhs, double* x) { return f3r::chol6_solve(upper, rhs, x) ? 1 : 0; }

}
