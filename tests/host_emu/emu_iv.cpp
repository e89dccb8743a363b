// TEST-ONLY host emulation of the implied-volatility arithmetic (option-pricing-ffn-lbfgs_b200/csrc/dhj_iv.cuh): the
// same scalar functions, compiled by g++ with FMA contraction off.  glibc has no erfcx, so one is supplied here from
// long-double erfc / exp (and an asymptotic series beyond 100); the emulation differs from the device only in libm.
// Built on the fly by tests/test_iv_cpu.py; nothing in the product loads it.
#include <math.h>
#include <stdint.h>

#include "dhj_iv.cuh"

namespace dhj {
namespace iv {
double erfcx_(double z) {
  if (z > 100.0) {
    const long double r = 1.0L / ((long double)z * z);
    const long double s = 1.0L - r * (0.5L - r * (0.75L - r * (1.875L - r * 6.5625L)));
    return (double)(s / ((long double)z * 1.7724538509055160273L));
  }
  if (z < -27.0) return INFINITY;
  const long double zl = z;
  return (double)(expl(zl * zl) * erfcl(zl));
}
}  // namespace iv
}  // namespace dhj

using namespace dhj::iv;

extern "C" {

void emu_implied_vol(int64_t n, const double* V, const double* S0, const double* K, const double* T, const double* r,
                     const double* q, const int32_t* is_call, double* out, int32_t* status, int32_t* iters) {
  for (int64_t i = 0; i < n; ++i) {
    int st, it;
    out[i] = implied_vol(V[i], S0[i], K[i], T[i], r[i], q[i], is_call[i] != 0, &st, &it);
    status[i] = st;
    iters[i] = it;
  }
}

void emu_bs_price(int64_t n, const double* sigma, const double* S0, const double* K, const double* T, const double* r,
                  const double* q, const int32_t* is_call, double* out) {
  for (int64_t i = 0; i < n; ++i) out[i] = bs_price(sigma[i], S0[i], K[i], T[i], r[i], q[i], is_call[i] != 0);
}

// b(x, s) (region chosen as in the solver), the series and the erfcx difference on their own, and the complement
void emu_b(int64_t n, const double* x, const double* s, double* b, double* series, double* plain, double* compl_) {
  for (int64_t i = 0; i < n; ++i) {
    const double h = x[i] / s[i], t = 0.5 * s[i];
    b[i] = b_norm(x[i], s[i]);
    series[i] = b_series(h, t);
    plain[i] = 0.5 * gauss2(h, t) * (erfcx_(-(h + t) * kInvSqrt2) - erfcx_((t - h) * kInvSqrt2));
    compl_[i] = b_complement(h, t);
  }
}

double emu_erfcx(double z) { return erfcx_(z); }
}
