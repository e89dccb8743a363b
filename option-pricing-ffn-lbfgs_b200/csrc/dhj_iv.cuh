// dhj_iv.cuh — Black–Scholes implied volatility (and its forward map) of option prices, one thread per option.
//
// Conventions (DESIGN.md §6d): F = S0 e^{(r-q)T}, D = e^{-rT}, x = ln(F/K), beta = V / (D sqrt(FK)), s = sigma sqrt(T).
// The normalised Black call price is b(x, s) = e^{x/2} Phi(x/s + s/2) - e^{-x/2} Phi(x/s - s/2).  The normalised
// intrinsic value iota is subtracted and put/call symmetry maps every option to the out-of-the-money call at
// x_o = -|x| <= 0, so the solver inverts b(x_o, s) = beta_o = beta - iota with 0 < beta_o < e^{x_o/2}.
//
// With h = x/s, t = s/2 and Y(z) = Phi(z)/phi(z) = sqrt(pi/2) erfcx(-z/sqrt2):
//     b = phi(h) e^{-t^2/2} [Y(h + t) - Y(h - t)],      db/ds = e^{-(h^2+t^2)/2} / sqrt(2 pi).
// The difference of the two Y values loses about |h|/s digits at small s (a few 1e-12 relative at s = 1e-3), so b
// is evaluated in three regions:
//   s < 0.5          odd Taylor series in t at fixed h: Y(h+t) - Y(h-t) = 2 sum_{k odd} M_k(h) t^k / k!, where
//                    M_k = Y^{(k)}(h) = int_0^inf u^k e^{hu - u^2/2} du > 0 (M_1 = 1 + h M_0,
//                    M_{k+1} = h M_k + k M_{k-1}); for h <= 0, M_{k+2} <= (k+1) M_k, so term k+2 is at most
//                    t^2/(k+2) of term k and nine terms (k <= 17) reach 1e-17 at t = 0.25;
//   h + t < 5        the erfcx difference above;
//   h + t >= 5       e^{x/2} Phi(h+t) - e^{-x/2} Phi(h-t) by erfc (b is within 1e-5 of e^{x/2}, nothing cancels).
// Solver: safeguarded Halley iteration on ln b, started at the inflection point s_c = sqrt(2|x_o|).  Below s_c (the
// lower branch, where b is exponentially flat) it steps in w = 1/s^2, in which ln b ~ -x^2 w / 2 is nearly linear;
// above s_c it steps in s (ln b is concave there, so the iteration is monotone from s_c).  When beta_o > e^{x/2}/2 it
// iterates on ln(e^{x/2} - b) instead: the complement, an erfcx sum, keeps the digits that b loses near its upper
// bound, and e^{x/2} - beta_o is exact there.  A bracket [lo, hi] is kept and a step that leaves it is replaced by
// bisection in log s.  Stop: |step| <= 2 eps s, or a residual below 1e-10 whose step stopped shrinking (the
// evaluation's rounding floor); 40 evaluations at most.
//
// Scalar functions are DHJ_HD: nvcc compiles them for the kernels below, g++ for the host emulation of the tests
// (tests/host_emu/emu_iv.cpp), which supplies erfcx (glibc has none).  Build with FMA contraction off.
#pragma once
#include <math.h>
#include <stdint.h>

#include "dhj_math.cuh"

namespace dhj {
namespace iv {

// status per option (include/dhj.h)
enum : int { kOk = 0, kBelowLower = 1, kAboveUpper = 2, kInvalid = 3, kNotConverged = 4 };

constexpr int kMaxIter = 40;
constexpr double kEps = 2.220446049250313e-16;     // 2^-52
constexpr double kInvSqrt2 = 0.7071067811865476;
constexpr double kInvSqrt2Pi = 0.3989422804014327;
constexpr double kSqrt2Pi = 2.5066282746310002;
constexpr double kSqrtHalfPi = 1.2533141373155003;
constexpr double kSeriesMaxS = 0.5;

#if defined(__CUDACC__)
DHJ_HD double erfcx_(double z) { return ::erfcx(z); }
#else
double erfcx_(double z);   // provided by the host emulation
#endif

// e^{-(h^2 + t^2)/2}
DHJ_HD double gauss2(double h, double t) { return exp(-0.5 * fma(h, h, t * t)); }

// db/ds = e^{-(h^2 + t^2)/2} / sqrt(2 pi) at h = x/s, t = s/2: the normalised vega the solver steps with
DHJ_HD double vega_norm(double x, double s) { return kInvSqrt2Pi * gauss2(x / s, 0.5 * s); }

// b(x, s) for s < kSeriesMaxS (h = x/s <= 0, t = s/2)
DHJ_HD double b_series(double h, double t) {
  if (h * h > 1500.0) return 0.0;   // e^{-h^2/2} underflows (and M_k would overflow)
  const double m0 = kSqrtHalfPi * erfcx_(-h * kInvSqrt2);
  double m_prev = m0, m = fma(h, m0, 1.0);   // M_{k-1}, M_k at k = 1
  const double t2 = t * t;
  double coef = t, sum = m * t;              // coef = t^k / k!
#pragma unroll
  for (int k = 1; k < 17; k += 2) {
    const double m1 = fma(h, m, (double)k * m_prev);
    const double m2 = fma(h, m1, (double)(k + 1) * m);
    m_prev = m1; m = m2;
    coef = coef * (t2 / ((double)(k + 1) * (double)(k + 2)));
    sum = fma(m, coef, sum);
  }
  return 2.0 * kInvSqrt2Pi * gauss2(h, t) * sum;
}

// normalised out-of-the-money call price b(x, s), x <= 0, s > 0
DHJ_HD double b_norm(double x, double s) {
  const double h = x / s, t = 0.5 * s;
  if (s < kSeriesMaxS) return b_series(h, t);
  if (h + t < 5.0) return 0.5 * gauss2(h, t) * (erfcx_(-(h + t) * kInvSqrt2) - erfcx_((t - h) * kInvSqrt2));
  return 0.5 * (exp(0.5 * x) * erfc(-(h + t) * kInvSqrt2) - gauss2(h, t) * erfcx_((t - h) * kInvSqrt2));
}

// e^{x/2} - b(x, s) = e^{x/2} Phi(-h-t) + e^{-x/2} Phi(h-t), for h + t >= 0
DHJ_HD double b_complement(double h, double t) {
  return 0.5 * gauss2(h, t) * (erfcx_((h + t) * kInvSqrt2) + erfcx_((t - h) * kInvSqrt2));
}

// s with b(x, s) = beta, for x <= 0 and 0 < beta < e^{x/2}.  *iters: evaluations used; *converged: 0 at the cap
// (the last iterate is returned).
DHJ_HD double solve_s(double x, double beta, int* iters, int* converged) {
  const double u = exp(0.5 * x);
  const double sc = sqrt(-2.0 * x);       // inflection point: b convex below, concave above
  // b(x, s) <= b(0, s) <= s / sqrt(2 pi): a lower bound of the root
  const double s_min = kSqrt2Pi * beta;
  const bool complement = beta > 0.5 * u;
  const double target = complement ? u - beta : beta;   // exact (Sterbenz) on the complement branch
  double lo, hi = INFINITY, s;
  bool lower = false;
  if (!complement && sc > 0.0 && beta < b_norm(x, sc)) {
    lower = true; lo = s_min; hi = sc; s = sc;
  } else {
    lo = fmax(sc, s_min); s = lo;         // upper branch: monotone from the left
  }
  *converged = 1;
  double d_prev = INFINITY;
  for (int it = 1; it <= kMaxIter; ++it) {
    *iters = it;
    const double h = x / s, t = 0.5 * s;
    const double vega = kInvSqrt2Pi * gauss2(h, t);          // db/ds
    const double curv = x * x / (s * s * s) - 0.25 * s;      // (d2b/ds2) / (db/ds)
    double g, gp, k;                                          // objective, its slope, g''/g'
    if (complement) {
      const double c = b_complement(h, t);
      g = log(c / target); gp = -vega / c; k = curv + vega / c;
    } else {
      const double b = b_norm(x, s);
      g = log(b / target); gp = vega / b; k = curv - vega / b;
    }
    if (g == 0.0) return s;
    if ((g < 0.0) != complement) lo = s; else hi = s;
    double sn;
    if (lower) {
      // in w = 1/s^2, where ln b ~ -x^2 w / 2 is nearly linear (in s, Newton from the left only grows s by ~1.5x
      // per step); ln b is convex and decreasing in w, so from s_c the iteration is monotone
      const double w = 1.0 / (s * s);
      const double gw = -0.5 * gp * s * s * s;                // dg/dw
      const double kw = -0.5 * s * s * fma(k, s, 3.0);        // (d2g/dw2) / (dg/dw)
      const double n = g / gw;
      double den = fma(-0.5 * n, kw, 1.0);
      if (!(den >= 0.5)) den = 1.0;
      const double wn = w - n / den;
      sn = (wn > 0.0) ? 1.0 / sqrt(wn) : INFINITY;
    } else {
      const double n = g / gp;
      double den = fma(-0.5 * n, k, 1.0);
      if (!(den >= 0.5)) den = 1.0;                           // Newton where Halley's correction is large
      sn = s - n / den;
    }
    // residual at rounding level and the step no longer shrinking: the evaluation's noise floor
    if (fabs(g) < 1e-10 && fabs(sn - s) > 0.5 * d_prev) return s;
    if (fabs(sn - s) <= 2.0 * kEps * s) return sn;
    if (!(sn > lo && sn < hi)) sn = (hi < INFINITY) ? sqrt(lo) * sqrt(hi) : 2.0 * s;
    d_prev = fabs(sn - s);
    s = sn;
  }
  *converged = 0;
  return s;
}

DHJ_HD bool valid_inputs(double S0, double K, double T, double r, double q) {
  return S0 > 0.0 && S0 < INFINITY && K > 0.0 && K < INFINITY && T > 0.0 && T < INFINITY && isfinite(r) &&
         isfinite(q);
}

// x = ln(F/K) = ln(S0/K) + (r - q) T with the rounding errors of S0/K, r - q and (r - q) T carried as corrections:
// an absolute error in x of eps/2 alone (the rounding of S0/K near 1) moves a short-dated near-the-money vol by
// hundreds of eps relative
DHJ_HD double log_moneyness(double S0, double K, double T, double r, double q) {
  const double k0 = S0 / K;
  const double k_rem = fma(-k0, K, S0);                   // S0 = k0 K + k_rem exactly
  const double d = r - q;
  const double dv = d - r;
  const double d_err = (r - (d - dv)) + (-q - dv);        // r - q = d + d_err exactly (two-sum)
  const double p = d * T;
  const double p_err = fma(d, T, -p);                     // d T = p + p_err exactly
  return (log(k0) + p) + (k_rem / S0 + fma(d_err, T, p_err));
}

// Black–Scholes implied volatility of price V; *status as in include/dhj.h, *iters: solver evaluations.
// vega (optional): dV/dsigma at the returned sigma, D sqrt(FK) sqrt(T) vega_norm(x_o, s) from the solver's own x_o
// and s (0 where sigma = 0, NaN where there is no sigma).
DHJ_HD double implied_vol(double V, double S0, double K, double T, double r, double q, bool call, int* status,
                          int* iters, double* vega = nullptr) {
  *iters = 0;
  if (vega) *vega = NAN;
  if (!isfinite(V) || !valid_inputs(S0, K, T, r, q)) { *status = kInvalid; return NAN; }
  const double Sq = S0 * exp(-q * T), KD = K * exp(-r * T);
  const double lower = call ? fmax(Sq - KD, 0.0) : fmax(KD - Sq, 0.0);
  const double upper = call ? Sq : KD;
  if (V < lower) { *status = kBelowLower; return NAN; }
  if (V >= upper) { *status = kAboveUpper; return NAN; }
  *status = kOk;
  if (vega) *vega = 0.0;
  if (V == lower) return 0.0;
  const double x = log_moneyness(S0, K, T, r, q);
  const double beta = V / (sqrt(Sq) * sqrt(KD));
  const double iota = ((call ? x : -x) > 0.0) ? 2.0 * sinh(0.5 * fabs(x)) : 0.0;
  const double beta_o = beta - iota, x_o = -fabs(x);
  if (!(beta_o > 0.0)) return 0.0;                          // within rounding of the intrinsic value
  if (!(beta_o < exp(0.5 * x_o))) { *status = kAboveUpper; if (vega) *vega = NAN; return NAN; }
  int converged;
  const double s = solve_s(x_o, beta_o, iters, &converged);
  if (!converged) *status = kNotConverged;
  if (vega) *vega = (sqrt(Sq) * sqrt(KD)) * sqrt(T) * vega_norm(x_o, s);
  return s / sqrt(T);
}

// Black–Scholes price of vol sigma (NaN for invalid inputs or sigma < 0 / NaN)
DHJ_HD double bs_price(double sigma, double S0, double K, double T, double r, double q, bool call) {
  if (!valid_inputs(S0, K, T, r, q) || !(sigma >= 0.0)) return NAN;
  const double Sq = S0 * exp(-q * T), KD = K * exp(-r * T);
  if (sigma == 0.0) return call ? fmax(Sq - KD, 0.0) : fmax(KD - Sq, 0.0);
  const double s = sigma * sqrt(T);
  if (!(s < INFINITY)) return call ? Sq : KD;
  const double x = log_moneyness(S0, K, T, r, q);
  const double iota = ((call ? x : -x) > 0.0) ? 2.0 * sinh(0.5 * fabs(x)) : 0.0;
  return sqrt(Sq) * sqrt(KD) * (b_norm(-fabs(x), s) + iota);
}

#if defined(__CUDACC__)
// Option-list layout of dhj_price_list: in/out [P][M], S0 stride 0 or 1, strike stride 0 or M (scale_by_spot:
// K = strike * S0 / 100), maturity[M], is_call[M]; all device pointers.  status may be null.
struct IvArgs {
  const double* in;
  const double* S0;
  long long s0_stride;
  const double* strike;
  long long strike_stride;
  int scale_by_spot;
  const double* maturity;
  const int32_t* is_call;
  double r, q;
  long long P;
  int M;
  double* out;
  int32_t* status;
};

__device__ __forceinline__ void iv_option(const IvArgs& a, long long i, double* S0, double* K, double* T, bool* call) {
  const long long p = i / a.M;
  const int j = (int)(i - p * a.M);
  *S0 = a.S0[p * a.s0_stride];
  *K = a.strike[p * a.strike_stride + j];
  if (a.scale_by_spot) *K = *K * *S0 / 100.0;
  *T = a.maturity[j];
  *call = a.is_call[j] != 0;
}

__global__ void __launch_bounds__(256) k_implied_vol(IvArgs a) {
  const long long n = a.P * (long long)a.M;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    double S0, K, T;
    bool call;
    iv_option(a, i, &S0, &K, &T, &call);
    int st, iters;
    a.out[i] = implied_vol(a.in[i], S0, K, T, a.r, a.q, call, &st, &iters);
    if (a.status) a.status[i] = st;
  }
}

__global__ void __launch_bounds__(256) k_bs_price(IvArgs a) {
  const long long n = a.P * (long long)a.M;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    double S0, K, T;
    bool call;
    iv_option(a, i, &S0, &K, &T, &call);
    a.out[i] = bs_price(a.in[i], S0, K, T, a.r, a.q, call);
  }
}
#endif

}  // namespace iv
}  // namespace dhj
