// dhj_ivloss.cuh — the implied-volatility calibration objective (DESIGN.md §6e).
//
// For one market with options o and market implied vols sigma^_o (NaN: the quote has no implied vol and is left out):
//   f(x) = (1/M_v) sum_{o valid} (sigma_o(x) - sigma^_o)^2 + Feller(p(x)),
// sigma_o(x) the Black–Scholes implied vol (q = 0, the market's S0, K, T, r) of the COS model price V_o, M_v the
// number of valid options of the market.  The gradient in the unconstrained x follows from the implicit-function rule
// dsigma/dp = (dV/dp) / vega(sigma):
//   g = (2/M_v) sum_{o valid} (sigma_o - sigma^_o) (dV_o/dp) / vega_o  dp/dx + dFeller,
// with dV/dp k_price_jac's frozen-range Jacobian and the tail (Feller, dp/dx) of k_loss_grad_reduce.
// f is the 1e10 sentinel and g = 0 when a valid option has a model price <= 0, inf or NaN, a model-price implied-vol
// status != 0, or a vega that is not a positive normal number.
//
// The path is  k_fd_expand -> launch_price -> k_iv_residual -> k_loss_iv_reduce (f; FD g and f_all) or
// k_loss_iv_grad_reduce (analytic g).  Both reductions are one optimiser state per thread, options in slice order
// (pos[]), no atomics: a state's (f, g) depends only on its x and its market.
#pragma once
#include "dhj_iv.cuh"
#include "dhj_jac.cuh"

namespace dhj {

struct IvResidualArgs {
  const double* prices;      // [n_units][M] model prices from the pricing kernel (caller order)
  const int* row_index;      // [n_units] market of each unit
  const double* S0;          // [n_markets]
  const double* strike;      // market strikes in caller order, row stride strike_stride (0: one shared row)
  long long strike_stride;
  const double* maturity;    // [M] caller order
  const int32_t* is_call;    // [M] caller order
  const double* mvol;        // [n_markets][M] market implied vols, NaN = excluded
  double r;
  long long n_units;
  int M, n_markets;
  double* vol;               // [n_units][M] sigma_o, NaN where a valid option is bad (the sentinel rule)
  double* inv_vega;          // [n_units][M] 1 / vega_o (may be null)
  int32_t* status;           // reporting mode (non-null): every option is inverted, vol = implied_vol's sigma and
                             // status its code; inv_vega is not written
};

// The checked build (DHJ_CHECK) verifies the market row of every unit, the slice-order option index and that every
// state has at least one valid option; these kernels use no shared memory.
//
// One thread per (unit, option), like k_implied_vol.  In loss mode an excluded option (mvol NaN) is skipped and its
// outputs are not written: the reductions never read them.
__global__ void __launch_bounds__(256) k_iv_residual(IvResidualArgs a) {
  const long long n = a.n_units * (long long)a.M;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long u = i / a.M;
    const int o = (int)(i - u * a.M);
    const long long row = a.row_index[u];
    DHJ_CHECK(row >= 0 && row < a.n_markets, kChkOutputIndex);
    if (!a.status && isnan(a.mvol[row * a.M + o])) continue;
    const double V = a.prices[i];
    const double S0 = a.S0[row], K = a.strike[row * a.strike_stride + o];
    int st, iters;
    double vega;
    const double sigma = iv::implied_vol(V, S0, K, a.maturity[o], a.r, 0.0, a.is_call[o] != 0, &st, &iters, &vega);
    if (a.status) {
      a.vol[i] = sigma;
      a.status[i] = st;
      continue;
    }
    const bool bad = !(V > 0.0) || isinf(V) || st != iv::kOk || !(vega >= 2.2250738585072014e-308) || isinf(vega);
    a.vol[i] = bad ? NAN : sigma;
    if (a.inv_vega) a.inv_vega[i] = 1.0 / vega;
  }
}

// f per unit, and on the FD path (fd = 1, units = 14 stencil points per state) scipy's forward difference
// (f(x + h e_i) - f(x)) / ((x_i + h) - x_i) and f_all, as k_loss_reduce
__global__ void k_loss_iv_reduce(const double* __restrict__ vol, const double* __restrict__ pv,
                                 const int* __restrict__ row_index, const double* __restrict__ mvol,
                                 const int* __restrict__ pos, int M, long long n_x, int fd, double h,
                                 const double* __restrict__ x, double* __restrict__ f_all, double* __restrict__ fg) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_x) return;
  const int per = fd ? kFdPoints : 1;
  double f0 = 0.0;
  for (int var = 0; var < per; ++var) {
    const long long unit = c * per + var;
    const double* sv = vol + unit * M;
    const double* mv = mvol + (long long)row_index[unit] * M;
    double sq = 0.0;
    int cnt = 0;
    bool bad = false;
    for (int i = 0; i < M; ++i) {
      const int o = pos[i];
      DHJ_CHECK(o >= 0 && o < M, kChkOutputIndex);
      const double mo = mv[o];
      if (isnan(mo)) continue;
      ++cnt;
      const double s = sv[o];
      if (isnan(s)) bad = true;
      const double d = s - mo;
      sq += d * d;
    }
    DHJ_CHECK(cnt > 0, kChkOutputIndex);                 // dhj_market_set_objective refuses a market without one
    const Params m = load_params(pv + kNumParams * unit);
    const double loss = bad ? kSentinel : sq / (double)cnt + feller_penalty(m);
    f_all[unit] = loss;
    if (fd) {
      if (var == 0) { f0 = loss; fg[kFdPoints * c] = loss; }
      else {
        const double xi = x[kNumParams * c + var - 1];
        fg[kFdPoints * c + var] = (loss - f0) / ((xi + h) - xi);
      }
    }
  }
}

// f and the analytic g per state, as k_loss_grad_reduce; fg[n][14] = (f, g[13])
__global__ void k_loss_iv_grad_reduce(const double* __restrict__ vol, const double* __restrict__ inv_vega,
                                      const double* __restrict__ jac, const double* __restrict__ pv,
                                      const int* __restrict__ row_index, const double* __restrict__ mvol,
                                      const int* __restrict__ pos, int M, long long n_x, double* __restrict__ fg) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_x) return;
  const double* sv = vol + c * M;
  const double* rv = inv_vega + c * M;
  const double* jr = jac + c * (long long)M * kNumParams;
  const double* mv = mvol + (long long)row_index[c] * M;
  double sq = 0.0, gp[kNumParams];
  for (int i = 0; i < kNumParams; ++i) gp[i] = 0.0;
  int cnt = 0;
  bool bad = false;
  for (int i = 0; i < M; ++i) {
    const int o = pos[i];
    DHJ_CHECK(o >= 0 && o < M, kChkOutputIndex);
    const double mo = mv[o];
    if (isnan(mo)) continue;
    ++cnt;
    const double s = sv[o];
    if (isnan(s)) bad = true;
    const double d = s - mo;
    sq += d * d;
    const double wgt = d * rv[o];
    for (int j = 0; j < kNumParams; ++j) gp[j] = fma(wgt, jr[(long long)o * kNumParams + j], gp[j]);
  }
  DHJ_CHECK(cnt > 0, kChkOutputIndex);
  const double* p = pv + kNumParams * c;
  const Params m = load_params(p);
  double* out = fg + kFdPoints * c;
  if (bad) {
    out[0] = kSentinel;
    for (int j = 0; j < kNumParams; ++j) out[1 + j] = 0.0;
    return;
  }
  out[0] = sq / (double)cnt + feller_penalty(m);
  const double two_m = 2.0 / (double)cnt;
  for (int j = 0; j < kNumParams; ++j) gp[j] *= two_m;
  loss_grad_tail(p, m, gp, out);
}

}  // namespace dhj
