// dhj_greeks.cuh — prices and their Greeks (delta, gamma, theta, rho, dividend rho) on an option list.
//
// All five are exact derivatives of the COS price with the truncation range [a, b] held at its value for the current
// inputs (the convention of the price Jacobian, dhj_jac.cuh).  [a, b] is a range of the log-return and does not
// depend on S0, except through the +-0.1 widening of a binding strike.
//
//   delta, gamma:  S0 enters only through the payoff integral over [x, b] (call) or [a, x] (put), x = log(K/S0), whose
//                  integrand (S0 e^y - K) cos(u (y - a)) is 0 at y = x.  So, with the rotation form of dhj_math.cuh
//                  (P_k, Q_k, A1, A3 of strike_const_part) and theta = pi (x - a)/(b - a):
//                    delta = disc ([call] A1 | [put] e^a A3  -  e^x sum_k (P_k cos k theta + Q_k sin k theta))
//                    gamma = disc (K / S0^2) tw sum_k G_k cos k theta                 (calls and puts alike)
//   theta, rho:    G_T = w_k Re(dX/dT e^{X - iua}), G_r = w_k Re(dX/dr e^{X - iua}) (cf_exponent_time) contracted like
//                  G; the discount exp(-r T) adds -T V to dV/dr and -r V to dV/dT:
//                    theta = -(disc C(G_T) - r V),  rho = disc C(G_r) - T V,  rho_q = -disc C(G_r) = -(rho + T V)
//
// k_price_greeks is k_price_jac's item loop and pass (chan_items / chan_pass) with 3 staged channels (G, G_T, G_r) and
// 5 accumulators per strike: G V, G_T V, G_r V, G (P' cos + Q' sin) and G cos, V the payoff basis value of
// dhj_jac.cuh.  With 5 accumulators instead of 14 a chunk holds kGreeksChunk = 224 strikes: a slice of up to 224
// strikes needs one CF evaluation per k.
#pragma once
#include "dhj_jac.cuh"

namespace dhj {

constexpr int kGreeks = 5;          // delta, gamma, theta, rho, rho_q (DHJ_N_GREEKS)
constexpr int kGreeksChunk = 224;

struct GreeksArgs {
  const double* params;      // [P][13] model parameters
  const double* S0;          // spot table
  long long s0_stride;       // 0 = scalar
  const int* row_index;      // optional [P]: row of S0 / strike tables used by set p (default p)
  long long P;
  double* out_price;         // [P][M]
  double* out_greeks;        // [P][M][5]
};

struct GreeksChannels {
  static constexpr int kTangents = 2, kStaged = 3, kAcc = 5, kChunk = kGreeksChunk;
  using Args = GreeksArgs;
  static __device__ __forceinline__ void exponent(const Params&, const SetConsts& s, double u, double T,
                                                  const fm::Tables* __restrict__ ltab, double* xr, double* xi,
                                                  Cplx* dX) {
    cf_exponent_time(s, u, T, ltab, xr, xi, dX);
  }
  // acc: C(G), C(G_T), C(G_r), sum G (P' cos + Q' sin), sum G cos
  template <class W>
  static __device__ __forceinline__ void term(double* acc, const W& w, int i, double c0, double s0, double Kt,
                                              double sex) {
    const double pq = fma(w.fQ[i], s0, w.fP[i] * c0);
    const double V = fma(s0, Kt * w.fR[i], -(sex * pq));
    const double g = w.G[0][i];
    acc[0] = fma(g, V, acc[0]);
    acc[1] = fma(w.G[1][i], V, acc[1]);
    acc[2] = fma(w.G[2][i], V, acc[2]);
    acc[3] = fma(g, pq, acc[3]);
    acc[4] = fma(g, c0, acc[4]);
  }
  // the pass's own (a, b) enter here: afterwards acc[3] is delta / disc and acc[4] is gamma S0^2 / (K disc)
  template <class W>
  static __device__ __forceinline__ void pass_end(W& w, int t, const PassConsts& pc) {
    const bool call = w.call[t] != 0;
    for (int c = 0; c < 3; ++c)
      w.acc[t][c] += strike_const_part(call, w.S0, w.K[t], w.x[t], pc, w.A[0][c], w.A[1][c], w.A[2][c], w.g0[c]);
    w.acc[t][3] = fma(-fm::exp_(w.x[t]), w.acc[t][3], call ? w.A[0][0] : pc.ea * w.A[2][0]);
    w.acc[t][4] *= pc.tw;
  }
  template <class W>
  static __device__ __forceinline__ void write(const Args& a, long long at, const W& w, int t, double r) {
    const double V = w.disc * w.acc[t][0];
    const double T = w.pass.T;
    const double dr = w.disc * w.acc[t][2];
    double* g = a.out_greeks + at * kGreeks;
    a.out_price[at] = V;
    g[0] = w.disc * w.acc[t][3];
    g[1] = ((w.disc * w.acc[t][4]) * w.K[t]) / (w.S0 * w.S0);
    g[2] = fma(r, V, -(w.disc * w.acc[t][1]));
    g[3] = fma(-T, V, dr);
    g[4] = -dr;
  }
};

__global__ void __launch_bounds__(32 * kJacWarps) k_price_greeks(SliceView v, GreeksArgs a) {
  chan_items<GreeksChannels>(v, a);
}

}  // namespace dhj
