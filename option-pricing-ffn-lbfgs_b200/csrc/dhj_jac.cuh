// dhj_jac.cuh — prices and their 13 model-parameter derivatives (the price Jacobian), and the analytic gradient of
// the calibration loss built on it.
//
// With phi = exp(X) the COS price is linear in G_k = w_k Re(phi(u_k) e^{-i u_k a}); every later step (payoff
// coefficients, A-sums, strike contraction) is linear in G.  dV/dp_i is therefore the same contraction with G_k
// replaced by G^i_k = w_k Re(dX/dp_i e^{X - i u_k a}) (cf_exponent_tangents), the truncation range [a, b] held at its
// value for the current parameters ("frozen range": [a, b] depends on the parameters through the cumulants, and that
// dependence is not differentiated).  The discount factor and the payoff basis do not depend on the parameters.
//
// k_price_jac: ONE WARP PER ITEM (parameter set, maturity slice), no block barrier in the item loop.
//   * lane 0 prepares the item (set constants, truncation range, pass constants) with the same scalar functions as
//     the pricing kernels;
//   * strikes are processed in chunks of kJacChunk: their constants and 14 accumulators (price + 13 derivatives)
//     live in the warp's private shared memory;
//   * per block of 32 cosine terms lane = k forms G and the 13 G^i and leaves them, with the strike-independent
//     payoff factors P'_k = tw/(1+u^2), Q'_k = P'_k u, R'_k = tw/u, in the warp's stage (channels x 32 k);
//     lanes 0..13 then add the block's share of channel c's A-sums (A1, A2, A3 of strike_const_part) in a fixed
//     order, and each lane contracts its strikes against all 14 channels at once: the payoff basis value
//     V_k(strike) = K R'_k sin(k theta) - S0 e^x (P'_k cos(k theta) + Q'_k sin(k theta)) is formed ONCE per
//     (strike, k) by the three-term recurrence of segment_sums and multiplied into the 14 channels;
//   * strikes whose +-0.1 widening binds get their own pass with their own (a, b), exactly as in the pricing kernels.
// Every sum has a fixed order that depends on nothing but the item, so an item's outputs do not depend on the launch.
// The item loop and the pass are templates on the channel set (JacChannels here; GreeksChannels in dhj_greeks.cuh).
#pragma once
#include "dhj_kernels.cuh"

namespace dhj {

constexpr int kJacChannels = kNumParams + 1;   // channel 0: the price; 1 + i: d/dp_i
constexpr int kJacWarps = 2;
constexpr int kJacChunk = 64;

// The item loop and the pass below are shared by every kernel that contracts G and some of its tangents against the
// payoff basis (k_price_jac here, k_price_greeks in dhj_greeks.cuh).  A channel set Ch supplies:
//   kTangents       complex tangents dX of the CF exponent; channel 0 is G, channel 1 + i is w_k Re(dX_i e^{X - iua})
//   kStaged         1 + kTangents channels staged per block of 32 k (each with its own A-sums)
//   kAcc, kChunk    accumulators per strike, strikes per chunk
//   Args            the kernel's arguments (params, S0, s0_stride, row_index, P and the outputs)
//   exponent()      X and the kTangents tangents at u
//   term()          one (strike, k) step: the basis value V_k and everything else the strike accumulates
//   pass_end()      the strike's constant parts, after the pass's A-sums are complete
//   write()         the outputs of one option
template <class Ch>
struct ChanWarp {
  Params m;
  SetConsts set;
  PassConsts pass;                                 // the pass being contracted: regular, or a binding strike's own
  double S0, disc, a0, b0;
  double G[Ch::kStaged][32];                       // stage: channel c of the block's 32 terms
  double fP[32], fQ[32], fR[32], f1[32], f2[32];   // P'_k, Q'_k, R'_k, P'_k (t1+t3)_k, R'_k sin(u_k (b-a))
  double A[3][Ch::kStaged], g0[Ch::kStaged];       // A1, A2, A3 and g0 of the pass, per channel
  double K[Ch::kChunk], x[Ch::kChunk], sex[Ch::kChunk], cth[Ch::kChunk], sth[Ch::kChunk];
  double acc[Ch::kChunk][Ch::kAcc];
  unsigned char call[Ch::kChunk], bind[Ch::kChunk];
#if defined(DHJ_CHECKED)
  unsigned wtag[32], rtag[32], epoch;              // as CoefStage: per-slot write epoch, per-lane read epoch
#endif
};

template <class Ch>
struct ChanSmem {
  ChanWarp<Ch> w[kJacWarps];
  fm::Tables ltab;
};

struct JacArgs {
  const double* params;      // [P][13] model parameters
  const double* S0;          // spot table
  long long s0_stride;       // 0 = scalar
  const int* row_index;      // optional [P]: row of S0 / strike tables used by set p (default p)
  long long P;
  double* out_price;         // [P][M]
  double* out_jac;           // [P][M][13]
};

// 14 channels (the price and its 13 parameter derivatives), one accumulator each
struct JacChannels {
  static constexpr int kTangents = kNumParams, kStaged = kJacChannels, kAcc = kJacChannels, kChunk = kJacChunk;
  using Args = JacArgs;
  static __device__ __forceinline__ void exponent(const Params& m, const SetConsts& s, double u, double T,
                                                  const fm::Tables* __restrict__ ltab, double* xr, double* xi,
                                                  Cplx* dX) {
    cf_exponent_tangents(m, s, u, T, ltab, xr, xi, dX);
  }
  template <class W>
  static __device__ __forceinline__ void term(double* acc, const W& w, int i, double c0, double s0, double Kt,
                                              double sex) {
    const double V = fma(s0, fma(Kt, w.fR[i], -(sex * w.fQ[i])), -(sex * (w.fP[i] * c0)));
#pragma unroll
    for (int c = 0; c < kJacChannels; ++c) acc[c] = fma(w.G[c][i], V, acc[c]);
  }
  template <class W>
  static __device__ __forceinline__ void pass_end(W& w, int t, const PassConsts& pc) {
    for (int c = 0; c < kJacChannels; ++c)
      w.acc[t][c] += strike_const_part(w.call[t] != 0, w.S0, w.K[t], w.x[t], pc, w.A[0][c], w.A[1][c], w.A[2][c],
                                       w.g0[c]);
  }
  template <class W>
  static __device__ __forceinline__ void write(const Args& a, long long at, const W& w, int t, double /*r*/) {
    a.out_price[at] = w.disc * w.acc[t][0];
    for (int i = 0; i < kNumParams; ++i) a.out_jac[at * kNumParams + i] = w.disc * w.acc[t][1 + i];
  }
};

// lane 0 prepares the item; the other lanes wait at the caller's __syncwarp
template <class Ch>
__device__ __forceinline__ void chan_prepare(ChanWarp<Ch>& W, const SliceView& v, const double* __restrict__ pp,
                                             double S0, double T) {
  W.m = load_params(pp);
  W.set = make_set_consts(W.m, v.r, v.q);
  double a0, b0;
  truncation_range(W.m, T, v.r, v.L, &a0, &b0);
  W.a0 = a0; W.b0 = b0;
  W.pass = make_pass_consts(W.set, a0, b0, T);
  W.S0 = S0;
  W.disc = fm::exp_(-v.r * T);
}

// One pass over n_cos terms with W.pass: every strike of the chunk with !bind (only < 0), or strike `only`.
template <class Ch>
__device__ __forceinline__ void chan_pass(ChanWarp<Ch>& W, int cnt, int only, int n_cos, int lane,
                                          const fm::Tables* __restrict__ ltab) {
  const PassConsts pc = W.pass;
  const double u1 = u_one(pc);
  for (int t = lane; t < cnt; t += 32) {
    if (only < 0 ? W.bind[t] != 0 : t != only) continue;
    fm::sincos_(u1 * (W.x[t] - pc.a), &W.sth[t], &W.cth[t]);
  }
  if (lane < Ch::kStaged) { W.A[0][lane] = 0.0; W.A[1][lane] = 0.0; W.A[2][lane] = 0.0; }
#pragma unroll 1
  for (int k0 = 0; k0 < n_cos; k0 += 32) {
    // ---- lane = k: G and its tangent channels -> stage ----
    const int k = k0 + lane;
    const double u = u_of_k(pc, k);
    double xr, xi;
    Cplx dX[Ch::kTangents];
    Ch::exponent(W.m, W.set, u, pc.T, ltab, &xr, &xi, dX);
    double sph, cph;
    fm::sincos_(fma(-u, pc.a, xi), &sph, &cph);
    const bool live = k < n_cos;                         // ragged last block: every channel is 0
    const double mag = fm::exp_tab(xr, ltab) * ((k == 0) ? 0.5 : 1.0);
    const double er = mag * cph, ei = mag * sph;          // w_k e^{X - iua}
    const KTerm kt = [&] {                               // payoff factors of make_kterm_f (its G is not needed)
      KTerm t;
      t.u = u;
      const double kf = (double)k;
      const double delta = fma(-kf, kPiLo, fma(-kf, kPi, u * pc.w));
      t.sb = fm::xor_sign(delta, k << 31);
      t.t1 = fm::xor_sign(pc.eb, k << 31);
      t.t3 = (u * t.sb) * pc.eb;
      t.inv1 = fm::rcp(fma(u, u, 1.0));
      t.invu = (k == 0) ? 0.0 : fm::rcp(u);
      return t;
    }();
    __syncwarp();                                        // the previous block's stage has been consumed
#if defined(DHJ_CHECKED)
    const unsigned epoch = W.epoch + 1;
    for (int l = 0; l < 32; ++l) DHJ_CHECK(W.rtag[l] == epoch - 1, kChkWriteBeforeConsumed);
    __syncwarp();
    W.wtag[lane] = epoch;
    if (lane == 0) W.epoch = epoch;
#endif
    W.G[0][lane] = live ? er : 0.0;
#pragma unroll
    for (int i = 0; i < Ch::kTangents; ++i) W.G[1 + i][lane] = live ? fma(dX[i].r, er, -(dX[i].i * ei)) : 0.0;
    W.fP[lane] = pc.tw * kt.inv1;
    W.fQ[lane] = W.fP[lane] * u;
    W.fR[lane] = pc.tw * kt.invu;
    W.f1[lane] = W.fP[lane] * (kt.t1 + kt.t3);
    W.f2[lane] = W.fR[lane] * kt.sb;
    __syncwarp();
#if defined(DHJ_CHECKED)
    for (int l = 0; l < 32; ++l) DHJ_CHECK(W.wtag[l] == epoch, kChkReadBeforeWrite);
#endif
    // ---- strike-independent sums of channel `lane`, k in order ----
    if (lane < Ch::kStaged) {
      double s1 = W.A[0][lane], s2 = W.A[1][lane], s3 = W.A[2][lane];
      for (int i = 0; i < 32; ++i) {
        const double gc = W.G[lane][i];
        s1 = fma(gc, W.f1[i], s1); s2 = fma(gc, W.f2[i], s2); s3 = fma(gc, W.fP[i], s3);
      }
      W.A[0][lane] = s1; W.A[1][lane] = s2; W.A[2][lane] = s3;
      if (k0 == 0) W.g0[lane] = W.G[lane][0] * pc.tw;
    }
    // ---- strikes: one basis value per (strike, k) into every accumulator ----
    const double u0 = u_of_k(pc, k0);
    for (int t = lane; t < cnt; t += 32) {
      if (only < 0 ? W.bind[t] != 0 : t != only) continue;
      DHJ_CHECK(t < Ch::kChunk, kChkSharedIndex);
      double acc[Ch::kAcc];
#pragma unroll
      for (int c = 0; c < Ch::kAcc; ++c) acc[c] = W.acc[t][c];
      double c0, s0;
      fm::sincos_(u0 * (W.x[t] - pc.a), &s0, &c0);
      const double cth = W.cth[t], sth = W.sth[t], two_c = cth + cth;
      const double Kt = W.K[t], sex = W.sex[t];
      double c1 = fma(c0, cth, -(s0 * sth)), s1 = fma(s0, cth, c0 * sth);
#pragma unroll 4
      for (int i = 0; i < 32; ++i) {
        Ch::term(acc, W, i, c0, s0, Kt, sex);
        const double c2 = fma(two_c, c1, -c0), s2 = fma(two_c, s1, -s0);
        c0 = c1; s0 = s1; c1 = c2; s1 = s2;
      }
#pragma unroll
      for (int c = 0; c < Ch::kAcc; ++c) W.acc[t][c] = acc[c];
    }
#if defined(DHJ_CHECKED)
    W.rtag[lane] = W.epoch;
#endif
  }
  __syncwarp();                                          // A-sums complete
  for (int t = lane; t < cnt; t += 32) {
    if (only < 0 ? W.bind[t] != 0 : t != only) continue;
    Ch::pass_end(W, t, pc);
  }
  __syncwarp();
}

// The item loop: one warp per (parameter set, maturity slice) item, strikes in chunks of Ch::kChunk.
template <class Ch>
__device__ __forceinline__ void chan_items(const SliceView& v, const typename Ch::Args& a) {
  __shared__ ChanSmem<Ch> sm;
  const int tid = threadIdx.x;
  // (load_log_table assumes >= 65 threads: the block has 64, so the tables are copied in a strided loop)
  for (int i = tid; i < 65; i += 32 * kJacWarps) {
    if (i < 64) { sm.ltab.log[i] = fm::kTables.log[i]; sm.ltab.exp2[i] = fm::kTables.exp2[i]; }
    sm.ltab.atan64[i] = fm::kTables.atan64[i];
  }
#if defined(DHJ_CHECKED)
  sm.w[tid >> 5].wtag[tid & 31] = 0u; sm.w[tid >> 5].rtag[tid & 31] = 0u;
  if ((tid & 31) == 0) sm.w[tid >> 5].epoch = 0u;
#endif
  __syncthreads();
  const int warp = __shfl_sync(kFullMask, tid >> 5, 0), lane = tid & 31;
  ChanWarp<Ch>& W = sm.w[warp];
  const long long n_items = a.P * (long long)v.n_slices;
  for (long long item = (long long)blockIdx.x * kJacWarps + warp; item < n_items;
       item += (long long)gridDim.x * kJacWarps) {
    const long long p = item / v.n_slices;
    const int s = (int)(item - p * v.n_slices);
    const long long row = a.row_index ? (long long)a.row_index[p] : p;
    const double* strike_row = v.strike + row * v.strike_stride;
    const int o_lo = v.slice_off[s], o_hi = v.slice_off[s + 1];
    __syncwarp();                                        // the previous item has left the warp's shared memory
    if (lane == 0) chan_prepare(W, v, a.params + kNumParams * p, a.S0[row * a.s0_stride], v.slice_T[s]);
    __syncwarp();
    const PassConsts regular = W.pass;
    for (int c_lo = o_lo; c_lo < o_hi; c_lo += Ch::kChunk) {
      const int cnt = min(Ch::kChunk, o_hi - c_lo);
      int n_bind = 0;
      for (int t0 = 0; t0 < cnt; t0 += 32) {             // warp-uniform trip count (the ballot needs every lane)
        const int t = t0 + lane;
        bool bind = false;
        if (t < cnt) {
          double K = strike_row[v.pos[c_lo + t]];
          if (v.scale_by_spot) K = K * W.S0 / 100.0;
          const StrikeConsts sc = make_strike_consts(K, W.S0);
          W.K[t] = sc.K; W.x[t] = sc.x; W.sex[t] = W.S0 * sc.ex;
          bind = ((sc.x - 0.1) < W.a0) || ((sc.x + 0.1) > W.b0);
          W.bind[t] = bind; W.call[t] = v.call[c_lo + t];
          for (int c = 0; c < Ch::kAcc; ++c) W.acc[t][c] = 0.0;
        }
        n_bind += __popc(__ballot_sync(kFullMask, bind));
      }
      __syncwarp();
      if (n_bind < cnt) {
        if (lane == 0) W.pass = regular;
        __syncwarp();
        chan_pass(W, cnt, -1, v.n_cos, lane, &sm.ltab);
      }
      if (n_bind > 0) {
        for (int t = 0; t < cnt; ++t) {
          if (!W.bind[t]) continue;                      // uniform: the flags live in shared memory
          __syncwarp();
          if (lane == 0) W.pass = make_pass_consts(W.set, py_min(W.a0, W.x[t] - 0.1), py_max(W.b0, W.x[t] + 0.1),
                                                   regular.T);
          __syncwarp();
          chan_pass(W, cnt, t, v.n_cos, lane, &sm.ltab);
        }
      }
      for (int t = lane; t < cnt; t += 32) {
        const int o = v.pos[c_lo + t];
        const long long at = p * (long long)v.n_options + o;
        DHJ_CHECK(o >= 0 && o < v.n_options && at < a.P * (long long)v.n_options && t < Ch::kChunk, kChkOutputIndex);
        Ch::write(a, at, W, t, v.r);
      }
      __syncwarp();
    }
  }
}

__global__ void __launch_bounds__(32 * kJacWarps) k_price_jac(SliceView v, JacArgs a) { chan_items<JacChannels>(v, a); }

// Loss and its analytic gradient in the unconstrained x, one optimiser state per thread, options in slice order as
// k_loss_reduce visits them; `prices` come from the pricing kernel (f has the bits of the loss path), `jac` from
// k_price_jac:
//   f = mean(rel^2) + Feller,  rel_o = (V_o - m_o) / m_o
//   df/dp = (2/M) sum_o (rel_o / m_o) dV_o/dp + dFeller/dp,  Feller term 1000 (2 sigma dsigma - 2 theta dkappa
//   - 2 kappa dtheta) where the excess sigma^2 - 2 kappa theta is > 0, else 0 (0 at the kink);
//   dp/dx = p for the exp parameters, 1 - rho^2 for the two tanh parameters, 1 for mu_j.
// Where the loss is the 1e10 sentinel (a price NaN, inf or <= 0) the gradient is 0.  fg[n][14] = (f, g[13]).
//
// loss_grad_tail is the part every analytic-gradient reduction shares (k_loss_grad_reduce here, k_loss_iv_grad_reduce
// in dhj_ivloss.cuh): gp[13] holds d(data term)/dp; the Feller derivative is added and out[1 + j] = gp_j dp_j/dx_j.
__device__ __forceinline__ void loss_grad_tail(const double* __restrict__ p, const Params& m, double* gp,
                                               double* __restrict__ out) {
  for (int f = 0; f < 2; ++f) {
    const double e = m.sigma[f] * m.sigma[f] - 2.0 * m.kappa[f] * m.theta[f];
    if (e > 0.0) {
      gp[5 * f + 3] += 2000.0 * m.sigma[f];
      gp[5 * f + 1] -= 2000.0 * m.theta[f];
      gp[5 * f + 2] -= 2000.0 * m.kappa[f];
    }
  }
  for (int j = 0; j < kNumParams; ++j) {
    const double dpdx = (j == 4 || j == 9) ? 1.0 - p[j] * p[j] : ((j == 11) ? 1.0 : p[j]);
    out[1 + j] = gp[j] * dpdx;
  }
}

__global__ void k_loss_grad_reduce(const double* __restrict__ prices, const double* __restrict__ jac,
                                   const double* __restrict__ pv, const int* __restrict__ row_index,
                                   const double* __restrict__ market, const int* __restrict__ pos, int M, long long n_x,
                                   double* __restrict__ fg) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_x) return;
  const double* pr = prices + c * M;
  const double* jr = jac + c * (long long)M * kNumParams;
  const double* mk = market + (long long)row_index[c] * M;
  double sq = 0.0, gp[kNumParams];
  for (int i = 0; i < kNumParams; ++i) gp[i] = 0.0;
  bool bad = false;
  for (int i = 0; i < M; ++i) {
    const int o = pos[i];
    const double price = pr[o];
    if (!(price > 0.0) || isinf(price)) bad = true;
    const double rel = (price - mk[o]) / mk[o];
    sq += rel * rel;
    const double wgt = rel / mk[o];
    for (int j = 0; j < kNumParams; ++j) gp[j] = fma(wgt, jr[(long long)o * kNumParams + j], gp[j]);
  }
  const double* p = pv + kNumParams * c;
  const Params m = load_params(p);
  double* out = fg + kFdPoints * c;
  if (bad) {
    out[0] = kSentinel;
    for (int j = 0; j < kNumParams; ++j) out[1 + j] = 0.0;
    return;
  }
  out[0] = sq / (double)M + feller_penalty(m);
  const double two_m = 2.0 / (double)M;
  for (int j = 0; j < kNumParams; ++j) gp[j] *= two_m;
  loss_grad_tail(p, m, gp, out);
}

}  // namespace dhj
