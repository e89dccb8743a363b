// TEST-ONLY host emulation of the Greeks arithmetic of k_price_greeks (option-pricing-ffn-lbfgs_b200/csrc/
// dhj_greeks.cuh): the same scalar functions of dhj_math.cuh (cf_exponent_time, u_of_k, strike_const_part), walked in
// the kernel's order for one option at a time — blocks of 32 k, channels G, G_T, G_r staged per block, A-sums per
// channel in k order, the strike's five accumulators by the three-term recurrence, the pass end and the epilogue of
// GreeksChannels.  Differs from the device only in libm.  Built on the fly by tests/test_greeks_cpu.py; nothing in the
// product loads it.
#include "dhj_math.cuh"

using namespace dhj;

static double u_one_h(const PassConsts& p) {
  const double q0 = kPi * p.rw;
  return fma(fma(-p.w, q0, kPi), p.rw, q0);
}

static void greeks_one(const Params& m, double S0, double K, double T, double r, double q, int is_call, int N, double L,
                       double* price, double* greeks) {
  constexpr int C = 3;
  const SetConsts s = make_set_consts(m, r, q);
  double a0, b0;
  truncation_range(m, T, r, L, &a0, &b0);
  const StrikeConsts sc = make_strike_consts(K, S0);
  const PassConsts pc = make_pass_consts(s, py_min(a0, sc.x - 0.1), py_max(b0, sc.x + 0.1), T);
  const double sex = S0 * sc.ex;
  double sth, cth;
  fm::sincos_(u_one_h(pc) * (sc.x - pc.a), &sth, &cth);
  double acc[5] = {0}, A[3][C] = {{0}}, g0[C] = {0};
  for (int k0 = 0; k0 < N; k0 += 32) {
    double G[C][32], fP[32], fQ[32], fR[32], f1[32], f2[32];
    for (int lane = 0; lane < 32; ++lane) {
      const int k = k0 + lane;
      const double u = u_of_k(pc, k);
      double xr, xi;
      Cplx dX[2];
      cf_exponent_time(s, u, T, &fm::kTables, &xr, &xi, dX);
      double sph, cph;
      fm::sincos_(fma(-u, pc.a, xi), &sph, &cph);
      const bool live = k < N;
      const double mag = fm::exp_tab(xr, &fm::kTables) * ((k == 0) ? 0.5 : 1.0);
      const double er = mag * cph, ei = mag * sph;
      G[0][lane] = live ? er : 0.0;
      for (int i = 0; i < 2; ++i) G[1 + i][lane] = live ? fma(dX[i].r, er, -(dX[i].i * ei)) : 0.0;
      const double kf = (double)k;
      const double delta = fma(-kf, kPiLo, fma(-kf, kPi, u * pc.w));
      const double sb = fm::xor_sign(delta, k << 31);
      const double t1 = fm::xor_sign(pc.eb, k << 31);
      const double t3 = (u * sb) * pc.eb;
      fP[lane] = pc.tw * fm::rcp(fma(u, u, 1.0));
      fQ[lane] = fP[lane] * u;
      fR[lane] = pc.tw * ((k == 0) ? 0.0 : fm::rcp(u));
      f1[lane] = fP[lane] * (t1 + t3);
      f2[lane] = fR[lane] * sb;
    }
    for (int c = 0; c < C; ++c) {
      for (int i = 0; i < 32; ++i) {
        A[0][c] = fma(G[c][i], f1[i], A[0][c]); A[1][c] = fma(G[c][i], f2[i], A[1][c]);
        A[2][c] = fma(G[c][i], fP[i], A[2][c]);
      }
      if (k0 == 0) g0[c] = G[c][0] * pc.tw;
    }
    double c0, s0;
    fm::sincos_(u_of_k(pc, k0) * (sc.x - pc.a), &s0, &c0);
    const double two_c = cth + cth;
    double c1 = fma(c0, cth, -(s0 * sth)), s1 = fma(s0, cth, c0 * sth);
    for (int i = 0; i < 32; ++i) {
      const double pq = fma(fQ[i], s0, fP[i] * c0);
      const double V = fma(s0, sc.K * fR[i], -(sex * pq));
      acc[0] = fma(G[0][i], V, acc[0]);
      acc[1] = fma(G[1][i], V, acc[1]);
      acc[2] = fma(G[2][i], V, acc[2]);
      acc[3] = fma(G[0][i], pq, acc[3]);
      acc[4] = fma(G[0][i], c0, acc[4]);
      const double c2 = fma(two_c, c1, -c0), s2 = fma(two_c, s1, -s0);
      c0 = c1; s0 = s1; c1 = c2; s1 = s2;
    }
  }
  const bool call = is_call != 0;
  for (int c = 0; c < C; ++c)
    acc[c] += strike_const_part(call, S0, sc.K, sc.x, pc, A[0][c], A[1][c], A[2][c], g0[c]);
  acc[3] = fma(-fm::exp_(sc.x), acc[3], call ? A[0][0] : pc.ea * A[2][0]);
  acc[4] *= pc.tw;
  const double disc = fm::exp_(-r * T);
  const double V = disc * acc[0];
  const double dr = disc * acc[2];
  *price = V;
  greeks[0] = disc * acc[3];
  greeks[1] = ((disc * acc[4]) * sc.K) / (S0 * S0);
  greeks[2] = fma(r, V, -(disc * acc[1]));
  greeks[3] = fma(-T, V, dr);
  greeks[4] = -dr;
}

extern "C" void emu_price_greeks(const double* params, const double* S0, const double* strike, const double* maturity,
                                 const int* is_call, double r, double q, long P, int M, int N, double L,
                                 double* out_price, double* out_greeks) {
  for (long p = 0; p < P; ++p) {
    const Params m = load_params(params + kNumParams * p);
    for (int o = 0; o < M; ++o)
      greeks_one(m, S0[p], strike[p * M + o], maturity[o], r, q, is_call[o], N, L, out_price + p * M + o,
                 out_greeks + (p * M + o) * 5);
  }
}
