// dhj_math.cuh — per-thread FP64 arithmetic of the COS pricer for the Double-Heston + Merton-jump model.
//
// Everything here is scalar code for ONE cosine index k of ONE (parameter set, maturity) pass, plus the
// segment sums of the strike contraction; the thread / warp / block organisation lives in dhj_batch.cuh
// (few strikes per maturity) and dhj_dense.cuh (many).
// The functions restate the formulas of the reference in float64:
//     truncation range   /root/reference/src/models/double_heston.py:100-139
//     characteristic fn  /root/reference/src/models/double_heston.py:48-97
//     payoff coefficients /root/reference/src/models/double_heston.py:141-158, 172-190
// The truncation range, u_k, the csqrt formula and the loss follow the reference's operation order;
// elsewhere the algebra is simplified (no g = (beta-d)/(beta+d); the three outer complex exponentials
// and e^{-iua} merged into one exp and one cos; strikes contracted by recurrences in k) and products and
// sums are fused.  DESIGN.md §4 lists every deviation and its measured effect.
//
// The file compiles with nvcc (device) and with g++ (tests/host_emu: a test-only emulation that
// lets the CPU test-suite check this arithmetic against the golden fixtures without a GPU; the
// product never runs it).  Build with FMA contraction OFF (-fmad=false / -ffp-contract=off):
// fused operations are written explicitly with fma() where wanted.  Elementary functions come from
// dhj_fastmath.cuh (branch-free, <= 1-2 ulp), not from libdevice.
#pragma once
#include <math.h>
#include <stdint.h>

#include "dhj_fastmath.cuh"

#if defined(__CUDACC__)
#define DHJ_HD __device__ __forceinline__
#else
#define DHJ_HD inline
#endif

namespace dhj {

constexpr int kNumParams = 13;
constexpr double kPi = 3.141592653589793;      // == numpy.pi
constexpr double kPiLo = 1.2246467991473532e-16; // pi - kPi

// 13 model parameters in calibrator x-vector order (lbfgs_calibrator.py:53-57)
struct Params {
  double v0[2], kappa[2], theta[2], sigma[2], rho[2];
  double lam, mu, sj;
};

DHJ_HD Params load_params(const double* __restrict__ p) {
  Params m;
  m.v0[0] = p[0]; m.kappa[0] = p[1]; m.theta[0] = p[2]; m.sigma[0] = p[3]; m.rho[0] = p[4];
  m.v0[1] = p[5]; m.kappa[1] = p[6]; m.theta[1] = p[7]; m.sigma[1] = p[8]; m.rho[1] = p[9];
  m.lam = p[10]; m.mu = p[11]; m.sj = p[12];
  return m;
}

// exp/tanh transform of the calibrator (lbfgs_calibrator.py:62-87)
DHJ_HD Params transform_params(const double* __restrict__ x) {
  Params m;
  // exp for the ten positive parameters in one rolled loop (one copy of the code), tanh from libm
  // (two calls per loss evaluation; accuracy near 0 matters more than speed here)
  double e[kNumParams];
#pragma unroll 1
  for (int i = 0; i < kNumParams; ++i) e[i] = fm::exp_(x[i]);
  m.v0[0] = e[0]; m.kappa[0] = e[1]; m.theta[0] = e[2]; m.sigma[0] = e[3];
  m.rho[0] = tanh(x[4]);
  m.v0[1] = e[5]; m.kappa[1] = e[6]; m.theta[1] = e[7]; m.sigma[1] = e[8];
  m.rho[1] = tanh(x[9]);
  m.lam = e[10]; m.mu = x[11]; m.sj = e[12];
  return m;
}

// 1000*(max(0, s1^2-2 k1 t1) + max(0, s2^2-2 k2 t2)); Python max(0, e) is `e if e > 0 else 0`
// so a NaN excess contributes 0 (lbfgs_calibrator.py:111-116)
DHJ_HD double feller_penalty(const Params& m) {
  double e1 = m.sigma[0] * m.sigma[0] - 2.0 * m.kappa[0] * m.theta[0];
  double e2 = m.sigma[1] * m.sigma[1] - 2.0 * m.kappa[1] * m.theta[1];
  double p1 = (e1 > 0.0) ? e1 : 0.0;
  double p2 = (e2 > 0.0) ? e2 : 0.0;
  return 1000.0 * (p1 + p2);
}

// quantities that depend on the parameter set (and r, q) only
struct SetConsts {
  double kappa[2], kk[2];      // kappa, kappa^2
  double two_kappa[2];
  double rs[2];                // rho*sigma
  double s2[2];                // sigma^2
  double v0[2];                // v0
  double c[2];                 // kappa*theta/sigma^2
  double drift;                // r - q - lam*(exp(mu + sj^2/2) - 1)       double_heston.py:82-83
  double lam, mu, hsj2;        // hsj2 = 0.5*sj^2
};

// factor j's share of SetConsts, and the jump / drift share: the batch kernel computes them in different lanes
DHJ_HD void set_consts_factor(const Params& m, int j, SetConsts& s) {
  s.kappa[j] = m.kappa[j];
  s.kk[j] = m.kappa[j] * m.kappa[j];
  s.rs[j] = m.rho[j] * m.sigma[j];
  s.s2[j] = m.sigma[j] * m.sigma[j];
  s.two_kappa[j] = m.kappa[j] + m.kappa[j];
  s.v0[j] = m.v0[j];
  s.c[j] = fm::div(m.kappa[j] * m.theta[j], s.s2[j]);
}
DHJ_HD void set_consts_jump(const Params& m, double r, double q, SetConsts& s) {
  s.hsj2 = 0.5 * (m.sj * m.sj);
  double comp = fm::exp_(m.mu + s.hsj2) - 1.0;
  s.drift = r - q - m.lam * comp;
  s.lam = m.lam; s.mu = m.mu;
}

DHJ_HD SetConsts make_set_consts(const Params& m, double r, double q) {
  SetConsts s;
  for (int j = 0; j < 2; ++j) set_consts_factor(m, j, s);
  set_consts_jump(m, r, q, s);
  return s;
}

// ---- truncation range ----------------------------------------------------------------------
// c1, c2 of one variance factor, in the reference's operation order (double_heston.py:101-119).
// Note r*tau enters once PER FACTOR and neither q nor the jump compensator appear: kept as is.
DHJ_HD void factor_cumulants(double tau, double r, double v0, double lm, double vbar, double vv, double rho,
                             double* c1, double* c2) {
  double e = fm::exp_(-lm * tau);
  double e2 = fm::exp_(-2.0 * lm * tau);
  double ome = 1.0 - e;
  *c1 = r * tau + fm::div(ome * (vbar - v0), 2.0 * lm) - vbar * tau / 2.0;
  double lm2 = lm * lm, vv2 = vv * vv;
  double t1 = vv * tau * lm * e * (v0 - vbar) * (8.0 * lm * rho - 4.0 * vv);
  double t2 = lm * rho * vv * ome * (16.0 * vbar - 8.0 * v0);
  double t3 = 2.0 * vbar * lm * tau * (-4.0 * lm * rho * vv + vv2 + 4.0 * lm2);
  double t4 = vv2 * ((vbar - 2.0 * v0) * e2 + vbar * (6.0 * e - 7.0) + 2.0 * v0);
  double t5 = 8.0 * lm2 * (v0 - vbar) * ome;
  *c2 = fm::rcp(8.0 * (lm2 * lm)) * ((((t1 + t2) + t3) + t4) + t5);
}

// a0, b0 = c1 -+ L*sqrt(|c2|) before the strike-dependent widening (double_heston.py:121-132), from the two
// factors' cumulants (c1 = 0 + c1_0 + c1_1 in the reference's order)
DHJ_HD void truncation_from_cumulants(const Params& m, double T, double L, double c1_0, double c2_0, double c1_1,
                                      double c2_1, double* a0, double* b0) {
  double c1 = 0.0, c2 = 0.0;
  c1 += c1_0; c2 += c2_0;
  c1 += c1_1; c2 += c2_1;
  c1 = c1 + m.lam * T * m.mu;
  c2 = c2 + m.lam * T * (m.sj * m.sj + m.mu * m.mu);
  double h = L * fm::sqrt_(fabs(c2));
  *a0 = c1 - h;
  *b0 = c1 + h;
}
DHJ_HD void truncation_range(const Params& m, double T, double r, double L, double* a0, double* b0) {
  double c1j[2], c2j[2];
#pragma unroll 1
  for (int j = 0; j < 2; ++j)                   // rolled: one copy of the cumulant code
    factor_cumulants(T, r, m.v0[j], m.kappa[j], m.theta[j], m.sigma[j], m.rho[j], &c1j[j], &c2j[j]);
  truncation_from_cumulants(m, T, L, c1j[0], c2j[0], c1j[1], c2j[1], a0, b0);
}

// Python `a = min(a, y)` / `b = max(b, y)` (double_heston.py:136-137): the second argument wins
// only on a strict comparison, so a NaN a/b survives and a NaN y is dropped.
DHJ_HD double py_min(double a, double y) { return (y < a) ? y : a; }
DHJ_HD double py_max(double b, double y) { return (y > b) ? y : b; }

// quantities of one COS pass = one (parameter set, maturity, [a,b]) triple
struct PassConsts {
  double a, b, w;     // a, b, b - a
  double rw;          // 1/(b-a) (seed for the correctly rounded u_k = (k pi)/(b-a))
  double tw;          // 2/(b-a)
  double T, lamT;     // maturity, lam*T
  double eb, ea;      // exp(b), exp(a)
};

DHJ_HD PassConsts make_pass_consts(const SetConsts& s, double a, double b, double T) {
  PassConsts p;
  p.a = a; p.b = b; p.w = b - a; p.rw = fm::rcp(p.w); p.tw = fm::div(2.0, p.w); p.T = T; p.lamT = s.lam * T;
  p.eb = fm::exp_(b); p.ea = fm::exp_(a);
  return p;
}

// ---- characteristic function ----------------------------------------------------------------
// One variance factor: A_j and B_j*v0_j.
//   beta = kappa - i rho sigma u ;  d = sqrt(beta^2 + sigma^2 u (u+i)) ;  E = exp(-d T)
//   m = beta - d ; pl = beta + d ; D = pl - m E          [1 - gE = D/pl ; 1 - g = 2d/pl]
//   B = (m/sigma^2) (1-E)/(1-gE) = (m/sigma^2) (1-E) pl / D
//   A = (kappa theta/sigma^2) (m T - 2 log((1-gE)/(1-g))) ,  (1-gE)/(1-g) = D/(2d)
// (double_heston.py:64-71, 85-87).  The csqrt formula follows glibc's; products and sums are fused into FMAs
// wherever possible (an FP64 instruction is the scarce resource); g itself is never formed.
// The factor's terms are ADDED to running sums with fused multiply-adds (an FP64 instruction is the scarce
// resource): aR, aI += A_j without its -2 c_j i arg(.) part, which goes to sli += c_j arg(.);
// xbr, xbi += B_j v0_j.  Scalars are folded: B_j v0_j = -(v0 u) (u + i) (1-E) conj(D) |D|^-2 (m pl = -sigma^2 u (u+i)), and
// -2 log|D/(2d)| = log(4 |z| / |D|^2) comes straight from the table-driven log (the 4 is an exponent offset).
DHJ_HD void heston_factor(const SetConsts& s, int j, double u, double T, const fm::TrigTables* __restrict__ ltab,
                          double& aR, double& aI, double& sli, double& xbr, double& xbi) {
  const double kap = s.kappa[j];
  const double bi = -(s.rs[j] * u);                 // Im beta
  const double s2u = s.s2[j] * u;
  // z = beta^2 + sigma^2 u (u+i):  Re = kappa^2 - bi^2 + s2u u,  Im = 2 kappa bi + s2u   (fused: 3 FMAs)
  const double zr = fma(s2u, u, fma(-bi, bi, s.kk[j]));
  const double zi = fma(s.two_kappa[j], bi, s2u);
  // d = csqrt(z) as glibc does it: h = |z|, t = sqrt((h + |zr|)/2), other = zi/(2t); the roles of t and
  // `other` swap when Re z < 0.  (Re z >= kappa^2 > 0 for |rho| <= 1; the other case is kept for safety.)
  // (square roots as x * rsqrt(x): <= 1 ulp instead of correctly rounded, no zero special case; z = 0 needs
  // kappa = 0 and u = 0, for which the reference divides by zero as well)
  const double n2 = fma(zr, zr, zi * zi);
  const double h = n2 * fm::rsqrt(n2);
  const double x2 = 0.5 * (h + fabs(zr));
  const double yt = fm::rsqrt(x2);
  const double t = x2 * yt;
  const double other = (0.5 * zi) * yt;
  // Re z = kappa^2 + sigma^2 u^2 (1 - rho^2) >= 0 whenever |rho| <= 1 (always, after the calibrator's tanh): the
  // other branch of glibc's formula is taken only if some lane of the warp needs it (one vote instead of four
  // selects and two sign operations per factor and k)
  double dr = t, di = other;
#if defined(__CUDA_ARCH__)
  if (__any_sync(__activemask(), fm::sign_bit(zr)))      // (sign bit: an integer test; -0.0 takes the general branch too)
#endif
  {
    const bool pos = !(zr < 0.0);
    dr = pos ? t : fabs(other);
    di = pos ? other : copysign(t, zi);
  }
  // E = exp(-d T)
  // (integer underflow test: if -dr T is NaN so is beta - d, and with it D and the factor's whole contribution)
  const double er = fm::exp_tab_neg_ix(-dr * T, ltab);
  double sn, cs;
  fm::sincos_tab(-di * T, ltab, &sn, &cs);
  const double Er = er * cs, Ei = er * sn;
  const double mr = kap - dr, mi = bi - di;         // beta - d
  const double pr = kap + dr, pi_ = bi + di;        // beta + d
  // D = pl - m*E
  const double Dr = fma(-mr, Er, fma(mi, Ei, pr));
  const double Di = fma(-mr, Ei, fma(-mi, Er, pi_));
  const double nD = fma(Dr, Dr, Di * Di);
  const double inD = fm::rcp(nD);
  // B v0 = (m pl) (1-E) conj(D) v0 / (sigma^2 |D|^2) with  m pl = beta^2 - d^2 = beta^2 - z = -sigma^2 u (u + i):
  //      = -(v0 u) * (u + i) * [(1-E) conj(D)] / |D|^2          (one complex product instead of three)
  const double ar = 1.0 - Er, ai = -Ei;
  const double Nr = fma(ar, Dr, ai * Di), Ni = fma(ai, Dr, -(ar * Di));
  const double Mr = fma(Nr, u, -Ni), Mi = fma(Ni, u, Nr);
  const double g = -((s.v0[j] * u) * inD);
  xbr = fma(Mr, g, xbr);
  xbi = fma(Mi, g, xbi);
  // A = c (m T - 2 log(D/(2d))):  -2 log|D/(2d)| = log(4 |z| / |D|^2), |d|^2 = |z| = h;  argument from D*conj(d)
  // (no NaN guard: a NaN h or 1/|D|^2 already makes B_j v0_j, hence the exponent and the price, NaN)
  const double L = fm::log_tab<false>(h * inD, ltab, 2);
  const double li = fm::atan2_tab_nz(fma(Di, dr, -(Dr * di)), fma(Dr, dr, Di * di), ltab);
  const double cT = s.c[j] * T;
  aR = fma(s.c[j], L, aR);
  aR = fma(cT, mr, aR);
  aI = fma(cT, mi, aI);
  sli = fma(s.c[j], li, sli);
}

// exponent X of cf_heston * cf_jump = exp(X) at frequency u  (double_heston.py:82-96):
//   X = ((A0 + A1) + A2) + B1 v01 + B2 v02  +  lamT (exp(i u mu - hsj2 u^2) - 1),  A0 = i (drift u) T
// The two factors are unrolled: with the table-driven elementary functions the body is small enough for the
// instruction cache, and the rolled loop's register shuffling cost more than the second copy.
// jump_trig(&cj, &sj, &ej) supplies cos / sin(u mu) and exp(-sj^2 u^2 / 2) AFTER the two Heston factors (where
// register pressure peaks): the batch kernel advances all three by recurrences from one block of k to the next
// instead of evaluating a sincos and an exp
// exp(-sigma_j^2 u^2 / 2) of the jump factor (double_heston.py:93)
DHJ_HD double jump_gauss(const SetConsts& s, double u, const fm::Tables* __restrict__ ltab) {
  return fm::exp_tab_neg(-(s.hsj2 * (u * u)), ltab);
}

template <class JumpTrig>
DHJ_HD void cf_exponent_f(const SetConsts& s, double u, double T, double lamT, const fm::TrigTables* __restrict__ ltab,
                          JumpTrig jump_trig, double* xr_out, double* xi_out) {
  double aR = 0.0, aI = (s.drift * u) * T, sli = 0.0, xbr = 0.0, xbi = 0.0;
#pragma unroll
  for (int j = 0; j < 2; ++j) heston_factor(s, j, u, T, ltab, aR, aI, sli, xbr, xbi);
  double xr = aR + xbr;
  double xi = fma(-2.0, sli, aI) + xbi;
  double cj, sj, ej;
  jump_trig(&cj, &sj, &ej);
  xr = fma(lamT, fma(ej, cj, -1.0), xr);
  xi = fma(lamT, ej * sj, xi);
  *xr_out = xr; *xi_out = xi;
}

DHJ_HD void cf_exponent(const SetConsts& s, double u, double T, double lamT, const fm::TrigTables* __restrict__ ltab,
                        double* xr_out, double* xi_out) {
  cf_exponent_f(s, u, T, lamT, ltab, [&](double* cj, double* sj, double* ej) {
    fm::sincos_(u * s.mu, sj, cj);
    *ej = jump_gauss(s, u, ltab);
  }, xr_out, xi_out);
}

// ---- parameter tangents of the CF exponent (analytic gradient, dhj_jac.cuh) ------------------------------------
// Forward-mode derivatives of X with respect to the 13 model parameters at one real u, with the truncation range
// held fixed (the price is linear in exp(X), so dV/dp_i is the COS contraction of Re(dX/dp_i e^{X - iua})).
struct Cplx { double r, i; };
DHJ_HD Cplx c_add(Cplx a, Cplx b) { return {a.r + b.r, a.i + b.i}; }
DHJ_HD Cplx c_sub(Cplx a, Cplx b) { return {a.r - b.r, a.i - b.i}; }
DHJ_HD Cplx c_mul(Cplx a, Cplx b) { return {fma(a.r, b.r, -(a.i * b.i)), fma(a.r, b.i, a.i * b.r)}; }
DHJ_HD Cplx c_scale(Cplx a, double f) { return {a.r * f, a.i * f}; }

// Factor j's value arithmetic for the tangent functions: heston_factor's operations without the warp vote (both
// branches of the csqrt are formed), the same running sums, and the intermediates the tangents need.
struct FactorState {
  double dr, di, h, Er, Ei, mr, mi, Dr, Di, inD, Mr, Mi, L, li;
};

DHJ_HD FactorState heston_factor_state(const SetConsts& s, int j, double u, double T,
                                       const fm::Tables* __restrict__ ltab, double& aR, double& aI, double& sli,
                                       double& xbr, double& xbi) {
  const double kap = s.kappa[j];
  const double bi = -(s.rs[j] * u);
  const double s2u = s.s2[j] * u;
  const double zr = fma(s2u, u, fma(-bi, bi, s.kk[j]));
  const double zi = fma(s.two_kappa[j], bi, s2u);
  const double n2 = fma(zr, zr, zi * zi);
  const double h = n2 * fm::rsqrt(n2);
  const double x2 = 0.5 * (h + fabs(zr));
  const double yt = fm::rsqrt(x2);
  const double t = x2 * yt;
  const double other = (0.5 * zi) * yt;
  const bool pos = !(zr < 0.0);
  const double dr = pos ? t : fabs(other);
  const double di = pos ? other : copysign(t, zi);
  const double er = fm::exp_tab_neg_ix(-dr * T, ltab);
  double sn, cs;
  fm::sincos_(-di * T, &sn, &cs);
  const double Er = er * cs, Ei = er * sn;
  const double mr = kap - dr, mi = bi - di;
  const double pr = kap + dr, pi_ = bi + di;
  const double Dr = fma(-mr, Er, fma(mi, Ei, pr));
  const double Di = fma(-mr, Ei, fma(-mi, Er, pi_));
  const double nD = fma(Dr, Dr, Di * Di);
  const double inD = fm::rcp(nD);
  const double ar = 1.0 - Er, ai = -Ei;
  const double Nr = fma(ar, Dr, ai * Di), Ni = fma(ai, Dr, -(ar * Di));
  const double Mr = fma(Nr, u, -Ni), Mi = fma(Ni, u, Nr);
  const double g = -((s.v0[j] * u) * inD);
  xbr = fma(Mr, g, xbr);
  xbi = fma(Mi, g, xbi);
  const double L = fm::log_tab<false>(h * inD, ltab, 2);
  const double li = fm::atan2_tab_nz(fma(Di, dr, -(Dr * di)), fma(Dr, dr, Di * di), ltab);
  const double cT = s.c[j] * T;
  aR = fma(s.c[j], L, aR);
  aR = fma(cT, mr, aR);
  aI = fma(cT, mi, aI);
  sli = fma(s.c[j], li, sli);
  return {dr, di, h, Er, Ei, mr, mi, Dr, Di, inD, Mr, Mi, L, li};
}

// Factor j: the value arithmetic of heston_factor_state plus dX/d(v0_j, kappa_j, theta_j, sigma_j, rho_j) -> dX[0..4].
// With z_p = dz/dp etc.:
//   d_p = z_p / (2d),  E_p = -T d_p E,  m_p = beta_p - d_p,  pl_p = beta_p + d_p,  D_p = pl_p - m_p E - m E_p
//   B = -u (u+i) (1-E) / D             B_p = u (u+i) (E_p + (1-E) D_p/D) / D
//   Ahat = m T - 2 log(D / (2d))       Ahat_p = m_p T - 2 (D_p/D - d_p/d)
//   A = c Ahat, c = kappa theta / sigma^2:  dX/dv0 = B,  dX/dtheta = (kappa/sigma^2) Ahat,
//   dX/dp = c_p Ahat + c Ahat_p + v0 B_p  for p = kappa (c_p = c/kappa), sigma (c_p = -2c/sigma), rho (c_p = 0)
DHJ_HD void heston_factor_tangents(const Params& mp, const SetConsts& s, int j, double u, double T,
                                   const fm::Tables* __restrict__ ltab, double& aR, double& aI, double& sli,
                                   double& xbr, double& xbi, Cplx* dX) {
  const FactorState f = heston_factor_state(s, j, u, T, ltab, aR, aI, sli, xbr, xbi);
  const double kap = s.kappa[j];
  const double bi = -(s.rs[j] * u);
  const double dr = f.dr, di = f.di, h = f.h, Er = f.Er, Ei = f.Ei, mr = f.mr, mi = f.mi, Dr = f.Dr, Di = f.Di;
  const double inD = f.inD, Mr = f.Mr, Mi = f.Mi, L = f.L, li = f.li;
  const double ar = 1.0 - Er, ai = -Ei;
  const Cplx E = {Er, Ei}, m = {mr, mi}, omE = {ar, ai};
  const Cplx uu = {u * u, u};                                  // u (u + i)
  const Cplx invD = {Dr * inD, -(Di * inD)};                   // 1/D
  const double ih = fm::rcp(h);
  const Cplx inv2d = {(0.5 * dr) * ih, -((0.5 * di) * ih)};    // 1/(2d) = conj(d) / (2|z|)
  const Cplx invd = {dr * ih, -(di * ih)};                     // 1/d
  const double mB = -u * inD;
  const Cplx B = {Mr * mB, Mi * mB};                           // B_j = (B_j v0_j) / v0_j without the division
  const Cplx Ahat = {fma(mr, T, L), fma(mi, T, -2.0 * li)};
  dX[0] = B;
  dX[2] = c_scale(Ahat, fm::div(kap, s.s2[j]));
  const double rho = mp.rho[j], sig = mp.sigma[j];
  const Cplx beta = {kap, bi};
  Cplx bp[3];                                                  // d beta / d(kappa, sigma, rho)
  bp[0] = {1.0, 0.0};
  bp[1] = {0.0, -(rho * u)};
  bp[2] = {0.0, -(sig * u)};
  const double cp[3] = {fm::div(s.c[j], kap), fm::div(-2.0 * s.c[j], sig), 0.0};
  const int slot[3] = {1, 3, 4};
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    Cplx zp = c_scale(c_mul(beta, bp[q]), 2.0);
    if (q == 1) { zp.r = fma(2.0 * sig, u * u, zp.r); zp.i = fma(2.0 * sig, u, zp.i); }
    const Cplx dp = c_mul(zp, inv2d);
    const Cplx Ep = c_scale(c_mul(dp, E), -T);
    const Cplx mp_ = c_sub(bp[q], dp), plp = c_add(bp[q], dp);
    const Cplx Dp = c_sub(c_sub(plp, c_mul(mp_, E)), c_mul(m, Ep));
    const Cplx DpD = c_mul(Dp, invD);
    const Cplx Bp = c_mul(c_mul(uu, c_add(Ep, c_mul(omE, DpD))), invD);
    const Cplx Ahp = c_sub(c_scale(mp_, T), c_scale(c_sub(DpD, c_mul(dp, invd)), 2.0));
    const Cplx Ap = c_add(c_scale(Ahat, cp[q]), c_scale(Ahp, s.c[j]));
    dX[slot[q]] = c_add(Ap, c_scale(Bp, s.v0[j]));
  }
}

// X at u (the same value arithmetic as cf_exponent) and dX/dp_i for the 13 parameters in calibrator order.
//   jump / drift:  dX/dlam = T (J - 1) - i u T (C - 1),  dX/dmu = i u lam T (J - C),
//                  dX/dsj = -lam T sj (i u C + u^2 J),   J = exp(i u mu - sj^2 u^2 / 2),  C = exp(mu + sj^2 / 2)
DHJ_HD void cf_exponent_tangents(const Params& mp, const SetConsts& s, double u, double T,
                                 const fm::Tables* __restrict__ ltab, double* xr_out, double* xi_out,
                                 Cplx* dX) {
  const double lamT = s.lam * T;
  double aR = 0.0, aI = (s.drift * u) * T, sli = 0.0, xbr = 0.0, xbi = 0.0;
  heston_factor_tangents(mp, s, 0, u, T, ltab, aR, aI, sli, xbr, xbi, dX);
  heston_factor_tangents(mp, s, 1, u, T, ltab, aR, aI, sli, xbr, xbi, dX + 5);
  double xr = aR + xbr;
  double xi = fma(-2.0, sli, aI) + xbi;
  double cj, sj;
  fm::sincos_(u * s.mu, &sj, &cj);
  const double ej = jump_gauss(s, u, ltab);
  xr = fma(lamT, fma(ej, cj, -1.0), xr);
  xi = fma(lamT, ej * sj, xi);
  *xr_out = xr; *xi_out = xi;
  const double Jr = ej * cj, Ji = ej * sj;
  const double C = fm::exp_(s.mu + s.hsj2);
  const double uT = u * T;
  dX[10] = {T * (Jr - 1.0), fma(-uT, C - 1.0, T * Ji)};
  const double ulT = u * lamT;
  dX[11] = {-(ulT * Ji), ulT * (Jr - C)};
  const double lts = lamT * mp.sj, u2 = u * u;
  dX[12] = {-(lts * (u2 * Jr)), -(lts * fma(u, C, u2 * Ji))};
}

// X at u (the value arithmetic of cf_exponent_tangents) and its derivatives in the maturity and the rate, for the
// Greeks (dhj_greeks.cuh): dX[0] = dX/dT, dX[1] = dX/dr.  beta, d and c do not depend on T; forward mode through
// E = exp(-d T):
//   E_T = -d E,  D_T = -m E_T,  B_T = u (u+i) (E_T + (1-E) D_T/D) / D,  Ahat_T = m - 2 D_T/D
//   dX/dT = sum_j (c_j Ahat_T + v0_j B_T) + i drift u + lam (J - 1),   dX/dr = i u T   (from A0 = i drift u T)
// (dX/dq = -dX/dr; the truncation range depends on T and r, and is held fixed.)
DHJ_HD void cf_exponent_time(const SetConsts& s, double u, double T, const fm::Tables* __restrict__ ltab,
                             double* xr_out, double* xi_out, Cplx* dX) {
  const double lamT = s.lam * T;
  double aR = 0.0, aI = (s.drift * u) * T, sli = 0.0, xbr = 0.0, xbi = 0.0;
  const Cplx uu = {u * u, u};                                  // u (u + i)
  Cplx dT = {0.0, s.drift * u};
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const FactorState f = heston_factor_state(s, j, u, T, ltab, aR, aI, sli, xbr, xbi);
    const Cplx E = {f.Er, f.Ei}, m = {f.mr, f.mi}, omE = {1.0 - f.Er, -f.Ei};
    const Cplx invD = {f.Dr * f.inD, -(f.Di * f.inD)};
    const Cplx ET = c_scale(c_mul({f.dr, f.di}, E), -1.0);
    const Cplx DTD = c_mul(c_scale(c_mul(m, ET), -1.0), invD);
    const Cplx BT = c_mul(c_mul(uu, c_add(ET, c_mul(omE, DTD))), invD);
    const Cplx AhT = c_sub(m, c_scale(DTD, 2.0));
    dT = c_add(dT, c_add(c_scale(AhT, s.c[j]), c_scale(BT, s.v0[j])));
  }
  double xr = aR + xbr;
  double xi = fma(-2.0, sli, aI) + xbi;
  double cj, sj;
  fm::sincos_(u * s.mu, &sj, &cj);
  const double ej = jump_gauss(s, u, ltab);
  xr = fma(lamT, fma(ej, cj, -1.0), xr);
  xi = fma(lamT, ej * sj, xi);
  *xr_out = xr; *xi_out = xi;
  const double Jr = ej * cj, Ji = ej * sj;
  dX[0] = {fma(s.lam, Jr - 1.0, dT.r), fma(s.lam, Ji, dT.i)};
  dX[1] = {0.0, u * T};
}

// everything the strike loop needs for one k
struct KTerm {
  double G;      // w_k Re(phi(u_k) e^{-i u_k a}), w_0 = 1/2     double_heston.py:187-188
  double u;      // (k*pi)/(b-a)                              double_heston.py:166
  double inv1;   // 1/(1+u^2)
  double invu;   // 1/u (0 for k = 0, where psi_0 is special-cased)
  double sb;     // sin(u (b-a))
  double t1;     // cos(u (b-a)) * e^b
  double t3;     // (u * sin(u (b-a))) * e^b
};

// u_k = (k*pi)/(b-a): quotient from the precomputed reciprocal plus one correction step
DHJ_HD double u_of_k(const PassConsts& p, int k) {
  const double kpi = (double)k * kPi;
  const double q0 = kpi * p.rw;
  return fma(fma(-p.w, q0, kpi), p.rw, q0);
}

// u = u_k; jump_trig as in cf_exponent_f
template <class JumpTrig>
DHJ_HD KTerm make_kterm_f(const SetConsts& s, const PassConsts& p, int k, const fm::TrigTables* __restrict__ ltab,
                          double u, JumpTrig jump_trig) {
  KTerm t;
  t.u = u;
  double xr, xi;
  cf_exponent_f(s, u, p.T, p.lamT, ltab, jump_trig, &xr, &xi);
  // Re( cf_heston * cf_jump * e^{-i u a} ) with the three exponentials merged
  // (the k = 0 weight 1/2 of double_heston.py:188 is folded in here: scaling by 2^-1 commutes exactly)
  t.G = (fm::exp_tab(xr, ltab) * fm::cos_tab(fma(-u, p.a, xi), ltab)) * ((k == 0) ? 0.5 : 1.0);
  // sin / cos of fl(u (b-a)) = k pi + delta, |delta| <~ 1e-13: sin = (-1)^k delta, cos = (-1)^k exactly in
  // double (what libm returns for this argument), with delta from a two-term pi
  const double kf = (double)k;
  const double delta = fma(-kf, kPiLo, fma(-kf, kPi, u * p.w));
  const double sbv = fm::xor_sign(delta, k << 31);
  t.sb = sbv;
  t.t1 = fm::xor_sign(p.eb, k << 31);
  t.t3 = (u * sbv) * p.eb;
  t.inv1 = fm::rcp(fma(u, u, 1.0));
  t.invu = (k == 0) ? 0.0 : fm::rcp(u);
  return t;
}

DHJ_HD KTerm make_kterm(const SetConsts& s, const PassConsts& p, int k, const fm::TrigTables* __restrict__ ltab) {
  const double u = u_of_k(p, k);
  return make_kterm_f(s, p, k, ltab, u, [&](double* cj, double* sj, double* ej) {
    fm::sincos_(u * s.mu, sj, cj);
    *ej = jump_gauss(s, u, ltab);
  });
}

// strike-dependent constants of one option
struct StrikeConsts {
  double K, x, ex;     // strike, log(K/S0), exp(x)
};

DHJ_HD StrikeConsts make_strike_consts(double K, double S0) {
  StrikeConsts c;
  c.K = K; c.x = fm::log_ratio(K, S0); c.ex = fm::exp_(c.x);
  return c;
}

// ---- rotation-based strike contraction -------------------------------------------------------------
// With theta = pi (x - a)/(b - a) the strike enters the payoff only through cos(k theta), sin(k theta):
//   sum_k w_k Re(phi_k e^{-i u_k a}) V_k
//     = [call] S0 A1 - K A2 - K g0 (b - x)   or   [put] S0 e^a A3 + K g0 (x - a)
//       + K sum_k R_k sin(k theta) - S0 e^x sum_k (P_k cos(k theta) + Q_k sin(k theta))
// with the strike-independent  P_k = G_k tw/(1+u_k^2), Q_k = P_k u_k, R_k = G_k tw/u_k (R_0 = 0),
// A1 = sum P_k (t1_k + t3_k), A2 = sum R_k sin(u_k (b-a)), A3 = sum P_k, g0 = G_0 tw.
// The trigonometric sums are evaluated in segments of consecutive k: one exact sincos at the segment
// start, then plane rotations by theta (<= 32 steps, error growth <= 32 * 1.5 ulp).  This replaces one
// sincos per (strike, k) by ~7 FMAs (SURVEY H5).
struct KCoef { double P, Q, R, a1, a2, g0; };

DHJ_HD KCoef make_kcoef(const KTerm& t, const PassConsts& p, int k) {
  KCoef c;
  const double gt = t.G * p.tw;
  c.P = gt * t.inv1;
  c.Q = c.P * t.u;
  c.R = gt * t.invu;                 // invu = 0 for k = 0
  c.a1 = c.P * (t.t1 + t.t3);
  c.a2 = c.R * t.sb;
  c.g0 = (k == 0) ? gt : 0.0;
  return c;
}

// sums over one segment: sum (P cos + Q sin) and sum R sin, starting from (c, s) = cos/sin(k0 theta).
// cos/sin((k0+i) theta) advance by the three-term recurrence  t_{i+1} = 2 cos(theta) t_i - t_{i-1}  (one FMA per
// sequence and step; the first step is a plane rotation by theta).  Its rounding error grows like i eps / sin(theta)
// over the <= 32 steps of a segment (theta = pi (x-a)/(b-a) is >= pi * 0.1/(b-a) by the +-0.1 widening).
#if defined(__CUDACC__)
using Pair = double2;                         // 16-byte aligned: one 128-bit shared-memory load
#else
struct alignas(16) Pair { double x, y; };
#endif

// PQ[i] = (P, Q) of term k0 + i; RR[i] = (R of term k0 + 2i, R of term k0 + 2i + 1); SEG even.
template <int SEG>
DHJ_HD void segment_sums(const Pair* __restrict__ PQ, const Pair* __restrict__ RR, double c, double s, double cth,
                         double sth, double* sum_pq, double* sum_r) {
  Pair pq = PQ[0], rr = RR[0];
  double apq = fma(pq.y, s, pq.x * c), ar = rr.x * s;
  double c1 = fma(c, cth, -(s * sth)), s1 = fma(s, cth, c * sth);     // (k0 + 1) theta
  const double two_c = cth + cth;
  pq = PQ[1];
  apq = fma(pq.x, c1, apq); apq = fma(pq.y, s1, apq); ar = fma(rr.y, s1, ar);
#pragma unroll
  for (int i = 2; i < SEG; i += 2) {
    double c2 = fma(two_c, c1, -c), s2 = fma(two_c, s1, -s);          // (k0 + i) theta
    c = c1; s = s1; c1 = c2; s1 = s2;
    pq = PQ[i]; rr = RR[i >> 1];
    apq = fma(pq.x, c1, apq); apq = fma(pq.y, s1, apq); ar = fma(rr.x, s1, ar);
    c2 = fma(two_c, c1, -c); s2 = fma(two_c, s1, -s);                 // (k0 + i + 1) theta
    c = c1; s = s1; c1 = c2; s1 = s2;
    pq = PQ[i + 1];
    apq = fma(pq.x, c1, apq); apq = fma(pq.y, s1, apq); ar = fma(rr.y, s1, ar);
  }
  *sum_pq = apq; *sum_r = ar;
}

// The same for TWO strikes at once (dense kernel): the coefficient loads are shared and the two recurrences are
// independent chains, which is what the FP64 pipe needs to stay busy with few warps.  Same operations per strike as
// segment_sums: same bits.
template <int SEG>
DHJ_HD void segment_sums2(const Pair* __restrict__ PQ, const Pair* __restrict__ RR, double ca, double sa, double ctha,
                          double stha, double cb, double sb, double cthb, double sthb, double* sum_pq_a,
                          double* sum_r_a, double* sum_pq_b, double* sum_r_b) {
  Pair pq = PQ[0], rr = RR[0];
  double apqa = fma(pq.y, sa, pq.x * ca), ara = rr.x * sa;
  double apqb = fma(pq.y, sb, pq.x * cb), arb = rr.x * sb;
  double c1a = fma(ca, ctha, -(sa * stha)), s1a = fma(sa, ctha, ca * stha);
  double c1b = fma(cb, cthb, -(sb * sthb)), s1b = fma(sb, cthb, cb * sthb);
  const double two_ca = ctha + ctha, two_cb = cthb + cthb;
  pq = PQ[1];
  apqa = fma(pq.x, c1a, apqa); apqa = fma(pq.y, s1a, apqa); ara = fma(rr.y, s1a, ara);
  apqb = fma(pq.x, c1b, apqb); apqb = fma(pq.y, s1b, apqb); arb = fma(rr.y, s1b, arb);
#pragma unroll
  for (int i = 2; i < SEG; i += 2) {
    double c2a = fma(two_ca, c1a, -ca), s2a = fma(two_ca, s1a, -sa);
    double c2b = fma(two_cb, c1b, -cb), s2b = fma(two_cb, s1b, -sb);
    ca = c1a; sa = s1a; c1a = c2a; s1a = s2a;
    cb = c1b; sb = s1b; c1b = c2b; s1b = s2b;
    pq = PQ[i]; rr = RR[i >> 1];
    apqa = fma(pq.x, c1a, apqa); apqa = fma(pq.y, s1a, apqa); ara = fma(rr.x, s1a, ara);
    apqb = fma(pq.x, c1b, apqb); apqb = fma(pq.y, s1b, apqb); arb = fma(rr.x, s1b, arb);
    c2a = fma(two_ca, c1a, -ca); s2a = fma(two_ca, s1a, -sa);
    c2b = fma(two_cb, c1b, -cb); s2b = fma(two_cb, s1b, -sb);
    ca = c1a; sa = s1a; c1a = c2a; s1a = s2a;
    cb = c1b; sb = s1b; c1b = c2b; s1b = s2b;
    pq = PQ[i + 1];
    apqa = fma(pq.x, c1a, apqa); apqa = fma(pq.y, s1a, apqa); ara = fma(rr.y, s1a, ara);
    apqb = fma(pq.x, c1b, apqb); apqb = fma(pq.y, s1b, apqb); arb = fma(rr.y, s1b, arb);
  }
  *sum_pq_a = apqa; *sum_r_a = ara; *sum_pq_b = apqb; *sum_r_b = arb;
}

// strike-dependent constant part (uses warp- or block-level sums A1, A2, A3, g0: it is linear in them)
DHJ_HD double strike_const_part(bool is_call, double S0, double K, double x, const PassConsts& p, double A1,
                                double A2, double A3, double g0) {
  return is_call ? (S0 * A1 - K * A2) - (K * g0) * (p.b - x)
                 : (S0 * p.ea) * A3 + (K * g0) * (x - p.a);
}

}  // namespace dhj
