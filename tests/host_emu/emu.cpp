// TEST-ONLY host emulation of the kernel arithmetic in option-pricing-ffn-lbfgs_b200/csrc/dhj_math.cuh.
//
// Compiles the very same scalar functions the CUDA kernels call (DHJ_HD expands to `inline` under
// g++) and walks k in the kernel's order (k = lane + 32*i, per-lane partial sums, xor-butterfly across
// the 32 lanes), so the CPU test-suite can check the kernel's algebra against the golden fixtures
// without a GPU.  It differs from the device only in libm (glibc vs CUDA sin/cos/exp/log/atan2).
// emu_price_walk also walks the orders of the current k_price_batch and k_price_dense (blocks of 32 k with the jump
// term's recurrences between exact blocks), which price_one (the r01 order, exact sincos everywhere) does not.
// This is NOT a CPU fallback: nothing in the product package loads it; tests/test_host_emu.py builds it
// on the fly with g++ into tests/host_emu/_build/.
#include "dhj_math.cuh"

using namespace dhj;

static double butterfly_total(double* v) {        // xor-butterfly over 32 lanes, as warp_sum does
  for (int off = 16; off >= 1; off >>= 1) {
    double t[32];
    for (int l = 0; l < 32; ++l) t[l] = v[l] + v[l ^ off];
    for (int l = 0; l < 32; ++l) v[l] = t[l];
  }
  return v[0];
}

static double u_of(const PassConsts& p, int k) {
  const double kpi = (double)k * kPi;
  const double q0 = kpi * p.rw;
  return fma(fma(-p.w, q0, kpi), p.rw, q0);
}

// one option, walked the way k_price_batch does it: blocks of 128 k, 4 warps of 32 lanes, strike-independent
// coefficients, four butterfly sums, 8-term rotation segments, partials per warp added in warp order
static double price_one(const Params& m, double S0, double K, double T, double r, double q, int is_call,
                        int N, double L, double* ab) {
  SetConsts s = make_set_consts(m, r, q);
  double a0, b0;
  truncation_range(m, T, r, L, &a0, &b0);
  StrikeConsts sc = make_strike_consts(K, S0);
  double a = py_min(a0, sc.x - 0.1), b = py_max(b0, sc.x + 0.1);
  if (ab) { ab[0] = a; ab[1] = b; }
  PassConsts p = make_pass_consts(s, a, b, T);
  double sth, cth;
  fm::sincos_(u_of(p, 1) * (sc.x - p.a), &sth, &cth);
  double partial[4] = {0, 0, 0, 0};
  for (int k0 = 0; k0 < N; k0 += 128) {
    for (int w = 0; w < 4; ++w) {
      Pair PQ[32];
      alignas(16) double R[32];
      double a1[32], a2[32], a3[32], g0[32];
      for (int lane = 0; lane < 32; ++lane) {
        const int k = k0 + 32 * w + lane;
        KCoef c; c.P = c.Q = c.R = c.a1 = c.a2 = c.g0 = 0.0;
        if (k < N) c = make_kcoef(make_kterm(s, p, k, &fm::kTables), p, k);
        PQ[lane].x = c.P; PQ[lane].y = c.Q; R[lane] = c.R; a1[lane] = c.a1; a2[lane] = c.a2; a3[lane] = c.P; g0[lane] = c.g0;
      }
      const double A1 = butterfly_total(a1), A2 = butterfly_total(a2), A3 = butterfly_total(a3), G0 = butterfly_total(g0);
      double val[4];
      for (int sg = 0; sg < 4; ++sg) {
        const int kstart = k0 + 32 * w + 8 * sg;
        double sn, cs, spq, sr;
        fm::sincos_(u_of(p, kstart) * (sc.x - p.a), &sn, &cs);
        segment_sums<8>(PQ + 8 * sg, reinterpret_cast<const Pair*>(R + 8 * sg), cs, sn, cth, sth, &spq, &sr);
        val[sg] = sc.K * sr - (S0 * sc.ex) * spq;
        if (sg == 0) val[sg] += strike_const_part(is_call != 0, S0, sc.K, sc.x, p, A1, A2, A3, G0);
      }
      partial[w] += (val[0] + val[1]) + (val[2] + val[3]);
    }
  }
  return fm::exp_(-r * T) * (((partial[0] + partial[1]) + partial[2]) + partial[3]);
}

// ---- the current kernels' orders (dhj_batch.cuh contract_pass / run_batch, dhj_dense.cuh dense_pass /
// dense_pass_single): blocks of 32 k, the jump term's cos / sin(u mu) and Gaussian advanced by recurrences between the
// exact blocks (every kReseed-th).  An option's price does not depend on the other strikes of its slice (the A-sums
// and the CF are strike-independent, a binding strike has a pass of its own), so both walks price one option at a time.
// Device-only helpers of dhj_batch.cuh, restated:
static constexpr int kReseedH = 8;                     // kReseed
static double u_one_h(const PassConsts& p) {
  const double q0 = kPi * p.rw;
  return fma(fma(-p.w, q0, kPi), p.rw, q0);
}
static void rotate_h(double& c, double& s, double cr, double sr) {
  const double c2 = fma(c, cr, -(s * sr)), s2 = fma(s, cr, c * sr);
  c = c2; s = s2;
}
static double jump_alpha_h(const PassConsts& p, double hsj2) {
  const double u1 = u_one_h(p);
  return hsj2 * (u1 * u1);
}

// per-lane state of the jump recurrences and one block's coefficients (lane = k - k0)
struct EmuLanes {
  double cj[32], sj[32], ej[32], rho[32];
  Pair PQ[32];
  alignas(16) double R[32];
  EmuLanes() { for (int l = 0; l < 32; ++l) { cj[l] = 1.0; sj[l] = 0.0; ej[l] = 1.0; rho[l] = 1.0; } }
};

// make_kterm_f with the recurrence of contract_pass / dense_coefficients for lane `lane` of block `blk`
static KTerm kterm_rec(const SetConsts& s, const PassConsts& pc, const double* jrot, EmuLanes& L, int k0, int lane,
                       int n_cos) {
  const int k = k0 + lane;
  const bool exact = ((k0 >> 5) % kReseedH) == 0;
  const double u = u_of_k(pc, k);
  KTerm t = make_kterm_f(s, pc, k, &fm::kTables, u, [&](double* cj_out, double* sj_out, double* ej_out) {
    if (exact) {
      fm::sincos_(u * s.mu, &L.sj[lane], &L.cj[lane]);
      L.ej[lane] = jump_gauss(s, u, &fm::kTables);
      L.rho[lane] = fm::exp_tab_neg(-(jump_alpha_h(pc, s.hsj2) * (double)(64 * k + 1024)), &fm::kTables);
    } else {
      L.ej[lane] *= L.rho[lane]; L.rho[lane] *= jrot[2];
      rotate_h(L.cj[lane], L.sj[lane], jrot[0], jrot[1]);
    }
    *cj_out = L.cj[lane]; *sj_out = L.sj[lane]; *ej_out = L.ej[lane];
  });
  t.G = (k < n_cos) ? t.G : 0.0;
  return t;
}

struct EmuItem {                                       // what prepare_item / dense_prepare leave for one option
  SetConsts set;
  PassConsts pass;                                     // regular pass (a0, b0)
  double disc, jrot[3];
  double K, x, sex;
  bool bind;
};

static EmuItem emu_item(const Params& m, double S0, double K, double T, double r, double q, double L) {
  EmuItem it;
  it.set = make_set_consts(m, r, q);
  double a0, b0;
  truncation_range(m, T, r, L, &a0, &b0);
  it.pass = make_pass_consts(it.set, a0, b0, T);
  it.disc = fm::exp_(-r * T);
  fm::sincos_((32.0 * u_one_h(it.pass)) * it.set.mu, &it.jrot[1], &it.jrot[0]);
  it.jrot[2] = fm::exp_neg(-2048.0 * jump_alpha_h(it.pass, it.set.hsj2));
  const StrikeConsts sc = make_strike_consts(K, S0);
  it.K = sc.K; it.x = sc.x; it.sex = S0 * sc.ex;
  it.bind = ((sc.x - 0.1) < a0) || ((sc.x + 0.1) > b0);
  return it;
}

// the binding strike's own pass constants and rotation steps (run_batch's lane 0 / dense_pass_single's lane 0)
static PassConsts emu_extra_pass(const EmuItem& it, double* jrot) {
  const PassConsts p = make_pass_consts(it.set, py_min(it.pass.a, it.x - 0.1), py_max(it.pass.b, it.x + 0.1),
                                        it.pass.T);
  fm::sincos_((32.0 * u_one_h(p)) * it.set.mu, &jrot[1], &jrot[0]);
  jrot[2] = fm::exp_neg(-2048.0 * jump_alpha_h(p, it.set.hsj2));
  return p;
}

// k_price_batch: one pass of contract_pass for one strike (regular or its own), four 8-term segments per block whose
// starts advance by the rotation by 32 theta between exact blocks, reduced as (v0 + v1) + (v2 + v3); A-sums per lane,
// one butterfly at the end
static double batch_option(const EmuItem& it, double S0, int is_call, int N) {
  double jrot[3] = {it.jrot[0], it.jrot[1], it.jrot[2]};
  const PassConsts pc = it.bind ? emu_extra_pass(it, jrot) : it.pass;
  double cth, sth, c32, s32;
  const double th = u_one_h(pc) * (it.x - pc.a);
  fm::sincos_(th, &sth, &cth);
  fm::sincos_(32.0 * th, &s32, &c32);
  EmuLanes L;
  double a1[32] = {0}, a2[32] = {0}, a3[32] = {0}, g0 = 0.0, acc = 0.0;
  double cs[4] = {1.0, 1.0, 1.0, 1.0}, sn[4] = {0.0, 0.0, 0.0, 0.0};
  for (int k0 = 0, blk = 0; k0 < N; k0 += 32, ++blk) {
    const bool exact = (blk % kReseedH) == 0;
    for (int lane = 0; lane < 32; ++lane) {
      const KTerm t = kterm_rec(it.set, pc, jrot, L, k0, lane, N);
      const KCoef c = make_kcoef(t, pc, k0 + lane);
      if (is_call) { a1[lane] = fma(c.P, t.t1 + t.t3, a1[lane]); a2[lane] = fma(c.R, t.sb, a2[lane]); }
      else a3[lane] += c.P;
      if (blk == 0 && lane == 0) g0 = c.g0;
      L.PQ[lane].x = c.P; L.PQ[lane].y = c.Q; L.R[lane] = c.R;
    }
    double val[4];
    for (int sg = 0; sg < 4; ++sg) {
      if (exact) fm::sincos_(u_of_k(pc, k0 + 8 * sg) * (it.x - pc.a), &sn[sg], &cs[sg]);
      else rotate_h(cs[sg], sn[sg], c32, s32);
      double spq, sr;
      segment_sums<8>(L.PQ + 8 * sg, reinterpret_cast<const Pair*>(L.R + 8 * sg), cs[sg], sn[sg], cth, sth, &spq, &sr);
      val[sg] = fma(it.K, sr, -(it.sex * spq));
    }
    acc += (val[0] + val[1]) + (val[2] + val[3]);
  }
  const double A1 = is_call ? butterfly_total(a1) : 0.0, A2 = is_call ? butterfly_total(a2) : 0.0;
  const double A3 = is_call ? 0.0 : butterfly_total(a3);
  acc += strike_const_part(is_call != 0, S0, it.K, it.x, pc, A1, A2, A3, g0);
  return it.disc * acc;
}

// k_price_dense: a regular strike is contracted over 32-term segments from an exact sincos per block (dense_pass), a
// binding one in its own pass over four 8-term segments, each from an exact sincos (dense_pass_single); A-sums as
// plain sums of the masked a1, a2 and of P
static double dense_option(const EmuItem& it, double S0, int is_call, int N) {
  double jrot[3] = {it.jrot[0], it.jrot[1], it.jrot[2]};
  const PassConsts pc = it.bind ? emu_extra_pass(it, jrot) : it.pass;
  double cth, sth;
  fm::sincos_(u_one_h(pc) * (it.x - pc.a), &sth, &cth);
  EmuLanes L;
  double a1[32] = {0}, a2[32] = {0}, a3[32] = {0}, g0 = 0.0, acc = 0.0;
  for (int k0 = 0; k0 < N; k0 += 32) {
    for (int lane = 0; lane < 32; ++lane) {
      const int k = k0 + lane;
      const KTerm t = kterm_rec(it.set, pc, jrot, L, k0, lane, N);
      KCoef c = make_kcoef(t, pc, k);
      c.a1 = (k < N) ? c.a1 : 0.0; c.a2 = (k < N) ? c.a2 : 0.0;
      a1[lane] += c.a1; a2[lane] += c.a2; a3[lane] += c.P;
      if (k0 == 0 && lane == 0) g0 = c.g0;
      L.PQ[lane].x = c.P; L.PQ[lane].y = c.Q; L.R[lane] = c.R;
    }
    double sn, cs, spq, sr;
    if (!it.bind) {
      fm::sincos_(u_of_k(pc, k0) * (it.x - pc.a), &sn, &cs);
      segment_sums<32>(L.PQ, reinterpret_cast<const Pair*>(L.R), cs, sn, cth, sth, &spq, &sr);
      acc += fma(it.K, sr, -(it.sex * spq));
    } else {
      double val[4];
      for (int sg = 0; sg < 4; ++sg) {
        fm::sincos_(u_of_k(pc, k0 + 8 * sg) * (it.x - pc.a), &sn, &cs);
        segment_sums<8>(L.PQ + 8 * sg, reinterpret_cast<const Pair*>(L.R + 8 * sg), cs, sn, cth, sth, &spq, &sr);
        val[sg] = fma(it.K, sr, -(it.sex * spq));
      }
      acc += (val[0] + val[1]) + (val[2] + val[3]);
    }
  }
  const double A1 = butterfly_total(a1), A2 = butterfly_total(a2), A3 = butterfly_total(a3);
  acc += strike_const_part(is_call != 0, S0, it.K, it.x, pc, A1, A2, A3, g0);
  return it.disc * acc;
}

extern "C" {

// walk: 0 = the r01 order (price_one), 1 = k_price_batch's, 2 = k_price_dense's; bind (optional, [P][M]) receives
// 1 where the strike's widening binds
void emu_price_walk(int walk, const double* params, const double* S0, const double* strike, const double* maturity,
                    const int* is_call, double r, double q, long P, int M, int N, double L, double* out,
                    unsigned char* bind) {
  for (long p = 0; p < P; ++p) {
    const Params m = load_params(params + 13 * p);
    for (int o = 0; o < M; ++o) {
      const EmuItem it = emu_item(m, S0[p], strike[p * M + o], maturity[o], r, q, L);
      if (bind) bind[p * M + o] = it.bind;
      out[p * M + o] = walk == 0 ? price_one(m, S0[p], strike[p * M + o], maturity[o], r, q, is_call[o], N, L, nullptr)
                     : walk == 1 ? batch_option(it, S0[p], is_call[o], N) : dense_option(it, S0[p], is_call[o], N);
    }
  }
}

void emu_price_list(const double* params, const double* S0, int s0_stride, const double* strike,
                    int strike_stride, const double* maturity, const int* is_call, double r, double q,
                    long P, int M, int N, double L, double* out, double* ab) {
  for (long p = 0; p < P; ++p) {
    Params m = load_params(params + 13 * p);
    for (int o = 0; o < M; ++o)
      out[p * M + o] = price_one(m, S0[p * s0_stride], strike[p * strike_stride + o], maturity[o], r, q,
                                 is_call[o], N, L, ab ? ab + 2 * (p * M + o) : nullptr);
  }
}

void emu_loss(const double* x, long B, double S0, double r, const double* strike, const double* maturity,
              const int* is_call, const double* market, int M, int N, double* out) {
  for (long b = 0; b < B; ++b) {
    Params m = transform_params(x + 13 * b);
    bool bad = false;
    double sq = 0.0;
    for (int o = 0; o < M; ++o) {
      double pr = price_one(m, S0, strike[o], maturity[o], r, 0.0, is_call[o], N, 10.0, nullptr);
      if (!(pr > 0.0) || isinf(pr)) bad = true;
      double rel = (pr - market[o]) / market[o];
      sq += rel * rel;
    }
    out[b] = bad ? 1e10 : sq / (double)M + feller_penalty(m);
  }
}

void emu_cf(const double* params, double r, double q, double tau, const double* us, int n, double* re, double* im) {
  // full CF value phi(u) (without the e^{-iua} rotation) for checking against cf_values.npz:
  // uses a = 0 so that G = Re(phi); the imaginary part comes from a second pass rotated by pi/2.
  Params m = load_params(params);
  SetConsts s = make_set_consts(m, r, q);
  for (int i = 0; i < n; ++i) {
    // w chosen so that u_k = (k*pi)/w reproduces us[i] for k = 1 is not exact; evaluate the factors directly
    double u = us[i];
    double xr, xi;
    cf_exponent(s, u, tau, s.lam * tau, &fm::kTables, &xr, &xi);
    re[i] = exp(xr) * cos(xi);
    im[i] = exp(xr) * sin(xi);
  }
}
}
