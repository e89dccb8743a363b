// dhj_dense.cuh — pricing kernel for slices with many strikes (the 200 x 20 dense surface of C3, or any
// option list with more than 8 strikes per maturity): ONE WARP PER ITEM (parameter set, maturity slice), no block
// barrier anywhere in the item loop.
//
//   * prologue: lanes 0 and 1 compute the two factors' constants and cumulants, lane 2 the jump / drift constants,
//     lane 3 the discount factor; the cumulants are shuffled, every lane forms (a0, b0), lanes 0..2 finish the pass
//     constants (same scalar functions as the batch kernel's prepare_item: same bits);
//   * strikes are processed in chunks of 224: the lanes prepare strike constants (K, log(K/S0), S0 exp(.),
//     binding / call flags, rotation step cos / sin(theta_j)) into the warp's private shared memory;
//   * per block of 32 cosine terms every lane evaluates the CF at its k and leaves the strike-independent
//     coefficients (P, Q, R) in the warp's stage; each lane then contracts ONE STRIKE per round against the 32
//     coefficients by the three-term recurrence (segment_sums, one exact sincos at the segment start) — 5 FMAs per
//     (strike, k) instead of a sincos + 15 flops; the strike-independent sums A1, A2, A3 are accumulated per lane
//     and reduced once per pass;
//   * strikes whose +-0.1 widening binds get their own pass (own (a,b), own CF), one strike at a time, contracted
//     by four lanes (8-term segments) as the batch kernel does.
// (r01 ran one BLOCK per item: thread 0 prepared the item behind two block barriers and 20 % of all warp samples
// sat at that barrier — profiles/ncu_k_dense_r02_base.txt.)
#pragma once
#include "dhj_batch.cuh"

namespace dhj {

constexpr int kDenseChunk = 224;
constexpr int kDenseWarps = 4;
#ifndef DHJ_DENSE_MINB
#define DHJ_DENSE_MINB 4
#endif

struct DenseWarp {
  SetConsts set;
  PassConsts pass, extra_pass;
  double S0, disc, a0, b0;
  double jrot[3], extra_jrot[3];                   // jump recurrences of the regular / extra pass: cos, sin(32 u_1 mu), exp(-2048 alpha)
  double extra_cth, extra_sth;
  CoefStage stage;
  double K[kDenseChunk], x[kDenseChunk], sex[kDenseChunk], cth[kDenseChunk], sth[kDenseChunk];   // sex = S0 exp(x)
  double part[kDenseChunk];                        // price accumulators of the chunk's strikes
  unsigned char call[kDenseChunk], bind[kDenseChunk];
};

struct DenseSmem {
  DenseWarp w[kDenseWarps];
  fm::TrigTables ltab;
};

// prologue of one item by its warp (see the header)
__device__ __forceinline__ void dense_prepare(DenseWarp& W, const SliceView& v, const double* __restrict__ pp,
                                              int transform, double S0, double T, int lane) {
  Params m;
  if (transform) {
    double* scratch = reinterpret_cast<double*>(&W.stage);
    if (lane < kNumParams) {
      const double x = pp[lane];
      scratch[lane] = (lane == 4 || lane == 9) ? tanh(x) : ((lane == 11) ? x : fm::exp_(x));
    }
    __syncwarp();
    m = load_params(scratch);
    __syncwarp();
  } else {
    m = load_params(pp);
  }
  double c1j = 0.0, c2j = 0.0;
  if (lane < 2) {
    set_consts_factor(m, lane, W.set);
    factor_cumulants(T, v.r, m.v0[lane], m.kappa[lane], m.theta[lane], m.sigma[lane], m.rho[lane], &c1j, &c2j);
  } else if (lane == 2) {
    set_consts_jump(m, v.r, v.q, W.set);
  } else if (lane == 3) {
    W.S0 = S0;
    W.disc = fm::exp_(-v.r * T);
  }
  const double c1_0 = __shfl_sync(kFullMask, c1j, 0), c2_0 = __shfl_sync(kFullMask, c2j, 0);
  const double c1_1 = __shfl_sync(kFullMask, c1j, 1), c2_1 = __shfl_sync(kFullMask, c2j, 1);
  double a0, b0;
  truncation_from_cumulants(m, T, v.L, c1_0, c2_0, c1_1, c2_1, &a0, &b0);
  if (lane == 0) {
    const double w = b0 - a0;
    W.pass.a = a0; W.pass.b = b0; W.pass.w = w; W.pass.rw = fm::rcp(w); W.pass.tw = fm::div(2.0, w);
    W.pass.T = T; W.pass.lamT = m.lam * T;
    W.a0 = a0; W.b0 = b0;
  } else if (lane == 1) {
    W.pass.eb = fm::exp_(b0);
  } else if (lane == 2) {
    W.pass.ea = fm::exp_(a0);
  } else if (lane == 3) {
    PassConsts pc;                                   // the two fields u_one() reads
    pc.w = b0 - a0; pc.rw = fm::rcp(pc.w);
    jump_rotation(pc, m.mu, &W.jrot[0], &W.jrot[1]);
    W.jrot[2] = fm::exp_neg(-2048.0 * jump_alpha(pc, 0.5 * (m.sj * m.sj)));
  }
}

// loop-carried state of the jump term's recurrences over the blocks of one pass (as in the batch kernel's
// contract_pass: exact every kReseed blocks, a rotation / two products in between)
struct JumpState { double cj = 1.0, sj = 0.0, ej = 1.0, rho = 1.0; };

// CF at this lane's k of the block [k0, k0 + 32) -> strike-independent coefficients in the warp's stage; the lanes'
// shares of A1, A2, A3 accumulate in a1, a2, a3; g0 (k = 0 only) is broadcast in the first block
__device__ __forceinline__ void dense_coefficients(DenseWarp& W, const PassConsts& pc, const double* __restrict__ jrot,
                                                   JumpState& js, int k0, int n_cos, int lane,
                                                   const fm::TrigTables* __restrict__ ltab, double& a1, double& a2,
                                                   double& a3, double& g0) {
  const int k = k0 + lane;
  const bool exact = ((k0 >> 5) % kReseed) == 0;        // uniform
  const double u = u_of_k(pc, k);
  KTerm t = make_kterm_f(W.set, pc, k, ltab, u, [&](double* cj_out, double* sj_out, double* ej_out) {
    if (exact) {
      fm::sincos_tab(u * W.set.mu, ltab, &js.sj, &js.cj);
      js.ej = jump_gauss(W.set, u, ltab);
      js.rho = fm::exp_tab_neg(-(jump_alpha(pc, W.set.hsj2) * (double)(64 * k + 1024)), ltab);
    } else {
      js.ej *= js.rho; js.rho *= jrot[2];
      rotate(js.cj, js.sj, jrot[0], jrot[1]);
    }
    *cj_out = js.cj; *sj_out = js.sj; *ej_out = js.ej;
  });
  t.G = (k < n_cos) ? t.G : 0.0;                         // ragged last block: every coefficient is a multiple of G
  KCoef c = make_kcoef(t, pc, k);
  c.a1 = (k < n_cos) ? c.a1 : 0.0; c.a2 = (k < n_cos) ? c.a2 : 0.0;
  a1 += c.a1; a2 += c.a2; a3 += c.P;
  if (k0 == 0) g0 = __shfl_sync(kFullMask, c.g0, 0);
  __syncwarp();                                        // the previous block's coefficients have been consumed
#if defined(DHJ_CHECKED)
  const unsigned epoch = W.stage.epoch + 1;
  for (int l = 0; l < 32; ++l) DHJ_CHECK(W.stage.rtag[l] == epoch - 1, kChkWriteBeforeConsumed);
  __syncwarp();
  W.stage.wtag[lane] = epoch;
  if (lane == 0) W.stage.epoch = epoch;
#endif
  W.stage.PQ[lane] = make_double2(c.P, c.Q); W.stage.R[lane] = c.R;
  __syncwarp();
#if defined(DHJ_CHECKED)
  for (int l = 0; l < 32; ++l) DHJ_CHECK(W.stage.wtag[l] == epoch, kChkReadBeforeWrite);
#endif
}
// checked build: this lane has finished reading the block's coefficients
__device__ __forceinline__ void dense_consumed(DenseWarp& W, int lane) {
#if defined(DHJ_CHECKED)
  W.stage.rtag[lane] = W.stage.epoch;
#endif
}

// regular pass: all strikes of the chunk whose widening does not bind, a lane per strike, rounds of 32
__device__ __forceinline__ void dense_pass(DenseWarp& W, int cnt, int n_cos, int lane,
                                           const fm::TrigTables* __restrict__ ltab) {
  const PassConsts& pc = W.pass;
  double a1 = 0.0, a2 = 0.0, a3 = 0.0, g0 = 0.0;
  JumpState js;
#pragma unroll 1
  for (int k0 = 0; k0 < n_cos; k0 += 32) {
    dense_coefficients(W, pc, W.jrot, js, k0, n_cos, lane, ltab, a1, a2, a3, g0);
    const double u0 = u_of_k(pc, k0);                   // frequency of the block's first term
    // two strikes per lane and trip (t, t + 32) while both exist, then single strikes: the pair shares the
    // coefficient loads and gives the pipe two independent chains
    int t = lane;
#pragma unroll 1
    for (; t + 32 < cnt; t += 64) {
      const int tb = t + 32;
      double sna, csa, snb, csb, spqa, sra, spqb, srb;
      fm::sincos_tab(u0 * (W.x[t] - pc.a), ltab, &sna, &csa);
      fm::sincos_tab(u0 * (W.x[tb] - pc.a), ltab, &snb, &csb);
      segment_sums2<32>(W.stage.PQ, reinterpret_cast<const Pair*>(W.stage.R), csa, sna, W.cth[t], W.sth[t], csb, snb,
                        W.cth[tb], W.sth[tb], &spqa, &sra, &spqb, &srb);
      if (!W.bind[t]) W.part[t] += fma(W.K[t], sra, -(W.sex[t] * spqa));
      if (!W.bind[tb]) W.part[tb] += fma(W.K[tb], srb, -(W.sex[tb] * spqb));
    }
    if (t < cnt && !W.bind[t]) {
      double sn, cs, spq, sr;
      fm::sincos_tab(u0 * (W.x[t] - pc.a), ltab, &sn, &cs);
      segment_sums<32>(W.stage.PQ, reinterpret_cast<const Pair*>(W.stage.R), cs, sn, W.cth[t], W.sth[t], &spq, &sr);
      W.part[t] += fma(W.K[t], sr, -(W.sex[t] * spq));
    }
    dense_consumed(W, lane);
  }
  const double A1 = warp_sum(a1), A2 = warp_sum(a2), A3 = warp_sum(a3);
  for (int t = lane; t < cnt; t += 32)
    if (!W.bind[t])
      W.part[t] += strike_const_part(W.call[t] != 0, W.S0, W.K[t], W.x[t], pc, A1, A2, A3, g0);
}

// pass of ONE strike with its own (a, b): four lanes contract 8-term segments, as in the batch kernel
__device__ __forceinline__ void dense_pass_single(DenseWarp& W, int t, int n_cos, int lane,
                                                  const fm::TrigTables* __restrict__ ltab) {
  if (lane == 0) {
    W.extra_pass = make_pass_consts(W.set, py_min(W.a0, W.x[t] - 0.1), py_max(W.b0, W.x[t] + 0.1), W.pass.T);
    fm::sincos_(u_one(W.extra_pass) * (W.x[t] - W.extra_pass.a), &W.extra_sth, &W.extra_cth);
    jump_rotation(W.extra_pass, W.set.mu, &W.extra_jrot[0], &W.extra_jrot[1]);
    W.extra_jrot[2] = fm::exp_neg(-2048.0 * jump_alpha(W.extra_pass, W.set.hsj2));
  }
  __syncwarp();
  const PassConsts& pc = W.extra_pass;
  double a1 = 0.0, a2 = 0.0, a3 = 0.0, g0 = 0.0, acc = 0.0;
  JumpState js;
#pragma unroll 1
  for (int k0 = 0; k0 < n_cos; k0 += 32) {
    dense_coefficients(W, pc, W.extra_jrot, js, k0, n_cos, lane, ltab, a1, a2, a3, g0);
    double val = 0.0;
    if (lane < 4) {
      double sn, cs, spq, sr;
      fm::sincos_tab(u_of_k(pc, k0 + 8 * lane) * (W.x[t] - pc.a), ltab, &sn, &cs);
      segment_sums<8>(W.stage.PQ + 8 * lane, reinterpret_cast<const Pair*>(W.stage.R + 8 * lane), cs, sn, W.extra_cth,
                      W.extra_sth, &spq, &sr);
      val = fma(W.K[t], sr, -(W.sex[t] * spq));
    }
    val += __shfl_xor_sync(kFullMask, val, 1);
    val += __shfl_xor_sync(kFullMask, val, 2);
    acc += val;                                        // meaningful in lane 0
    dense_consumed(W, lane);
  }
  const double A1 = warp_sum(a1), A2 = warp_sum(a2), A3 = warp_sum(a3);
  if (lane == 0) W.part[t] = acc + strike_const_part(W.call[t] != 0, W.S0, W.K[t], W.x[t], pc, A1, A2, A3, g0);
  __syncwarp();
}

}  // namespace dhj
