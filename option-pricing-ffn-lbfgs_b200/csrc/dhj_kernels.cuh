// dhj_kernels.cuh — the CUDA kernels of libdhj.so (sm_100a).
//
//   k_price_batch  slices of <= 8 strikes: warp per item, lane per cosine index, 32 items per block   (K1 / K3 of SURVEY §2)
//   k_price_dense  many strikes per slice: warp per item, lane per strike
//   k_loss_batch   K2: exp/tanh transform + prices of every market option + relative-MSE + Feller penalty +
//                  1e10 sentinel; in FD mode the 14 stencil points of an optimiser state are 14 units and the
//                  thread that finishes the last one assembles scipy's gradient — ONE launch per optimiser step
//   k_fd_expand / k_loss_reduce  K2 around the pricing kernels: markets with > 8 strikes per maturity, and any
//                  batch of >= 8 192 loss evaluations (full 32-item batches balance the warps better)
//   k_cf / k_cf_complex / k_truncation_range / k_chi_psi  the remaining public methods of DoubleHeston
//   k_fp64_peak    DFMA-chain probe for the FP64 roofline denominator
#pragma once
#include "dhj_engine.cuh"
#include "dhj_batch.cuh"
#include "dhj_dense.cuh"

namespace dhj {

constexpr int kFdPoints = kNumParams + 1;      // f(x) and 13 forward points
constexpr double kSentinel = 1e10;             // lbfgs_calibrator.py:152-153

struct PriceArgs {
  const double* params;      // [P][13] model parameters, or unconstrained x when transform != 0
  const double* S0;          // spot table
  long long s0_stride;       // 0 = scalar
  const int* row_index;      // optional [P]: row of S0 / strike tables used by set p (default p)
  long long P;
  int transform;
  double* out;               // [P][M]
  int items_per_batch;       // <= kPriceItems; set by launch_price
};

// Slices of <= 8 strikes: see dhj_batch.cuh.
// FULL: batches of kPriceItems items (a compile-time constant: large launches); otherwise a.items_per_batch, chosen per
// launch for mid-size launches that are only a few waves of blocks long (launch_price)
template <bool FULL>
__global__ void __launch_bounds__(kBatchThreads, DHJ_BATCH_MINB) k_price_batch(SliceView v, PriceArgs a) {
  __shared__ PriceSmem sm;
  const int tid = threadIdx.x;
  load_log_table<kBatchThreads>(&sm.ltab, tid);
  stage_check_init(sm.stage[tid >> 5], tid & 31);
  const long long n_items = a.P * (long long)v.n_slices;
  const int ipb = FULL ? kPriceItems : a.items_per_batch;
  const long long n_batches = (n_items + ipb - 1) / ipb;
  for (long long batch = blockIdx.x; batch < n_batches; batch += gridDim.x) {
    const long long base = batch * ipb;
    const int cnt_items = (int)min((long long)ipb, n_items - base);
    // ---- phase 1: one thread per item ----------------------------------------------------------
#if defined(DHJ_COALESCED_PARAMS)
    // (experiment, profiles/README.md r02: the batch's parameter rows, contiguous in global memory, swept into shared
    // memory by all 128 threads with coalesced loads, then read per item from there)
    __shared__ double s_params[(kPriceItems + 2) * kNumParams];
    const long long p_first = base / v.n_slices, p_last = (base + cnt_items - 1) / v.n_slices;
    const int n_rows = (int)(p_last - p_first + 1);
    for (int e = tid; e < n_rows * kNumParams; e += kBatchThreads) s_params[e] = a.params[p_first * kNumParams + e];
    __syncthreads();
#endif
    if (tid < cnt_items) {
      const long long item = base + tid;
      const long long p = item / v.n_slices;
      const int s = (int)(item - p * v.n_slices);
      const long long row = a.row_index ? (long long)a.row_index[p] : p;
#if defined(DHJ_COALESCED_PARAMS)
      const double* pp = s_params + (p - p_first) * kNumParams;
#else
      const double* pp = a.params + kNumParams * p;
#endif
      const Params m = a.transform ? transform_params(pp) : load_params(pp);
      prepare_item(sm.items[tid], v, m, a.S0[row * a.s0_stride], v.strike + row * v.strike_stride, s,
                   p * (long long)v.n_options);
      tag_item(sm.items[tid], (unsigned long long)batch + 1);
    }
    __syncthreads();
    // ---- phase 2: a warp per item, a lane per cosine index; the warp writes its prices -------------------
    run_batch(sm, v, cnt_items, tid, (unsigned long long)batch + 1, [&](int, int j, const ItemRec& it, double price) {
      const long long at = it.out_row + v.pos[it.o_lo + j];
      DHJ_CHECK(at >= 0 && at < a.P * (long long)v.n_options, kChkOutputIndex);
      a.out[at] = price;
    });
    __syncthreads();
  }
}

// Many strikes per slice: one WARP per item, lane per strike (dhj_dense.cuh); no block barrier in the item loop.
__global__ void __launch_bounds__(32 * kDenseWarps, DHJ_DENSE_MINB) k_price_dense(SliceView v, PriceArgs a) {
  extern __shared__ __align__(16) unsigned char dense_smem_raw[];
  DenseSmem& sm = *reinterpret_cast<DenseSmem*>(dense_smem_raw);
  const int tid = threadIdx.x;
  load_log_table<32 * kDenseWarps>(&sm.ltab, tid);
  stage_check_init(sm.w[tid >> 5].stage, tid & 31);
  __syncthreads();
  const int warp = __shfl_sync(kFullMask, tid >> 5, 0), lane = tid & 31;
  DenseWarp& W = sm.w[warp];
  const long long n_items = a.P * (long long)v.n_slices;
  for (long long item = (long long)blockIdx.x * kDenseWarps + warp; item < n_items;
       item += (long long)gridDim.x * kDenseWarps) {
    const long long p = item / v.n_slices;
    const int s = (int)(item - p * v.n_slices);
    const long long row = a.row_index ? (long long)a.row_index[p] : p;
    const double* strike_row = v.strike + row * v.strike_stride;
    const int o_lo = v.slice_off[s], o_hi = v.slice_off[s + 1];
    __syncwarp();                                        // the previous item has left the warp's shared memory
    dense_prepare(W, v, a.params + kNumParams * p, a.transform, a.S0[row * a.s0_stride], v.slice_T[s], lane);
    __syncwarp();
    double* out_row = a.out + p * (long long)v.n_options;
    for (int c_lo = o_lo; c_lo < o_hi; c_lo += kDenseChunk) {
      const int cnt = min(kDenseChunk, o_hi - c_lo);
      const double u1 = u_one(W.pass);
      int n_bind = 0;
      for (int t0 = 0; t0 < cnt; t0 += 32) {              // warp-uniform trip count (the ballot needs every lane)
        const int t = t0 + lane;
        bool bind = false;
        if (t < cnt) {
          double K = strike_row[v.pos[c_lo + t]];
          if (v.scale_by_spot) K = K * W.S0 / 100.0;
          const StrikeConsts sc = make_strike_consts(K, W.S0);
          W.K[t] = sc.K; W.x[t] = sc.x; W.sex[t] = W.S0 * sc.ex;
          fm::sincos_(u1 * (sc.x - W.a0), &W.sth[t], &W.cth[t]);
          bind = ((sc.x - 0.1) < W.a0) || ((sc.x + 0.1) > W.b0);
          W.bind[t] = bind; W.call[t] = v.call[c_lo + t];
          W.part[t] = 0.0;
        }
        n_bind += __popc(__ballot_sync(kFullMask, bind));
      }
      __syncwarp();
      if (n_bind < cnt) dense_pass(W, cnt, v.n_cos, lane, &sm.ltab);
      if (n_bind > 0) {
        for (int t = 0; t < cnt; ++t) {
          if (!W.bind[t]) continue;                       // uniform: the flags live in shared memory
          __syncwarp();
          dense_pass_single(W, t, v.n_cos, lane, &sm.ltab);
        }
      }
      __syncwarp();
      for (int t = lane; t < cnt; t += 32) {
        DHJ_CHECK(v.pos[c_lo + t] >= 0 && v.pos[c_lo + t] < v.n_options && t < kDenseChunk, kChkOutputIndex);
        out_row[v.pos[c_lo + t]] = W.disc * W.part[t];
      }
      __syncwarp();
    }
  }
}

// Fused loss kernel on the batch engine (slices of <= 8 strikes, <= 32 slices): a "unit" is one loss evaluation
// (one x; in FD mode one of the 14 stencil points of an optimiser state); a block batch holds
// `units_per_batch` whole units (= units_per_batch * n_slices <= kPriceItems items), prices them as k_price_batch does,
// then one thread per unit forms mean(rel^2) + Feller / the 1e10 sentinel, and the thread that completes a
// state's 14th point assembles scipy's forward-difference gradient.
struct LossBatchArgs {
  const double* x;           // [B][13] (fd: [C][13]) unconstrained
  const int* market_index;   // optional, per x
  const double* S0;          // [n_markets]
  const double* market;      // [n_markets][M] caller order
  int fd;
  double h;
  long long n_units;         // B, or C*14
  int units_per_batch;
  double* f_all;             // [n_units]
  double* fg;                // fd: [C][14]
  unsigned int* counters;    // fd: [C]
};

__global__ void __launch_bounds__(kBatchThreads, DHJ_BATCH_MINB) k_loss_batch(SliceView v, LossBatchArgs a) {
  __shared__ PriceSmem sm;
  __shared__ double s_feller[kPriceItems];
  const int tid = threadIdx.x;
  load_log_table<kBatchThreads>(&sm.ltab, tid);
  stage_check_init(sm.stage[tid >> 5], tid & 31);
  const int nS = v.n_slices;
  const long long n_batches = (a.n_units + a.units_per_batch - 1) / a.units_per_batch;
  for (long long batch = blockIdx.x; batch < n_batches; batch += gridDim.x) {
    const long long base_unit = batch * a.units_per_batch;
    const int n_units_here = (int)min((long long)a.units_per_batch, a.n_units - base_unit);
    const int cnt_items = n_units_here * nS;
    // ---- phase 1 -----------------------------------------------------------------------------------
    if (tid < cnt_items) {
      const int ul = tid / nS, s = tid - ul * nS;
      const long long unit = base_unit + ul;
      const long long c = a.fd ? unit / kFdPoints : unit;
      const int var = a.fd ? (int)(unit - c * kFdPoints) : 0;
      double xv[kNumParams];
#pragma unroll
      for (int i = 0; i < kNumParams; ++i) xv[i] = a.x[kNumParams * c + i];
#pragma unroll
      for (int i = 0; i < kNumParams; ++i)
        if (var == i + 1) xv[i] = xv[i] + a.h;         // scipy's forward point x_i + h
      const Params m = transform_params(xv);
      const long long mi = a.market_index ? a.market_index[c] : 0;
      prepare_item(sm.items[tid], v, m, a.S0[mi], v.strike + mi * v.strike_stride, s, mi * (long long)v.n_options);
      tag_item(sm.items[tid], (unsigned long long)batch + 1);
      if (s == 0) s_feller[ul] = feller_penalty(m);
    }
    __syncthreads();
    // ---- phase 2 (as k_price_batch): prices -> shared memory, in the item's ex[] slots (exp(x_j) is dead once
    // the item's passes are done; only the warp that owns the item touches them) -----------------------------
    run_batch(sm, v, cnt_items, tid, (unsigned long long)batch + 1, [&](int i, int j, const ItemRec&, double price) {
      DHJ_CHECK(i >= 0 && i < kPriceItems && j >= 0 && j < kBatchMaxStrikes, kChkSharedIndex);
      sm.items[i].ex[j] = price;
    });
    __syncthreads();
    // ---- phase 4: one thread per unit: loss, and the gradient when a state's stencil is complete ----------
    if (tid < n_units_here) {
      const long long unit = base_unit + tid;
      const long long c = a.fd ? unit / kFdPoints : unit;
      double sq = 0.0;
      bool bad = false;
      for (int s = 0; s < nS; ++s) {
        const ItemRec& it = sm.items[tid * nS + s];
        const double* market_row = a.market + it.out_row;           // out_row = market index * M
        const int cnt = __popc(it.valid_mask);
        for (int j = 0; j < cnt; ++j) {
          const double price = it.ex[j];
          if (!(price > 0.0) || isinf(price)) bad = true;           // lbfgs_calibrator.py:152
          const double mk = market_row[v.pos[it.o_lo + j]];
          const double rel = (price - mk) / mk;                     // :163
          sq += rel * rel;
        }
      }
      const double loss = bad ? kSentinel : sq / (double)v.n_options + s_feller[tid];   // :164-169
      a.f_all[unit] = loss;
      if (a.fd) {
        __threadfence();
        const unsigned prev = atomicAdd(&a.counters[c], 1u);
        if (prev == (unsigned)(kFdPoints - 1)) {
          __threadfence();
          const double* f = a.f_all + kFdPoints * c;
          const double f0 = __ldcg(f);
          a.fg[kFdPoints * c] = f0;
          for (int i = 0; i < kNumParams; ++i) {
            const double xi = a.x[kNumParams * c + i];
            const double dx = (xi + a.h) - xi;
            a.fg[kFdPoints * c + 1 + i] = (__ldcg(f + 1 + i) - f0) / dx;
          }
          a.counters[c] = 0u;
        }
      }
    }
    __syncthreads();
  }
}

// General loss path (slices with more than 8 strikes or more than 32 slices, or a large batch): k_fd_expand builds the
// stencil points and transforms them to model parameters ONCE per loss evaluation (exp / tanh of the calibrator; the
// pricing kernel then runs without its per-item transform), k_price_batch / k_price_dense price them, k_loss_reduce
// forms the losses and gradients.
__global__ void k_fd_expand(const double* __restrict__ x, const int* __restrict__ market_index, long long n_x, int fd,
                            double h, double* __restrict__ pv, int* __restrict__ row_index) {
  const long long unit = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int per = fd ? kFdPoints : 1;
  if (unit >= n_x * per) return;
  const long long c = unit / per;
  const int var = (int)(unit - c * per);
  double xv[kNumParams];
#pragma unroll
  for (int i = 0; i < kNumParams; ++i) {
    const double xi = x[kNumParams * c + i];
    xv[i] = (var == i + 1) ? xi + h : xi;          // scipy's forward point x_i + h
  }
  const Params m = transform_params(xv);
  double* out = pv + kNumParams * unit;
  out[0] = m.v0[0]; out[1] = m.kappa[0]; out[2] = m.theta[0]; out[3] = m.sigma[0]; out[4] = m.rho[0];
  out[5] = m.v0[1]; out[6] = m.kappa[1]; out[7] = m.theta[1]; out[8] = m.sigma[1]; out[9] = m.rho[1];
  out[10] = m.lam; out[11] = m.mu; out[12] = m.sj;
  row_index[unit] = market_index ? market_index[c] : 0;
}

// (options are visited in slice order, pos[i], exactly as k_loss_batch does: the two paths give the same bits)
__global__ void k_loss_reduce(const double* __restrict__ prices, const double* __restrict__ pv,
                              const int* __restrict__ row_index, const double* __restrict__ market,
                              const int* __restrict__ pos, int M,
                              long long n_x, int fd, double h, const double* __restrict__ x,
                              double* __restrict__ f_all, double* __restrict__ fg) {
  const long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= n_x) return;
  const int per = fd ? kFdPoints : 1;
  double f0 = 0.0;
  for (int var = 0; var < per; ++var) {
    const long long unit = c * per + var;
    const double* pr = prices + unit * M;
    const double* mk = market + (long long)row_index[unit] * M;
    double sq = 0.0;
    bool bad = false;
    for (int i = 0; i < M; ++i) {
      const int o = pos[i];
      const double price = pr[o];
      if (!(price > 0.0) || isinf(price)) bad = true;
      const double rel = (price - mk[o]) / mk[o];
      sq += rel * rel;
    }
    const Params m = load_params(pv + kNumParams * unit);
    const double loss = bad ? kSentinel : sq / (double)M + feller_penalty(m);
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

// ---- the remaining public methods of DoubleHeston, one thread per element ----------------------
// characteristic_function(phi, tau) for n frequencies of one parameter set (double_heston.py:48-97)
__global__ void k_cf(const double* __restrict__ params, double r, double q, double tau,
                     const double* __restrict__ u_in, int n, double* __restrict__ out_re,
                     double* __restrict__ out_im) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Params m = load_params(params);
  const SetConsts s = make_set_consts(m, r, q);
  const double u = u_in[i];
  double xr, xi;
  cf_exponent(s, u, tau, s.lam * tau, &fm::kTables, &xr, &xi);
  double sn, cs;
  fm::sincos_(xi, &sn, &cs);
  const double mag = fm::exp_(xr);
  out_re[i] = mag * cs;
  out_im[i] = mag * sn;
}

// characteristic_function(phi, tau) for COMPLEX phi (the reference's ufunc arithmetic accepts it, double_heston.py:48-97;
// nothing on the pricing path needs it).  Plain complex arithmetic in the reference's own operation order — Smith's
// division as NumPy does it, glibc-style csqrt, libdevice exp / log / sincos / atan2 — one thread per frequency.
struct Cx { double re, im; };
__device__ __forceinline__ Cx cx_add(Cx a, Cx b) { return {a.re + b.re, a.im + b.im}; }
__device__ __forceinline__ Cx cx_sub(Cx a, Cx b) { return {a.re - b.re, a.im - b.im}; }
__device__ __forceinline__ Cx cx_mul(Cx a, Cx b) { return {a.re * b.re - a.im * b.im, a.re * b.im + a.im * b.re}; }
__device__ __forceinline__ Cx cx_scale(Cx a, double f) { return {a.re * f, a.im * f}; }
__device__ __forceinline__ Cx cx_div(Cx a, Cx b) {
  if (fabs(b.re) >= fabs(b.im)) {
    const double rat = b.im / b.re, scl = 1.0 / (b.re + b.im * rat);
    return {(a.re + a.im * rat) * scl, (a.im - a.re * rat) * scl};
  }
  const double rat = b.re / b.im, scl = 1.0 / (b.re * rat + b.im);
  return {(a.re * rat + a.im) * scl, (a.im * rat - a.re) * scl};
}
__device__ __forceinline__ Cx cx_sqrt(Cx z) {
  const double h = hypot(z.re, z.im);
  if (h == 0.0) return {0.0, z.im};
  if (z.re > 0.0) { const double t = sqrt(0.5 * (h + z.re)); return {t, 0.5 * (z.im / t)}; }
  const double t = sqrt(0.5 * (h - z.re));
  return {fabs(0.5 * (z.im / t)), copysign(t, z.im)};
}
__device__ __forceinline__ Cx cx_exp(Cx z) {
  double sn, cs;
  sincos(z.im, &sn, &cs);
  const double e = exp(z.re);
  return {e * cs, e * sn};
}
__device__ __forceinline__ Cx cx_log(Cx z) { return {log(hypot(z.re, z.im)), atan2(z.im, z.re)}; }

__global__ void k_cf_complex(const double* __restrict__ params, double r, double q, double tau,
                             const double* __restrict__ u_re, const double* __restrict__ u_im, int n,
                             double* __restrict__ out_re, double* __restrict__ out_im) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Params m = load_params(params);
  const Cx u = {u_re[i], u_im[i]};
  const Cx iu = {-u.im, u.re};                                           // i u
  const Cx one = {1.0, 0.0};
  const double comp = exp(m.mu + 0.5 * m.sj * m.sj) - 1.0;               // :82
  Cx A = cx_scale(iu, (r - q - m.lam * comp) * tau);                     // :83
  Cx BV = {0.0, 0.0};
  const Cx uu = cx_mul(u, Cx{u.re, u.im + 1.0});                         // u (u + i)
  for (int j = 0; j < 2; ++j) {
    const double s2 = m.sigma[j] * m.sigma[j];
    const Cx beta = {m.kappa[j] - m.rho[j] * m.sigma[j] * iu.re, -(m.rho[j] * m.sigma[j]) * iu.im};   // :64, :73
    const Cx d = cx_sqrt(cx_add(cx_mul(beta, beta), cx_scale(uu, s2)));                                 // :65, :74
    const Cx bm = cx_sub(beta, d);
    const Cx g = cx_div(bm, cx_add(beta, d));                                                           // :67, :76
    const Cx E = cx_exp(cx_scale(d, -tau));
    const Cx one_gE = cx_sub(one, cx_mul(g, E));
    const Cx B = cx_mul(cx_scale(bm, 1.0 / s2), cx_div(cx_sub(one, E), one_gE));                        // :70-71, :79-80
    const Cx lg = cx_log(cx_div(one_gE, cx_sub(one, g)));
    A = cx_add(A, cx_scale(cx_sub(cx_scale(bm, tau), cx_scale(lg, 2.0)), m.kappa[j] * m.theta[j] / s2));   // :85-91
    BV = cx_add(BV, cx_scale(B, m.v0[j]));
  }
  const Cx je = cx_exp(cx_sub(cx_scale(iu, m.mu), cx_scale(cx_mul(u, u), 0.5 * m.sj * m.sj)));
  const Cx cf_jump = cx_exp(cx_scale(cx_sub(je, one), m.lam * tau));                                    // :93
  const Cx cf = cx_mul(cx_exp(cx_add(A, BV)), cf_jump);                                                  // :94-96
  out_re[i] = cf.re;
  out_im[i] = cf.im;
}

// truncationRange(L) for P parameter sets x M (S0, K, T) triples (double_heston.py:100-139)
__global__ void k_truncation_range(const double* __restrict__ params, long long P, const double* __restrict__ S0,
                                   long long s0_stride, const double* __restrict__ strike,
                                   const double* __restrict__ maturity, int M, double r, double L,
                                   double* __restrict__ out_ab) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P * M) return;
  const long long p = i / M;
  const int o = (int)(i - p * M);
  const Params m = load_params(params + kNumParams * p);
  double a0, b0;
  truncation_range(m, maturity[o], r, L, &a0, &b0);
  const double x = fm::log_ratio(strike[o], S0[p * s0_stride]);
  out_ab[2 * i] = py_min(a0, x - 0.1);
  out_ab[2 * i + 1] = py_max(b0, x + 0.1);
}

// chi_k, psi_k for n values of k (double_heston.py:141-158)
__global__ void k_chi_psi(const int* __restrict__ k_in, int n, double c, double d, double a, double b,
                          double* __restrict__ chi, double* __restrict__ psi) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int k = k_in[i];
  const double ed = fm::exp_(d), ec = fm::exp_(c);
  if (k == 0) { chi[i] = ed - ec; psi[i] = d - c; return; }
  const double u = fm::div((double)k * kPi, b - a);
  double sd, cd, sc, cc;
  fm::sincos_(u * (d - a), &sd, &cd);
  fm::sincos_(u * (c - a), &sc, &cc);
  chi[i] = fm::rcp(1.0 + u * u) * (((cd * ed - cc * ec) + (u * sd) * ed) - (u * sc) * ec);
  psi[i] = fm::rcp(u) * (sd - sc);
}

// 8 independent FMA chains per thread; 2 flop per FMA.  Two operand forms: all three operands from vector registers
// (`DFMA R, R, R, R`: the register file caps this form at ~92 % of the pipe's rate on B200), and one multiplicand
// from a uniform register (`DFMA R, R, UR, R`: the pipe's own rate, 64 FMA/clk/SM).  The addend is made
// thread-dependent in the second form so that ptxas keeps only the multiplicand uniform.
constexpr int kPeakChains = 8;
constexpr int kPeakUnroll = 8;
template <bool UNIFORM>
__global__ void __launch_bounds__(256) k_fp64_peak(double* out, int iters, double x, double y) {
  double acc[kPeakChains];
  const double yv = UNIFORM ? y * (double)(threadIdx.x + 1) : y;
#pragma unroll
  for (int j = 0; j < kPeakChains; ++j) acc[j] = 1.0 + 1e-3 * (double)(threadIdx.x + j);
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int r = 0; r < kPeakUnroll; ++r) {
#pragma unroll
      for (int j = 0; j < kPeakChains; ++j) acc[j] = fma(acc[j], x, yv);
    }
  }
  double s = 0.0;
#pragma unroll
  for (int j = 0; j < kPeakChains; ++j) s += acc[j];
  out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

}  // namespace dhj
