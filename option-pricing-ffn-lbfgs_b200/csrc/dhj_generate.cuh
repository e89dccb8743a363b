// dhj_generate.cuh — device-resident synthetic dataset sweep (SURVEY §2 "K3", BASELINE config C4): everything
// /root/reference/src/data/synthetic_generator.py:98-157 does per sample, without a host round trip.
//
// The reference draws from ONE sequential NumPy stream (13 uniforms, [1 normal], 15 normals per sample) — kept,
// bit for bit, by dhj_draws.cpp for seeded drop-in runs.  A 100 M-sample sweep sharded over GPUs needs draws that
// are a function of the SAMPLE INDEX only, so that a shard does not depend on how many ranks there are.  This
// file defines that stream ("counter stream", spec below; restated by the test suite's CPU checker):
//
//   generator   Philox4x32-10 (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy as 1, 2, 3", SC'11),
//               key = (seed low word, seed high word), counter = (i low, i high, slot, 0x44484A31) for sample i;
//               the four output words give two 64-bit words w0 = x0 | x1 << 32, w1 = x2 | x3 << 32
//   uniform     U(w) = (w >> 11) * 2^-53 in [0, 1)
//   normal pair u1 = ((w0 >> 11) + 1) * 2^-53 in (0, 1], u2 = U(w1);  R = sqrt(-2 ln u1);
//               z0 = R cos(2 pi u2), z1 = R sin(2 pi u2)                                   (Box-Muller)
//   sample i    belongs to path q = i / path_len at step t = i % path_len; a path is one reference-style history
//               (synthetic_generator.py:98-116):
//     slots 0..6   raw_j = lo_j + (hi_j - lo_j) * U(word j % 2 of slot j / 2), j = 0..12      (:100-102)
//                  p_j(t) = raw_j at t = 0, else persistence * p_j(t-1) + (1 - persistence) * raw_j   (:105-109)
//     slot 7       ret = ret_mean + ret_sd * z0;  spot(0) = spot0, spot(t) = spot(t-1) * (1 + ret)    (:112-116)
//     slots 8..    noise_m = noise_sd * z_{m % 2} of slot 8 + m / 2, m = 0..n_options-1             (:141)
//   prices       K = K_rel * spot / 100, call, r (:123-138) — the pricing kernel (k_price_batch / k_price_dense)
//   market       model + noise * model (:141-142);  loss = mean(((model - market) / market)^2) (:154-157)
//
// Kernels: k_gen_draws (a warp per path: the 32 lanes draw 32 consecutive steps in parallel, lanes 0..13 then
// advance the 14 recurrences through them; rows leave the warp coalesced) -> pricing kernel -> k_gen_market
// (HBM-bound epilogue: a block stages 128 samples' prices through shared memory, one thread per sample draws the
// noise, forms market prices and the sample's loss; coalesced in and out).
#pragma once
#include <stdint.h>

#include "dhj_math.cuh"

namespace dhj {

constexpr uint32_t kPhiloxM0 = 0xD2511F53u, kPhiloxM1 = 0xCD9E8D57u;
constexpr uint32_t kPhiloxW0 = 0x9E3779B9u, kPhiloxW1 = 0xBB67AE85u;
constexpr uint32_t kStreamTag = 0x44484A31u;   // "DHJ1": fourth counter word of every draw of this stream

struct Philox4 { uint32_t x[4]; };

DHJ_HD Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int round = 0; round < 10; ++round) {
    const uint64_t p0 = (uint64_t)kPhiloxM0 * c0, p1 = (uint64_t)kPhiloxM1 * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += kPhiloxW0; k1 += kPhiloxW1;
  }
  Philox4 r;
  r.x[0] = c0; r.x[1] = c1; r.x[2] = c2; r.x[3] = c3;
  return r;
}

// the two 64-bit words of (sample i, slot)
DHJ_HD void counter_words(uint64_t seed, uint64_t i, uint32_t slot, uint64_t* w0, uint64_t* w1) {
  const Philox4 r = philox4x32_10((uint32_t)i, (uint32_t)(i >> 32), slot, kStreamTag, (uint32_t)seed,
                                  (uint32_t)(seed >> 32));
  *w0 = (uint64_t)r.x[0] | ((uint64_t)r.x[1] << 32);
  *w1 = (uint64_t)r.x[2] | ((uint64_t)r.x[3] << 32);
}

DHJ_HD double counter_uniform(uint64_t w) { return (double)(w >> 11) * 1.1102230246251565e-16; }          // 2^-53
DHJ_HD double counter_uniform_open0(uint64_t w) { return (double)((w >> 11) + 1) * 1.1102230246251565e-16; }

// Box-Muller pair of two stream words.  The library's own branch-free log / sqrt / sincos (dhj_fastmath.cuh,
// <= 1-2 ulp): with libdevice's the noise epilogue was bound by their instruction count at 2.5 TB/s, 38 % of the HBM
// rate.  Host-compilable, so that the test suite's g++ emulations run the device's arithmetic.
DHJ_HD void box_muller(uint64_t w0, uint64_t w1, double* z0, double* z1) {
  const double R = fm::sqrt_(-2.0 * fm::log_(counter_uniform_open0(w0)));
  double sn, cs;
  fm::sincos_(6.283185307179586 * counter_uniform(w1), &sn, &cs);
  *z0 = R * cs; *z1 = R * sn;
}

#if defined(__CUDACC__)

// Box-Muller pair of (sample i, slot)
__device__ __forceinline__ void counter_normal_pair(uint64_t seed, uint64_t i, uint32_t slot, double* z0, double* z1) {
  uint64_t w0, w1;
  counter_words(seed, i, slot, &w0, &w1);
  box_muller(w0, w1, z0, z1);
}

struct GenArgs {
  uint64_t seed;
  long long first, n;            // samples [first, first + n) of the stream
  int path_len;
  double lo[kNumParams], range[kNumParams];     // range = hi - lo
  double persistence, spot0, ret_mean, ret_sd, noise_sd;
};

constexpr int kGenWarps = 4;
constexpr int kGenCols = kNumParams + 1;       // 13 parameters + the spot return / spot

// A warp per path.  Output rows are relative to `first`: params[(i - first)][13], spots[i - first].
__global__ void __launch_bounds__(32 * kGenWarps) k_gen_draws(GenArgs a, double* __restrict__ params,
                                                              double* __restrict__ spots) {
  __shared__ double sh[kGenWarps][32][kGenCols];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long q_first = a.first / a.path_len, q_last = (a.first + a.n - 1) / a.path_len;
  const long long q = q_first + (long long)blockIdx.x * kGenWarps + warp;
  if (q > q_last) return;
  const long long i0 = q * a.path_len;
  // steps of this path that anybody asked for: [0, t_end)
  const int t_end = (int)min((long long)a.path_len, a.first + a.n - i0);
  double (*buf)[kGenCols] = sh[warp];
  double state = 0.0;                            // lane j < 13: parameter j; lane 13: spot
  const double one_minus = 1.0 - a.persistence;
  for (int t0 = 0; t0 < t_end; t0 += 32) {
    const int t = t0 + lane;
    const uint64_t i = (uint64_t)(i0 + t);
    // the expensive part, one step per lane: 7 generator calls for the parameters, one normal pair for the return
#pragma unroll
    for (int s = 0; s < 7; ++s) {
      uint64_t w0, w1;
      counter_words(a.seed, i, (uint32_t)s, &w0, &w1);
      buf[lane][2 * s] = a.lo[2 * s] + a.range[2 * s] * counter_uniform(w0);
      if (2 * s + 1 < kNumParams) buf[lane][2 * s + 1] = a.lo[2 * s + 1] + a.range[2 * s + 1] * counter_uniform(w1);
    }
    double z0, z1;
    counter_normal_pair(a.seed, i, 7u, &z0, &z1);
    buf[lane][kNumParams] = a.ret_mean + a.ret_sd * z0;
    __syncwarp();
    // the recurrences, one column per lane
    if (lane < kGenCols) {
      const int steps = min(32, t_end - t0);
      for (int s = 0; s < steps; ++s) {
        const double v = buf[s][lane];
        if (t0 + s == 0) state = (lane < kNumParams) ? v : a.spot0;
        else state = (lane < kNumParams) ? a.persistence * state + one_minus * v : state * (1.0 + v);
        buf[s][lane] = state;
      }
    }
    __syncwarp();
    // rows out: the 32 x 13 parameter block is contiguous in global memory
    const long long row0 = i0 + t0 - a.first;      // may be negative: steps before `first` are not written
    const int steps = min(32, t_end - t0);
    for (int e = lane; e < steps * kNumParams; e += 32) {
      const int s = e / kNumParams, j = e - s * kNumParams;
      if (row0 + s >= 0) params[(row0 + s) * kNumParams + j] = buf[s][j];
    }
    if (lane < steps && row0 + lane >= 0) spots[row0 + lane] = buf[lane][kNumParams];
    __syncwarp();
  }
}

// market = model + noise * model and the per-sample loss.  M options per sample (M <= kGenMaxOptions); a block
// stages kGenMarketSamples rows through shared memory so that global loads and stores are coalesced.
constexpr int kGenMarketSamples = 128;
constexpr int kGenMaxOptions = 32;

__global__ void __launch_bounds__(kGenMarketSamples) k_gen_market(uint64_t seed, long long first, long long n, int M,
                                                                  double noise_sd, const double* __restrict__ model,
                                                                  double* __restrict__ market,
                                                                  double* __restrict__ loss) {
  extern __shared__ double rows[];                 // [kGenMarketSamples][M | 1]: odd row pitch, no bank conflicts
  const int pitch = M | 1;
  const long long base = (long long)blockIdx.x * kGenMarketSamples;
  const int cnt = (int)min((long long)kGenMarketSamples, n - base);
  // element e = tid, tid + 128, ... of the block's cnt x M tile sits at (row, col) = (e / M, e % M): one division per
  // thread, then (row, col) advance by (128 / M, 128 % M) with a carry
  const int step_row = kGenMarketSamples / M, step_col = kGenMarketSamples % M;
  {
    int row = threadIdx.x / M, col = threadIdx.x - row * M;
    for (int e = threadIdx.x; e < cnt * M; e += kGenMarketSamples) {
      rows[row * pitch + col] = model[base * M + e];
      row += step_row; col += step_col;
      if (col >= M) { col -= M; ++row; }
    }
  }
  __syncthreads();
  if (threadIdx.x < cnt) {
    double* row = rows + threadIdx.x * pitch;
    const uint64_t i = (uint64_t)(first + base + threadIdx.x);
    double sq = 0.0;
    for (int m = 0; m < M; m += 2) {
      double z[2];
      counter_normal_pair(seed, i, 8u + (uint32_t)(m >> 1), &z[0], &z[1]);
#pragma unroll
      for (int h = 0; h < 2; ++h)
        if (m + h < M) {
          const double price = row[m + h];
          const double mk = price + (noise_sd * z[h]) * price;          // synthetic_generator.py:141-142
          const double rel = fm::div(price - mk, mk);                     // :154
          sq += rel * rel;
          row[m + h] = mk;
        }
    }
    loss[base + threadIdx.x] = sq / (double)M;                            // :155 (np.mean)
  }
  __syncthreads();
  int row = threadIdx.x / M, col = threadIdx.x - row * M;
  for (int e = threadIdx.x; e < cnt * M; e += kGenMarketSamples) {
    market[base * M + e] = rows[row * pitch + col];
    row += step_row; col += step_col;
    if (col >= M) { col -= M; ++row; }
  }
}

#endif  // __CUDACC__

}  // namespace dhj
