// dhj_mc.cuh — Monte Carlo pricing of path-dependent options (Asian, discretely monitored barriers) under the model
// whose characteristic function the COS kernels price: two independent Heston variance factors and Merton jumps.
//
// Model (calibrator order v0_j, kappa_j, theta_j, sigma_j, rho_j for j = 1, 2, then lambda, mu_J, sigma_J):
//   dv_j = kappa_j (theta_j - v_j) dt + sigma_j sqrt(v_j) dZ_j,  corr(dW_j, dZ_j) = rho_j, the factors independent;
//   d ln S = (r - q - lambda kbar - (v_1 + v_2) / 2) dt + sqrt(v_1) dW_1 + sqrt(v_2) dW_2 + dJ,
//   kbar = e^{mu_J + sigma_J^2 / 2} - 1, J compound Poisson (intensity lambda) with N(mu_J, sigma_J^2) log-jumps.
//
// Scheme: n_steps equal steps dt = T / n_steps; full-truncation Euler for the variances (Lord, Koekkoek, van Dijk,
// "A comparison of biased simulation schemes for stochastic volatility models", Quant. Finance 10 (2010)), log-Euler
// for the spot.  With v+ = (v < 0 ? 0 : v) (a NaN stays NaN) and both updates from the start of the step:
//   x   += (r - q - lambda kbar - (v1+ + v2+) / 2) dt + sqrt(v1+ dt)(rho1 Z1 + sqrt(1 - rho1^2) Z1p)
//                                                    + sqrt(v2+ dt)(rho2 Z2 + sqrt(1 - rho2^2) Z2p) + J
//   v_j += kappa_j (theta_j - v_j+) dt + sigma_j sqrt(v_j+ dt) Z_j
//   J    = N mu_J + sigma_J sqrt(N) z,  N ~ Poisson(lambda dt)  (J = 0 when N = 0)
// Given the start of a step, E[e^{dx}] = e^{(r - q) dt}: the diffusion part is lognormal and E[e^J] = e^{lambda kbar dt},
// so e^{-(r-q)t} S_t is an exact martingale of the scheme.  The variance is discretised, so prices are not unbiased
// estimates of the continuous-time price (the bias at the generator's parameters is measured in DESIGN.md §6f).
//
// Random stream ("DHJ2"; restated in NumPy by the test suite):
//   generator   Philox4x32-10, key = (seed low word, seed high word),
//               counter = (path low word, path high word, 4 step + j, 0x44484A32); the generator's stream
//               (dhj_generate.cuh) uses the tag 0x44484A31, so the two never share a counter
//   words       w0 = x0 | x1 << 32, w1 = x2 | x3 << 32; U(w) and the Box-Muller pair as in dhj_generate.cuh
//   j = 0       Box-Muller pair (w0, w1) -> (Z1, Z1p)
//   j = 1       Box-Muller pair (w0, w1) -> (Z2, Z2p)
//   j = 2       U = U(w0); N = the smallest n with U < F(n), F the Poisson(lambda dt) CDF summed in order
//               (p_0 = e^{-lambda dt}, p_n = p_{n-1} lambda dt / n), capped at kMcMaxJumps
//   j = 3       drawn only when N > 0: z = z0 of its Box-Muller pair
// Draws depend on (seed, path, step) only, never on the parameter set: every set of a call sees the same numbers.
//
// Path statistics: n_obs divides n_steps; observations at the ends of steps i n_steps / n_obs, i = 1..n_obs (S0 is not
// one).  A path keeps S_T = S0 e^x, the sum, the maximum and the minimum of S at the observations; every payoff is a
// function of these four, so a path's registers do not grow with the number of options:
//   vanilla(X) = max(+-(X - K), 0) (a NaN stays NaN);  EUROPEAN vanilla(S_T), ASIAN vanilla(sum / n_obs),
//   UP_OUT vanilla(S_T) [max < B], UP_IN [max >= B], DOWN_OUT [min > B], DOWN_IN [min <= B]  (the indicator multiplies).
//
// Kernels: k_mc_paths — one path per thread, one block per chunk of kMcChunk consecutive paths of one parameter set;
// the option table sits in shared memory; at the end of the path every thread forms its M payoffs and the block
// reduces them per option into the chunk's (mean, M2) in a fixed order (xor-butterfly per warp, lane 0's sum, the warps
// in order; two passes: the mean, then the squared deviations from it).  k_mc_finalize — one thread per (set, option)
// combines the chunk partials in chunk order (Chan, Golub, LeVeque pairwise update), carrying (n, mean, M2) in global
// memory from one launch to the next when the host splits a set's chunks, so the result has the same bits however the
// call is cut; the last launch writes price = e^{-rT} mean and stderr = e^{-rT} sqrt(M2 / (n - 1) / n).
#pragma once
#include <stdint.h>

#include "dhj_generate.cuh"
#if defined(__CUDACC__)
#include "dhj_engine.cuh"
#endif

namespace dhj {
namespace mc {

constexpr uint32_t kMcStreamTag = 0x44484A32u;   // "DHJ2"
constexpr int kMcMaxJumps = 64;                  // cap of the Poisson inversion
constexpr int kMcMaxOptions = 64;                // options per call (the shared option table)
constexpr int kMcMaxSteps = 1 << 28;             // 4 step + 3 fits the 32-bit counter word
constexpr int kMcChunk = 256;                    // paths per block = threads per block
constexpr int kMcWarps = kMcChunk / 32;

enum McKind { kEuropean = 0, kAsian = 1, kUpOut = 2, kUpIn = 3, kDownOut = 4, kDownIn = 5, kMcKinds = 6 };

// the two 64-bit words of (path, 4 step + j)
DHJ_HD void mc_words(uint64_t seed, uint64_t path, uint32_t ctr, uint64_t* w0, uint64_t* w1) {
  const Philox4 r = philox4x32_10((uint32_t)path, (uint32_t)(path >> 32), ctr, kMcStreamTag, (uint32_t)seed,
                                  (uint32_t)(seed >> 32));
  *w0 = (uint64_t)r.x[0] | ((uint64_t)r.x[1] << 32);
  *w1 = (uint64_t)r.x[2] | ((uint64_t)r.x[3] << 32);
}

// smallest n with U < F(n) for the Poisson(lam_dt) CDF F, p0 = e^{-lam_dt}; capped at kMcMaxJumps (a NaN stops at 0)
DHJ_HD int poisson_inverse(double U, double p0, double lam_dt) {
  double p = p0, F = p0;
  int n = 0;
  while (n < kMcMaxJumps && U >= F) {
    ++n;
    p = (p * lam_dt) / (double)n;
    F += p;
  }
  return n;
}

// per-set constants of the scheme
struct McSet {
  double v0[2], kappa[2], theta[2], sigma[2], rho[2], rhob[2];   // rhob = sqrt(1 - rho^2)
  double mu, sj;
  double drift;     // r - q - lambda kbar
  double lam_dt;    // lambda dt
  double p0;        // e^{-lambda dt}
  double dt;
};

DHJ_HD McSet make_mc_set(const double* __restrict__ p, double r, double q, double dt) {
  McSet s;
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    s.v0[j] = p[5 * j]; s.kappa[j] = p[5 * j + 1]; s.theta[j] = p[5 * j + 2]; s.sigma[j] = p[5 * j + 3];
    s.rho[j] = p[5 * j + 4];
    s.rhob[j] = fm::sqrt_(1.0 - s.rho[j] * s.rho[j]);
  }
  const double lam = p[10];
  s.mu = p[11]; s.sj = p[12];
  const double kbar = fm::exp_(s.mu + 0.5 * s.sj * s.sj) - 1.0;
  s.drift = r - q - lam * kbar;
  s.dt = dt;
  s.lam_dt = lam * dt;
  s.p0 = fm::exp_(-s.lam_dt);
  return s;
}

struct McState { double x, v1, v2; };

// one step of the scheme for path `path` at step `step`
DHJ_HD void mc_step(const McSet& s, uint64_t seed, uint64_t path, int step, McState* st) {
  const uint32_t c = 4u * (uint32_t)step;
  uint64_t w0, w1;
  double z1, z1p, z2, z2p;
  mc_words(seed, path, c, &w0, &w1);
  box_muller(w0, w1, &z1, &z1p);
  mc_words(seed, path, c + 1u, &w0, &w1);
  box_muller(w0, w1, &z2, &z2p);
  mc_words(seed, path, c + 2u, &w0, &w1);
  const int N = poisson_inverse(counter_uniform(w0), s.p0, s.lam_dt);
  double J = 0.0;
  if (N > 0) {
    double zj, unused;
    mc_words(seed, path, c + 3u, &w0, &w1);
    box_muller(w0, w1, &zj, &unused);
    const double n = (double)N;
    J = n * s.mu + (s.sj * fm::sqrt_(n)) * zj;
  }
  const double a1 = (st->v1 < 0.0) ? 0.0 : st->v1;
  const double a2 = (st->v2 < 0.0) ? 0.0 : st->v2;
  const double sq1 = fm::sqrt_(a1 * s.dt), sq2 = fm::sqrt_(a2 * s.dt);
  st->x += (s.drift - 0.5 * (a1 + a2)) * s.dt + sq1 * (s.rho[0] * z1 + s.rhob[0] * z1p) +
           sq2 * (s.rho[1] * z2 + s.rhob[1] * z2p) + J;
  st->v1 += (s.kappa[0] * (s.theta[0] - a1)) * s.dt + (s.sigma[0] * sq1) * z1;
  st->v2 += (s.kappa[1] * (s.theta[1] - a2)) * s.dt + (s.sigma[1] * sq2) * z2;
}

struct PathStats { double ST, sum, mx, mn; };

// the whole path: n_steps steps, observations every n_steps / n_obs steps
DHJ_HD PathStats mc_path(const McSet& s, double S0, uint64_t seed, uint64_t path, int n_steps, int n_obs) {
  McState st{0.0, s.v0[0], s.v0[1]};
  const int every = n_steps / n_obs;
  PathStats ps{0.0, 0.0, -INFINITY, INFINITY};
  int step = 0;
  for (int i = 0; i < n_obs; ++i) {
    for (int k = 0; k < every; ++k, ++step) mc_step(s, seed, path, step, &st);
    ps.ST = S0 * fm::exp_(st.x);
    ps.sum += ps.ST;
    ps.mx = (ps.ST > ps.mx) ? ps.ST : ps.mx;
    ps.mn = (ps.ST < ps.mn) ? ps.ST : ps.mn;
  }
  return ps;
}

// payoff of one option on a path; avg = sum / n_obs
DHJ_HD double mc_payoff(int kind, int call, double K, double B, const PathStats& ps, double avg) {
  const double X = (kind == kAsian) ? avg : ps.ST;
  const double d = call ? X - K : K - X;
  const double v = (d < 0.0) ? 0.0 : d;
  bool in = true;
  if (kind == kUpOut) in = ps.mx < B;
  else if (kind == kUpIn) in = ps.mx >= B;
  else if (kind == kDownOut) in = ps.mn > B;
  else if (kind == kDownIn) in = ps.mn <= B;
  return v * (in ? 1.0 : 0.0);
}

// paths of chunk c of a set of n_paths
DHJ_HD int chunk_paths(long long n_paths, long long c) {
  const long long rem = n_paths - c * kMcChunk;
  return (int)(rem < kMcChunk ? rem : kMcChunk);
}

#if defined(__CUDACC__)

struct McArgs {
  const double* params;            // [sets][13] of this launch
  const double* S0;                // [sets] (s0_stride 1) or [1] (0)
  long long s0_stride;
  const int* opt;                  // [M][2]: kind, is_call
  const double* opt_kb;            // [M][2]: strike, barrier
  double r, q, dt;
  int n_steps, n_obs, M;
  uint64_t seed;
  long long n_paths;
  long long chunk0, chunks;        // chunks [chunk0, chunk0 + chunks) of each set
  int sets;
  double2* partial;                // [sets][chunks][M]: (mean, M2) of each chunk
};

__global__ void __launch_bounds__(kMcChunk) k_mc_paths(McArgs a) {
  __shared__ int s_opt[kMcMaxOptions][2];
  __shared__ double s_kb[kMcMaxOptions][2];
  __shared__ double s_red[kMcWarps][kMcMaxOptions];
  __shared__ double s_mean[kMcMaxOptions];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long set = (long long)blockIdx.x / a.chunks, cl = (long long)blockIdx.x - set * a.chunks;
  const long long c = a.chunk0 + cl;
  for (int m = tid; m < a.M; m += kMcChunk) {
    DHJ_CHECK(m < kMcMaxOptions, kChkSharedIndex);
    s_opt[m][0] = a.opt[2 * m]; s_opt[m][1] = a.opt[2 * m + 1];
    s_kb[m][0] = a.opt_kb[2 * m]; s_kb[m][1] = a.opt_kb[2 * m + 1];
  }
  const int cnt = chunk_paths(a.n_paths, c);
  const bool active = tid < cnt;
  PathStats ps{0.0, 0.0, 0.0, 0.0};
  double avg = 0.0;
  if (active) {
    const McSet s = make_mc_set(a.params + set * kNumParams, a.r, a.q, a.dt);
    const double S0 = a.S0[set * a.s0_stride];
    ps = mc_path(s, S0, a.seed, (uint64_t)(c * kMcChunk + tid), a.n_steps, a.n_obs);
    avg = ps.sum / (double)a.n_obs;
  }
  __syncthreads();
  // pass 1: the chunk mean of each option
  for (int m = 0; m < a.M; ++m) {
    DHJ_CHECK(m < kMcMaxOptions, kChkSharedIndex);
    const double v = active ? mc_payoff(s_opt[m][0], s_opt[m][1], s_kb[m][0], s_kb[m][1], ps, avg) : 0.0;
    const double w = warp_sum(v);
    if (lane == 0) s_red[warp][m] = w;
  }
  __syncthreads();
  if (tid < a.M) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < kMcWarps; ++w) t += s_red[w][tid];
    s_mean[tid] = t / (double)cnt;
  }
  __syncthreads();
  // pass 2: the sum of squared deviations from it
  for (int m = 0; m < a.M; ++m) {
    double v = 0.0;
    if (active) {
      const double d = mc_payoff(s_opt[m][0], s_opt[m][1], s_kb[m][0], s_kb[m][1], ps, avg) - s_mean[m];
      v = d * d;
    }
    const double w = warp_sum(v);
    if (lane == 0) s_red[warp][m] = w;
  }
  __syncthreads();
  if (tid < a.M) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < kMcWarps; ++w) t += s_red[w][tid];
    const long long o = (set * a.chunks + cl) * a.M + tid;
    DHJ_CHECK(o >= 0 && o < (long long)a.sets * a.chunks * a.M, kChkOutputIndex);
    a.partial[o] = make_double2(s_mean[tid], t);
  }
}

struct McFinalArgs {
  const double2* partial;          // k_mc_paths' output of the same launch
  double* acc;                     // [sets][M][3]: (n, mean, M2) carried between the launches of a split set
  double* price;                   // [sets][M]
  double* stderr_;                 // [sets][M]
  long long n_paths, chunk0, chunks;
  int sets, M;
  int first, last;                 // the launch holds the set's first / last chunk
  double disc;                     // e^{-rT}
};

__global__ void __launch_bounds__(128) k_mc_finalize(McFinalArgs a) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)a.sets * a.M) return;
  const long long set = i / a.M, m = i - set * a.M;
  const double2* part = a.partial + set * a.chunks * a.M + m;
  double n, mean, M2;
  long long k = 0;
  if (a.first) {
    const double2 p = part[0];
    n = (double)chunk_paths(a.n_paths, a.chunk0); mean = p.x; M2 = p.y;
    k = 1;
  } else {
    n = a.acc[3 * i]; mean = a.acc[3 * i + 1]; M2 = a.acc[3 * i + 2];
  }
  for (; k < a.chunks; ++k) {
    const double2 p = part[k * a.M];
    const double nb = (double)chunk_paths(a.n_paths, a.chunk0 + k);
    const double nn = n + nb;
    const double f = fm::div(nb, nn);        // inline: the IEEE division's slow-path call serialised the loop
    const double d = p.x - mean;
    mean = mean + d * f;
    M2 = M2 + p.y + (d * d) * (n * f);
    n = nn;
  }
  if (a.last) {
    DHJ_CHECK(i >= 0 && i < (long long)a.sets * a.M, kChkOutputIndex);
    a.price[i] = a.disc * mean;
    a.stderr_[i] = a.disc * sqrt(M2 / (n - 1.0) / n);
  } else {
    a.acc[3 * i] = n; a.acc[3 * i + 1] = mean; a.acc[3 * i + 2] = M2;
  }
}

#endif  // __CUDACC__

}  // namespace mc
}  // namespace dhj
