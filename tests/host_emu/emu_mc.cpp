// TEST-ONLY host emulation of the Monte Carlo path scheme (option-pricing-ffn-lbfgs_b200/csrc/dhj_mc.cuh): the same
// DHJ_HD stream, step and payoff functions, compiled by g++ with FMA contraction off.  Built on the fly by
// tests/test_mc_cpu.py; nothing in the product loads it.
#include <stdint.h>

#include "dhj_mc.cuh"

using namespace dhj;
using namespace dhj::mc;

extern "C" {

void emu_mc_words(uint64_t seed, int64_t n, const uint64_t* path, const uint32_t* ctr, uint64_t* w0, uint64_t* w1) {
  for (int64_t i = 0; i < n; ++i) mc_words(seed, path[i], ctr[i], w0 + i, w1 + i);
}

void emu_box_muller(int64_t n, const uint64_t* w0, const uint64_t* w1, double* z0, double* z1) {
  for (int64_t i = 0; i < n; ++i) box_muller(w0[i], w1[i], z0 + i, z1 + i);
}

void emu_poisson_inverse(int64_t n, const double* U, double lam_dt, int32_t* out) {
  const double p0 = fm::exp_(-lam_dt);
  for (int64_t i = 0; i < n; ++i) out[i] = poisson_inverse(U[i], p0, lam_dt);
}

// path statistics of paths[n] for one parameter set: out[n][4] = (S_T, sum, max, min)
void emu_mc_paths(const double* params, double S0, double r, double q, double T, int32_t n_steps, int32_t n_obs,
                  uint64_t seed, int64_t n, const uint64_t* path, double* out) {
  const McSet s = make_mc_set(params, r, q, T / (double)n_steps);
  for (int64_t i = 0; i < n; ++i) {
    const PathStats ps = mc_path(s, S0, seed, path[i], n_steps, n_obs);
    out[4 * i] = ps.ST; out[4 * i + 1] = ps.sum; out[4 * i + 2] = ps.mx; out[4 * i + 3] = ps.mn;
  }
}

// payoffs of one option on path statistics stats[n][4]
void emu_mc_payoff(int64_t n, const double* stats, int32_t n_obs, int32_t kind, int32_t call, double K, double B,
                   double* out) {
  for (int64_t i = 0; i < n; ++i) {
    const PathStats ps{stats[4 * i], stats[4 * i + 1], stats[4 * i + 2], stats[4 * i + 3]};
    out[i] = mc_payoff(kind, call, K, B, ps, ps.sum / (double)n_obs);
  }
}
}

