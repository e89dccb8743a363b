// dhj_lbfgs.cpp — batched L-BFGS-B driver for UNCONSTRAINED problems (host side, no CUDA).
//
// The reference calibrates with scipy.optimize.minimize(method='L-BFGS-B', jac=None, no bounds)
// (/root/reference/src/calibration/lbfgs_calibrator.py:259-269).  For one calibration the drop-in keeps scipy.
// For thousands of simultaneous calibrations (BASELINE config C5) Python cannot drive 30 000 scipy state
// machines, so this file restates the same algorithm as a lock-step batch: every state is an independent
// L-BFGS-B instance; `ask` returns the points of all states that need an evaluation, the caller evaluates them
// with ONE GPU launch (dhj_loss_fd) and `tell`s f and g back.
//
// Algorithm, for no bounds, as in L-BFGS-B 3.0 (Byrd, Lu, Nocedal, Zhu; Morales, Nocedal) which scipy wraps:
//   * direction: d = -H g, H the limited-memory BFGS inverse (m = 10 pairs, H0 = (s'y / y'y) I); without
//     bounds L-BFGS-B's Cauchy point / subspace minimisation reduce to exactly this Newton-like step; the
//     first direction (and the one after a memory reset) is -g;
//   * line search: More'-Thuente (MINPACK-2 dcsrch/dcstep) with ftol = 1e-3, gtol = 0.9, xtol = 0.1,
//     stpmin = 0, stpmax = 1e10, first trial step 1/||d|| in the very first iteration and 1 afterwards,
//     at most `maxls` (20) backtracks;
//   * a pair (s, y) is stored only if s'y > eps * ||y||... precisely: dr = (gd - gdold) * stp > eps * (-gdold * stp);
//   * a failed line search restores the point, drops the memory and restarts from -g once; a second failure
//     (or a non-descent direction with empty memory) ends the state as ABNORMAL;
//   * stopping: max|g_i| <= pgtol ; (f_old - f) <= ftol * max(|f_old|, |f|, 1) ; iteration / evaluation limits
//     (scipy: factr = ftol / eps, maxfun = 15000).
// Floating-point details (two-loop recursion instead of the compact matrix form) differ from scipy's C code in
// rounding only; tests/test_lbfgs_batch.py compares iteration counts and minimisers on smooth test functions.
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <new>
#include <vector>
#include <omp.h>

#include "dhj.h"

namespace {

constexpr double kEps = 2.220446049250313e-16;
constexpr double kBig = 1e10;

enum Status : int32_t {
  kRunning = -1,
  kConvPgtol = 0,      // CONVERGENCE: NORM OF PROJECTED GRADIENT <= PGTOL
  kConvFtol = 1,       // CONVERGENCE: RELATIVE REDUCTION OF F <= FACTR*EPSMCH
  kMaxIter = 2,        // STOP: TOTAL NO. OF ITERATIONS REACHED LIMIT
  kMaxFun = 3,         // STOP: TOTAL NO. OF F,G EVALUATIONS EXCEEDS LIMIT
  kAbnormal = 4,       // ABNORMAL (line search failed twice / no descent)
};

// ---- More'-Thuente safeguarded step (MINPACK-2 dcstep) ---------------------------------------------------------
void mt_step(double& stx, double& fx, double& dx, double& sty, double& fy, double& dy, double& stp, double fp,
             double dp, bool& brackt, double stpmin, double stpmax) {
  const double sgnd = dp * (dx / std::fabs(dx));
  double stpf;
  if (fp > fx) {                                   // case 1: higher function value: minimum is bracketed
    const double theta = 3.0 * (fx - fp) / (stp - stx) + dx + dp;
    const double s = std::max({std::fabs(theta), std::fabs(dx), std::fabs(dp)});
    double gamma = s * std::sqrt((theta / s) * (theta / s) - (dx / s) * (dp / s));
    if (stp < stx) gamma = -gamma;
    const double p = (gamma - dx) + theta, q = ((gamma - dx) + gamma) + dp, r = p / q;
    const double stpc = stx + r * (stp - stx);
    const double stpq = stx + ((dx / ((fx - fp) / (stp - stx) + dx)) / 2.0) * (stp - stx);
    stpf = (std::fabs(stpc - stx) < std::fabs(stpq - stx)) ? stpc : stpc + (stpq - stpc) / 2.0;
    brackt = true;
  } else if (sgnd < 0.0) {                         // case 2: derivatives of opposite sign: bracketed
    const double theta = 3.0 * (fx - fp) / (stp - stx) + dx + dp;
    const double s = std::max({std::fabs(theta), std::fabs(dx), std::fabs(dp)});
    double gamma = s * std::sqrt((theta / s) * (theta / s) - (dx / s) * (dp / s));
    if (stp > stx) gamma = -gamma;
    const double p = (gamma - dp) + theta, q = ((gamma - dp) + gamma) + dx, r = p / q;
    const double stpc = stp + r * (stx - stp);
    const double stpq = stp + (dp / (dp - dx)) * (stx - stp);
    stpf = (std::fabs(stpc - stp) > std::fabs(stpq - stp)) ? stpc : stpq;
    brackt = true;
  } else if (std::fabs(dp) < std::fabs(dx)) {      // case 3: derivative magnitude decreases
    const double theta = 3.0 * (fx - fp) / (stp - stx) + dx + dp;
    const double s = std::max({std::fabs(theta), std::fabs(dx), std::fabs(dp)});
    double gamma = s * std::sqrt(std::max(0.0, (theta / s) * (theta / s) - (dx / s) * (dp / s)));
    if (stp > stx) gamma = -gamma;
    const double p = (gamma - dp) + theta, q = (gamma + (dx - dp)) + gamma, r = p / q;
    double stpc;
    if (r < 0.0 && gamma != 0.0) stpc = stp + r * (stx - stp);
    else stpc = (stp > stx) ? stpmax : stpmin;
    const double stpq = stp + (dp / (dp - dx)) * (stx - stp);
    if (brackt) {
      stpf = (std::fabs(stpc - stp) < std::fabs(stpq - stp)) ? stpc : stpq;
      if (stp > stx) stpf = std::min(stp + 0.66 * (sty - stp), stpf);
      else stpf = std::max(stp + 0.66 * (sty - stp), stpf);
    } else {
      stpf = (std::fabs(stpc - stp) > std::fabs(stpq - stp)) ? stpc : stpq;
      stpf = std::max(stpmin, std::min(stpmax, stpf));
    }
  } else {                                         // case 4: derivative does not decrease
    if (brackt) {
      const double theta = 3.0 * (fp - fy) / (sty - stp) + dy + dp;
      const double s = std::max({std::fabs(theta), std::fabs(dy), std::fabs(dp)});
      double gamma = s * std::sqrt((theta / s) * (theta / s) - (dy / s) * (dp / s));
      if (stp > sty) gamma = -gamma;
      const double p = (gamma - dp) + theta, q = ((gamma - dp) + gamma) + dy, r = p / q;
      stpf = stp + r * (sty - stp);
    } else {
      stpf = (stp > stx) ? stpmax : stpmin;
    }
  }
  if (fp > fx) { sty = stp; fy = fp; dy = dp; }
  else {
    if (sgnd < 0.0) { sty = stx; fy = fx; dy = dx; }
    stx = stp; fx = fp; dx = dp;
  }
  stp = stpf;
}

// ---- More'-Thuente line search state (MINPACK-2 dcsrch) ---------------------------------------------------------
struct LineSearch {
  bool brackt;
  int stage;
  double ginit, gtest, gx, gy, finit, fx, fy, stx, sty, stmin, stmax, width, width1;
  static constexpr double ftol = 1e-3, gtol = 0.9, xtol = 0.1, stpmin = 0.0, stpmax = kBig;

  void start(double f, double g, double stp) {
    brackt = false; stage = 1;
    finit = f; ginit = g; gtest = ftol * ginit;
    width = stpmax - stpmin; width1 = width / 0.5;
    stx = 0.0; fx = finit; gx = ginit;
    sty = 0.0; fy = finit; gy = ginit;
    stmin = 0.0; stmax = stp + 4.0 * stp;
  }
  // returns true when the search is over (converged or warning); otherwise `stp` holds the next trial step
  bool advance(double f, double g, double& stp) {
    const double ftest = finit + stp * gtest;
    if (stage == 1 && f <= ftest && g >= 0.0) stage = 2;
    bool done = false;
    if (brackt && (stp <= stmin || stp >= stmax)) done = true;            // rounding errors prevent progress
    if (brackt && stmax - stmin <= xtol * stmax) done = true;             // xtol test satisfied
    if (stp == stpmax && f <= ftest && g <= gtest) done = true;
    if (stp == stpmin && (f > ftest || g >= gtest)) done = true;
    if (f <= ftest && std::fabs(g) <= gtol * (-ginit)) done = true;       // strong Wolfe conditions hold
    if (done) return true;
    if (stage == 1 && f <= fx && f > ftest) {
      double fm = f - stp * gtest, fxm = fx - stx * gtest, fym = fy - sty * gtest;
      double gm = g - gtest, gxm = gx - gtest, gym = gy - gtest;
      mt_step(stx, fxm, gxm, sty, fym, gym, stp, fm, gm, brackt, stmin, stmax);
      fx = fxm + stx * gtest; fy = fym + sty * gtest; gx = gxm + gtest; gy = gym + gtest;
    } else {
      mt_step(stx, fx, gx, sty, fy, gy, stp, f, g, brackt, stmin, stmax);
    }
    if (brackt) {
      if (std::fabs(sty - stx) >= 0.66 * width1) stp = stx + 0.5 * (sty - stx);
      width1 = width; width = std::fabs(sty - stx);
    }
    if (brackt) { stmin = std::min(stx, sty); stmax = std::max(stx, sty); }
    else { stmin = stp + 1.1 * (stp - stx); stmax = stp + 4.0 * (stp - stx); }
    stp = std::max(stp, stpmin); stp = std::min(stp, stpmax);
    if ((brackt && (stp <= stmin || stp >= stmax)) || (brackt && stmax - stmin <= xtol * stmax)) stp = stx;
    return false;
  }
};

struct State {
  Status status = kRunning;
  bool need_eval = true;          // waiting for f,g at `xt`
  bool first_eval = true;
  int iter = 0, nfev = 0, col = 0, head = 0, ifun = 0;
  bool restarted = false;
  double f = 0, fold = 0, stp = 0, gd = 0, gdold = 0, dnorm = 0;
  LineSearch ls;
};

}  // namespace

struct dhj_lbfgs {
  int64_t n = 0;
  int dim = 0, m = 10, maxiter = 300, maxfun = 15000, maxls = 20;
  double ftol = 1e-9, pgtol = 1e-6;
  std::vector<State> st;
  std::vector<double> x, g, xold, gold, d, xt;      // [n][dim]
  std::vector<double> S, Y, rho;                    // [n][m][dim], [n][m]
  std::vector<int64_t> asked;                       // indices handed out by the last ask()

  double* row(std::vector<double>& v, int64_t i) { return v.data() + i * dim; }

  void direction(int64_t i) {
    State& s = st[i];
    double* di = row(d, i);
    const double* gi = row(g, i);
    for (int k = 0; k < dim; ++k) di[k] = -gi[k];
    if (s.col == 0) return;
    double alpha[64];
    const double* Si = S.data() + i * (int64_t)m * dim;
    const double* Yi = Y.data() + i * (int64_t)m * dim;
    const double* ri = rho.data() + i * m;
    for (int j = s.col - 1; j >= 0; --j) {                  // newest to oldest
      const int p = (s.head + j) % m;
      double a = 0.0;
      for (int k = 0; k < dim; ++k) a += Si[p * dim + k] * di[k];
      a *= ri[p];
      alpha[j] = a;
      for (int k = 0; k < dim; ++k) di[k] -= a * Yi[p * dim + k];
    }
    const int pl = (s.head + s.col - 1) % m;                // H0 = (s'y / y'y) I of the newest pair
    double yy = 0.0;
    for (int k = 0; k < dim; ++k) yy += Yi[pl * dim + k] * Yi[pl * dim + k];
    const double gamma = 1.0 / (ri[pl] * yy);
    for (int k = 0; k < dim; ++k) di[k] *= gamma;
    for (int j = 0; j < s.col; ++j) {                       // oldest to newest
      const int p = (s.head + j) % m;
      double b = 0.0;
      for (int k = 0; k < dim; ++k) b += Yi[p * dim + k] * di[k];
      b *= ri[p];
      for (int k = 0; k < dim; ++k) di[k] += (alpha[j] - b) * Si[p * dim + k];
    }
  }

  // start a line search from the current (x, f, g); returns false if the state ended instead
  bool begin_line_search(int64_t i) {
    State& s = st[i];
    for (;;) {
      direction(i);
      const double* di = row(d, i);
      const double* gi = row(g, i);
      double dtd = 0.0, gd = 0.0;
      for (int k = 0; k < dim; ++k) { dtd += di[k] * di[k]; gd += gi[k] * di[k]; }
      s.dnorm = std::sqrt(dtd);
      s.gd = gd;
      if (!(gd < 0.0)) {                                     // not a descent direction
        if (s.col == 0) { s.status = kAbnormal; s.need_eval = false; return false; }
        s.col = 0; s.head = 0;                               // drop the memory, restart from -g
        continue;
      }
      break;
    }
    s.stp = (s.iter == 0) ? std::min(1.0 / s.dnorm, kBig) : 1.0;
    memcpy(row(xold, i), row(x, i), dim * sizeof(double));
    memcpy(row(gold, i), row(g, i), dim * sizeof(double));
    s.fold = s.f; s.gdold = s.gd; s.ifun = 0;
    s.ls.start(s.f, s.gd, s.stp);
    trial_point(i);
    return true;
  }

  void trial_point(int64_t i) {
    State& s = st[i];
    const double* xo = row(xold, i);
    const double* di = row(d, i);
    double* t = row(xt, i);
    for (int k = 0; k < dim; ++k) t[k] = s.stp * di[k] + xo[k];
    s.need_eval = true;
  }

  void receive(int64_t i, double fv, const double* gv) {
    State& s = st[i];
    s.nfev++;
    if (s.first_eval) {
      s.first_eval = false;
      s.f = fv;
      memcpy(row(x, i), row(xt, i), dim * sizeof(double));
      memcpy(row(g, i), gv, dim * sizeof(double));
      double gn = 0.0;
      for (int k = 0; k < dim; ++k) gn = std::max(gn, std::fabs(gv[k]));
      if (gn <= pgtol) { s.status = kConvPgtol; s.need_eval = false; return; }
      begin_line_search(i);
      return;
    }
    // inside a line search: f, g at xold + stp d
    const double* di = row(d, i);
    double gd = 0.0;
    for (int k = 0; k < dim; ++k) gd += gv[k] * di[k];
    s.ifun++;
    double stp = s.stp;
    const bool done = s.ls.advance(fv, gd, stp);
    if (!done) {
      if (s.ifun >= maxls) {                                   // iback = ifun - 1 >= maxls before the next trial
        line_search_failed(i);
        return;
      }
      s.stp = stp;
      trial_point(i);
      return;
    }
    // accept the step
    s.f = fv; s.gd = gd;
    memcpy(row(x, i), row(xt, i), dim * sizeof(double));
    memcpy(row(g, i), gv, dim * sizeof(double));
    s.iter++;
    s.restarted = false;
    // scipy's wrapper looks at the limits when L-BFGS-B reports NEW_X, i.e. before the convergence tests
    if (s.iter >= maxiter) { s.status = kMaxIter; s.need_eval = false; return; }
    if (s.nfev > maxfun) { s.status = kMaxFun; s.need_eval = false; return; }
    double gn = 0.0;
    for (int k = 0; k < dim; ++k) gn = std::max(gn, std::fabs(gv[k]));
    if (gn <= pgtol) { s.status = kConvPgtol; s.need_eval = false; return; }
    const double ddum = std::max({std::fabs(s.fold), std::fabs(s.f), 1.0});
    if (s.fold - s.f <= ftol * ddum) { s.status = kConvFtol; s.need_eval = false; return; }
    // curvature pair: s = stp d, y = g - gold
    const double dr = (s.gd - s.gdold) * s.stp, dd = -s.gdold * s.stp;
    if (dr > kEps * dd) {
      int slot;
      if (s.col < m) { slot = (s.head + s.col) % m; s.col++; }
      else { slot = s.head; s.head = (s.head + 1) % m; }
      double* Si = S.data() + (i * (int64_t)m + slot) * dim;
      double* Yi = Y.data() + (i * (int64_t)m + slot) * dim;
      const double* go = row(gold, i);
      double sy = 0.0;
      for (int k = 0; k < dim; ++k) {
        Si[k] = s.stp * di[k];
        Yi[k] = gv[k] - go[k];
        sy += Si[k] * Yi[k];
      }
      rho[i * m + slot] = 1.0 / sy;
    }
    begin_line_search(i);
  }

  void line_search_failed(int64_t i) {
    State& s = st[i];
    memcpy(row(x, i), row(xold, i), dim * sizeof(double));
    memcpy(row(g, i), row(gold, i), dim * sizeof(double));
    s.f = s.fold;
    if (s.col == 0) {                                        // already steepest descent: give up (nit unchanged,
      s.status = kAbnormal;                                  // scipy counts iterations on NEW_X only)
      s.need_eval = false;
      return;
    }
    s.col = 0; s.head = 0;                                   // refresh the memory and restart from -g
    begin_line_search(i);
  }
};

extern "C" {

int dhj_lbfgs_create(int64_t n_states, int32_t dim, int32_t m, int32_t maxiter, int32_t maxfun, int32_t maxls,
                     double ftol, double pgtol, const double* x0, dhj_lbfgs** out) {
  if (!out) return DHJ_ERR_ARG;
  *out = nullptr;
  if (n_states < 0 || dim < 1 || m < 1 || m > 64 || maxiter < 0 || maxfun < 1 || maxls < 1 || !x0) return DHJ_ERR_ARG;
  dhj_lbfgs* o = new (std::nothrow) dhj_lbfgs();
  if (!o) return DHJ_ERR_NOMEM;
  try {
    o->n = n_states; o->dim = dim; o->m = m; o->maxiter = maxiter; o->maxfun = maxfun; o->maxls = maxls;
    o->ftol = ftol; o->pgtol = pgtol;
    const size_t nd = (size_t)n_states * dim;
    o->st.resize(n_states);
    o->x.assign(nd, 0.0); o->g.assign(nd, 0.0); o->xold.assign(nd, 0.0); o->gold.assign(nd, 0.0);
    o->d.assign(nd, 0.0); o->xt.assign(x0, x0 + nd);
    o->S.assign(nd * m, 0.0); o->Y.assign(nd * m, 0.0); o->rho.assign((size_t)n_states * m, 0.0);
    if (maxiter == 0)
      for (auto& s : o->st) s.need_eval = true;              // scipy still evaluates f, g at x0
  } catch (const std::bad_alloc&) {
    delete o;
    return DHJ_ERR_NOMEM;
  }
  *out = o;
  return DHJ_OK;
}

int dhj_lbfgs_destroy(dhj_lbfgs* o) {
  delete o;
  return DHJ_OK;
}

// threads of the library's host-side parallel loops (optimiser states, staging copies); 0 = all cores.  Several
// lock-step pipelines on one host (dhj.calibrate_many) divide the cores among themselves with this.
static int g_host_threads = 0;
int dhj_host_threads() { return g_host_threads > 0 ? g_host_threads : omp_get_num_procs(); }
int dhj_set_host_threads(int32_t n) {
  if (n < 0) return DHJ_ERR_ARG;
  g_host_threads = n;
  return DHJ_OK;
}

int dhj_lbfgs_ask(dhj_lbfgs* o, int64_t* n_active, int64_t* idx, double* x) {
  if (!o || !n_active || !idx || !x) return DHJ_ERR_ARG;
  o->asked.clear();
  for (int64_t i = 0; i < o->n; ++i)
    if (o->st[i].status == kRunning && o->st[i].need_eval) o->asked.push_back(i);
  *n_active = (int64_t)o->asked.size();
  const int64_t na = (int64_t)o->asked.size();
#pragma omp parallel for schedule(static) num_threads(dhj_host_threads()) if (na > 4096)
  for (int64_t a = 0; a < na; ++a) {
    idx[a] = o->asked[a];
    memcpy(x + a * o->dim, o->row(o->xt, o->asked[a]), o->dim * sizeof(double));
  }
  return DHJ_OK;
}

int dhj_lbfgs_tell(dhj_lbfgs* o, int64_t n_active, const double* f, const double* g) {
  if (!o || !f || !g || n_active != (int64_t)o->asked.size()) return DHJ_ERR_ARG;
  // states are independent: advance them on all host cores (30 000 states per round in config C5)
#pragma omp parallel for schedule(static) num_threads(dhj_host_threads()) if (n_active > 256)
  for (int64_t a = 0; a < n_active; ++a) {
    const int64_t i = o->asked[a];
    o->st[i].need_eval = false;
    o->receive(i, f[a], g + a * o->dim);
    // maxiter = 0: one evaluation, then stop like scipy does
    if (o->maxiter == 0 && o->st[i].status == kRunning) { o->st[i].status = kMaxIter; o->st[i].need_eval = false; }
  }
  o->asked.clear();
  return DHJ_OK;
}

// library-internal (not in dhj.h): state count and dimension, for callers that size buffers per ask
int dhj_lbfgs_shape(const dhj_lbfgs* o, int64_t* n, int32_t* dim) {
  if (!o || !n || !dim) return DHJ_ERR_ARG;
  *n = o->n; *dim = o->dim;
  return DHJ_OK;
}

int dhj_lbfgs_result(const dhj_lbfgs* o, double* x, double* f, int32_t* nit, int32_t* nfev, int32_t* status) {
  if (!o) return DHJ_ERR_ARG;
  for (int64_t i = 0; i < o->n; ++i) {
    const State& s = o->st[i];
    if (x) memcpy(x + i * o->dim, o->x.data() + i * o->dim, o->dim * sizeof(double));
    if (f) f[i] = s.f;
    if (nit) nit[i] = s.iter;
    if (nfev) nfev[i] = s.nfev;
    if (status) status[i] = (int32_t)s.status;
  }
  return DHJ_OK;
}

}  // extern "C"
