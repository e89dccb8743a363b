/* dhj.h — C ABI of libdhj.so: B200 (sm_100a) COS pricing of the Double-Heston + Merton-jump model.
 *
 * This is the drop-in boundary for the ONE hot path this repository accelerates.  The reference
 * (zenthepen/Option-Pricing-FFN-LBFGS, mounted at /root/reference while building) is pure Python and
 * has no FFI of its own; its boundary is the Python API of three modules.  Each entry point below
 * names the reference interface it replaces (file:line under /root/reference); INTEGRATION.md shows
 * the ctypes binding a maintainer of the reference would add.
 *
 * Conventions
 *   - plain C, no C++/torch types; every array is C-contiguous float64 (or int32 where said), owned by
 *     the caller and only read/written during the call; the library owns its device scratch, pinned
 *     staging buffers and streams;
 *   - the 13 model parameters are always in calibrator order (src/calibration/lbfgs_calibrator.py:53-57):
 *       v01, kappa1, theta1, sigma1, rho1, v02, kappa2, theta2, sigma2, rho2, lambda_j, mu_j, sigma_j
 *   - every function returns 0 on success or a negative DHJ_ERR_* code and never throws; the text of the
 *     last error is available from dhj_last_error();
 *   - a context is bound to one CUDA device; calls on one context must be serialised by the caller
 *     (the reference is single-threaded: SURVEY §8b);
 *   - there is no CPU fallback: without a CUDA device dhj_init fails with DHJ_ERR_CUDA.
 *   - `*_dev` entry points take CUDA DEVICE pointers and a cudaStream_t (passed as void*), enqueue the
 *     work and return without synchronising; they exist so that callers that already hold data in HBM
 *     (bench.py's kernel-only arm, a torch pipeline) skip the host copies.
 */
#ifndef DHJ_H_
#define DHJ_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DHJ_ABI_VERSION 1
#define DHJ_N_PARAMS 13

#define DHJ_OK 0
#define DHJ_ERR_ARG (-1)     /* bad argument (null pointer, non-positive size, N < 1 ...) */
#define DHJ_ERR_CUDA (-2)    /* CUDA runtime error, no device, wrong architecture */
#define DHJ_ERR_NOMEM (-3)   /* host or device allocation failed */

#if defined(__GNUC__)
#define DHJ_API __attribute__((visibility("default")))
#else
#define DHJ_API
#endif

typedef struct dhj_ctx dhj_ctx;
typedef struct dhj_market dhj_market;

/* ---- context -------------------------------------------------------------------------------- */
DHJ_API int dhj_abi_version(void);
DHJ_API int dhj_device_count(int* count);
DHJ_API int dhj_init(int device, dhj_ctx** ctx);
DHJ_API int dhj_destroy(dhj_ctx* ctx);
/* text of the last error on `ctx` (or of the last failed dhj_init when ctx is NULL); never NULL */
DHJ_API const char* dhj_last_error(const dhj_ctx* ctx);
/* number of kernels this context has launched since dhj_init (bench.py's gpu_launches) */
DHJ_API int dhj_launch_count(const dhj_ctx* ctx, int64_t* count);

/* ---- pricing -------------------------------------------------------------------------------- */
/* Replaces P x M constructions of DoubleHeston(S0,K,T,r,<13 params>,option_type,q).pricing(N)
 * (src/models/double_heston.py:26-46, 160-192) on an arbitrary option LIST.
 *   params[P][13]; S0: s0_stride==0 -> one spot S0[0] for all sets, ==1 -> S0[P];
 *   strike: strike_stride==0 -> strike[M] shared, ==M -> strike[P][M]; maturity[M];
 *   is_call[M] (1 = call, 0 = put: the reference's first-letter rule double_heston.py:172 is applied
 *   by the Python host); N >= 1 cosine terms; L = truncation multiplier (reference default 10,
 *   double_heston.py:100); out[P][M].  Options are grouped by maturity internally; a strike whose
 *   +-0.1 widening binds (double_heston.py:135-137) gets its own truncation range exactly as in the
 *   reference. */
DHJ_API int dhj_price_list(dhj_ctx* ctx, const double* params, int64_t P, const double* S0, int64_t s0_stride,
                   double r, double q, const double* strike, int64_t strike_stride, const double* maturity,
                   const int32_t* is_call, int32_t M, int32_t N, double L, double* out);

/* Grid fast path, output maturity-major out[P][nT][nK] like the generator's loop
 * (src/data/synthetic_generator.py:123-138).  scale_by_spot != 0 -> K = strikes[j]*S0/100
 * (synthetic_generator.py:125), else K = strikes[j]. */
DHJ_API int dhj_price_grid(dhj_ctx* ctx, const double* params, int64_t P, const double* S0, int64_t s0_stride,
                   double r, double q, const double* strikes, int32_t nK, const double* maturities,
                   int32_t nT, int32_t scale_by_spot, int32_t is_call, int32_t N, double L, double* out);

/* Same, with params / S0 / out already in device memory; strikes and maturities are host arrays
 * (tiny tables).  Asynchronous on `stream` (a cudaStream_t; NULL = CUDA's default stream, which is
 * what `torch.cuda.current_stream().cuda_stream` is unless the caller changed it). */
DHJ_API int dhj_price_grid_dev(dhj_ctx* ctx, const double* d_params, int64_t P, const double* d_S0,
                       int64_t s0_stride, double r, double q, const double* strikes, int32_t nK,
                       const double* maturities, int32_t nT, int32_t scale_by_spot, int32_t is_call,
                       int32_t N, double L, double* d_out, void* stream);

/* ---- calibration loss ----------------------------------------------------------------------- */
/* A market = what DoubleHestonJumpCalibrator.__init__ stores (src/calibration/lbfgs_calibrator.py:47-60):
 * spot, risk-free rate and the option list (strike, maturity, price, type).  `n_markets` markets that
 * share maturities / option types can be held in one object (one per calibration instance when many
 * calibrations are batched): S0[n_markets]; strike[n_markets][M] (strike_stride = M) or strike[M]
 * (strike_stride = 0); maturity[M]; is_call[M]; price[n_markets][M].  N is the COS size used by the
 * loss (the reference always uses 128: lbfgs_calibrator.py:150). */
DHJ_API int dhj_market_create(dhj_ctx* ctx, int32_t n_markets, int32_t M, const double* S0, double r,
                      const double* strike, int64_t strike_stride, const double* maturity,
                      const int32_t* is_call, const double* price, int32_t N, dhj_market** market);
DHJ_API int dhj_market_destroy(dhj_market* market);

/* compute_loss(x) for B unconstrained vectors x[B][13] (lbfgs_calibrator.py:118-177): exp/tanh
 * transform (:62-87), prices of every option, 1e10 if any price is NaN/inf/<=0 (:152-153), else
 * mean(((model-market)/market)^2) + Feller penalty (:111-116, :163-169).  market_index[B] selects
 * the market of each vector (NULL -> market 0).  out_loss[B]. */
DHJ_API int dhj_loss_batch(dhj_ctx* ctx, const dhj_market* market, const double* x, const int32_t* market_index,
                   int64_t B, double* out_loss);

/* One launch for what scipy's L-BFGS-B asks per step with jac=None: f(x) and the 13 forward
 * differences g_i = (f(x + h e_i) - f(x)) / ((x_i + h) - x_i)  (scipy/optimize/_numdiff.py
 * _dense_difference, '2-point', abs_step = h; called from lbfgs_calibrator.py:259-269), for C
 * optimiser states x[C][13] at once.  The 14 variants are built on the device.
 * out_f[C], out_g[C][13]; out_f_all (optional, may be NULL) receives the 14 losses [C][14] in
 * evaluation order (f(x), f(x+h e_0), ...), which the host needs to keep the reference's
 * `best_loss` / `n_calls` bookkeeping (lbfgs_calibrator.py:120, 171-172). */
DHJ_API int dhj_loss_fd(dhj_ctx* ctx, const dhj_market* market, const double* x, const int32_t* market_index,
                int64_t C, double h, double* out_f, double* out_g, double* out_f_all);

/* Model prices of every market option at the transformed x (calibrate()'s re-pricing at the optimum,
 * lbfgs_calibrator.py:274-299).  out_prices[B][M] in the caller's option order. */
DHJ_API int dhj_market_prices(dhj_ctx* ctx, const dhj_market* market, const double* x, const int32_t* market_index,
                      int64_t B, double* out_prices);

/* ---- the remaining public methods of DoubleHeston ------------------------------------------- */
/* characteristic_function(phi, tau) at n real frequencies u[n] (double_heston.py:48-97). */
DHJ_API int dhj_cf(dhj_ctx* ctx, const double* params, double r, double q, double tau, const double* u, int32_t n,
           double* out_re, double* out_im);
/* Same for COMPLEX frequencies u = u_re + i u_im (the reference's method accepts them; the pricing path does not use
 * them): the reference's own operation order in complex arithmetic. */
DHJ_API int dhj_cf_complex(dhj_ctx* ctx, const double* params, double r, double q, double tau, const double* u_re,
                           const double* u_im, int32_t n, double* out_re, double* out_im);
/* truncationRange(L): (a,b) for P sets x M options, out_ab[P][M][2] (double_heston.py:100-139). */
DHJ_API int dhj_truncation_range(dhj_ctx* ctx, const double* params, int64_t P, const double* S0, int64_t s0_stride,
                         double r, const double* strike, const double* maturity, int32_t M, double L,
                         double* out_ab);
/* chi_k(k,c,d,a,b) and psi_k(k,c,d,a,b) for n integers k[n] (double_heston.py:141-158). */
DHJ_API int dhj_chi_psi(dhj_ctx* ctx, const int32_t* k, int32_t n, double c, double d, double a, double b,
                double* out_chi, double* out_psi);

/* ---- batched host optimiser (many simultaneous calibrations) --------------------------------- */
/* Lock-step batch of independent, unconstrained L-BFGS-B instances: the algorithm scipy runs for
 * minimize(method='L-BFGS-B') without bounds (lbfgs_calibrator.py:259-269; m = 10, More'-Thuente line search
 * with at most maxls = 20 trials, stop on max|g| <= pgtol or (f_old - f) <= ftol * max(|f_old|,|f|,1), iteration
 * and evaluation limits), restated so that one `ask` / one GPU launch (dhj_loss_fd) / one `tell` advances
 * every calibration at once.  Host-only code.  status[i]: 0 converged (pgtol), 1 converged (ftol),
 * 2 iteration limit, 3 evaluation limit, 4 abnormal (line search failed).
 * `maxfun` counts (f, g) requests (one dhj_loss_fd row each).  The reference runs scipy with jac=None, where a
 * request costs 14 loss evaluations against scipy's default maxfun = 15000 (lbfgs_calibrator.py:259-269 sets no
 * maxfun): pass 15000 / 14 = 1071 for the reference's limit. */
typedef struct dhj_lbfgs dhj_lbfgs;
DHJ_API int dhj_lbfgs_create(int64_t n_states, int32_t dim, int32_t m, int32_t maxiter, int32_t maxfun, int32_t maxls,
                             double ftol, double pgtol, const double* x0, dhj_lbfgs** out);
DHJ_API int dhj_lbfgs_destroy(dhj_lbfgs* opt);
/* states that wait for an evaluation: idx[n_active] (state numbers) and x[n_active][dim]; n_active = 0: all done */
DHJ_API int dhj_lbfgs_ask(dhj_lbfgs* opt, int64_t* n_active, int64_t* idx, double* x);
/* f[n_active], g[n_active][dim] in the order of the last ask */
DHJ_API int dhj_lbfgs_tell(dhj_lbfgs* opt, int64_t n_active, const double* f, const double* g);
/* any output may be NULL: x[n][dim], f[n], nit[n], nfev[n], status[n] */
DHJ_API int dhj_lbfgs_result(const dhj_lbfgs* opt, double* x, double* f, int32_t* nit, int32_t* nfev, int32_t* status);

/* The whole lock-step loop in one call (what dhj.calibrate_many runs per pipeline): ask -> dhj_loss_fd over every
 * state that waits for an evaluation, state i on market state_market[i] (NULL: market 0) -> tell, until all n_states
 * optimisers of `opt` have stopped.  rounds = launches, state_rounds = sum of evaluated states over the rounds,
 * seconds[3] = host time in ask / in the loss calls (copies + launch + wait) / in tell.  Outputs may be NULL.
 * n_states must equal the optimiser's state count (state_market[n_states]) and its dimension must be 13;
 * otherwise the call fails with DHJ_ERR_ARG before the first ask. */
DHJ_API int dhj_lbfgs_minimize_fd(dhj_lbfgs* opt, dhj_ctx* ctx, const dhj_market* market, const int32_t* state_market,
                                  int64_t n_states, double h, int64_t* rounds, int64_t* state_rounds, double* seconds);

/* ---- analytic parameter gradient ------------------------------------------------------------
 * Derivatives with respect to the 13 model parameters (calibrator order) are exact derivatives of the COS price with
 * the truncation range [a, b] held at its value for the current parameters ("frozen range", the usual convention for
 * COS sensitivities; [a, b] depends on the parameters only through the cumulants, and that dependence is below the
 * rounding noise of a finite difference).  Every other step, including the own range of a strike whose +-0.1
 * widening binds, is as in dhj_price_list.
 *
 * dhj_price_jacobian: dhj_price_list's arguments, out_price[P][M] and out_jac[P][M][13] = d price / d param (host
 * buffers, chunked synchronously through device scratch).
 *
 * dhj_loss_grad: dhj_loss_fd's shapes, out_f[C] = compute_loss(x) and out_g[C][13] = the exact gradient in the
 * unconstrained x (chain rule through the exp / tanh transform: p, 1 - rho^2 or 1 per parameter); out_f has the
 * bits of dhj_loss_batch (same prices, same reduction order).  The Feller
 * penalty contributes 1000 (2 sigma dsigma - 2 theta dkappa - 2 kappa dtheta) per factor whose excess
 * sigma^2 - 2 kappa theta is > 0 and nothing otherwise (0 at the kink).  Where the loss is the 1e10 sentinel
 * (any price NaN, inf or <= 0), g = 0.  Each state's (f, g) is formed by one thread in a fixed order: it does not
 * depend on the other states of the call.
 *
 * dhj_lbfgs_minimize_grad: the dhj_lbfgs_minimize_fd loop with dhj_loss_grad as the evaluator (one loss evaluation
 * per request).  n_states must equal the optimiser's state count (state_market[n_states]). */
DHJ_API int dhj_price_jacobian(dhj_ctx* ctx, const double* params, int64_t P, const double* S0, int64_t s0_stride,
                               double r, double q, const double* strike, int64_t strike_stride, const double* maturity,
                               const int32_t* is_call, int32_t M, int32_t N, double L, double* out_price,
                               double* out_jac);
DHJ_API int dhj_loss_grad(dhj_ctx* ctx, const dhj_market* market, const double* x, const int32_t* market_index,
                          int64_t C, double* out_f, double* out_g);
DHJ_API int dhj_lbfgs_minimize_grad(dhj_lbfgs* opt, dhj_ctx* ctx, const dhj_market* market,
                                    const int32_t* state_market, int64_t n_states, int64_t* rounds,
                                    int64_t* state_rounds, double* seconds);

/* ---- Greeks -----------------------------------------------------------------------------------
 * dhj_price_greeks: dhj_price_list's arguments, out_price[P][M] and out_greeks[P][M][DHJ_N_GREEKS] in the caller's
 * option order, per option in this order:
 *   delta = dV/dS0,  gamma = d2V/dS0^2,  theta = -dV/dT (per year, at fixed spot),  rho = dV/dr,  rho_q = dV/dq.
 * All five are exact derivatives of the COS price with the truncation range [a, b] held at its value for the current
 * inputs (the frozen range of dhj_price_jacobian).  [a, b] is a range of the log-return and does not move with S0, so
 * for a strike whose +-0.1 widening does not bind, delta and gamma are the exact derivatives of the price itself.  A
 * binding strike's own range (log(K/S0) +- 0.1) moves with S0; its frozen-range value is reported.  The discount
 * exp(-rT) does not depend on q and the truncation range ignores q (as the reference's does), so
 * rho_q = -(rho + T V).  NaN wherever the price is NaN.  Host buffers, chunked synchronously through device scratch. */
#define DHJ_N_GREEKS 5
DHJ_API int dhj_price_greeks(dhj_ctx* ctx, const double* params, int64_t P, const double* S0, int64_t s0_stride,
                             double r, double q, const double* strike, int64_t strike_stride, const double* maturity,
                             const int32_t* is_call, int32_t M, int32_t N, double L, double* out_price,
                             double* out_greeks);

/* ---- Implied volatility ------------------------------------------------------------------------
 * Black-Scholes implied volatility of option prices, one thread per option, in the option-list layout of
 * dhj_price_list: price[P][M], S0 with stride 0 or 1, strike[M] (strike_stride 0) or [P][M] (strike_stride M),
 * maturity[M], is_call[M] (nonzero: call), scalar r and q (continuous rates).  sigma solves V = BS(S0, K, T, r, q, sigma)
 * with F = S0 e^{(r-q)T} and discount e^{-rT}.
 * out_status[P][M] (may be NULL):
 *   0 ok (a price exactly at the lower bound gives sigma = 0)
 *   1 price below the no-arbitrage lower bound e^{-rT} max(+-(F - K), 0)             -> NaN
 *   2 price at or above the upper bound S0 e^{-qT} (call) or K e^{-rT} (put)         -> NaN
 *   3 invalid input: V, r or q not finite, or S0, K, T not finite and > 0             -> NaN
 *   4 not converged within 40 solver iterations                                       -> the last iterate
 * Accuracy: with sigma* the exact implied vol of the double V and vega = dV/dsigma,
 *   |sigma - sigma*| <= 64 eps (sigma* + V / vega),  eps = 2^-52,
 * where V / vega is the option's own conditioning (tested for sigma in [0.01, 3], T in [1/365, 10],
 * |ln(F/K)| / (sigma sqrt T) <= 6, calls and puts in and out of the money).
 * dhj_implied_vol: host arrays, synchronous chunks through device scratch. */
DHJ_API int dhj_implied_vol(dhj_ctx* ctx, const double* price, int64_t P, const double* S0, int64_t s0_stride,
                            double r, double q, const double* strike, int64_t strike_stride, const double* maturity,
                            const int32_t* is_call, int32_t M, double* out_vol, int32_t* out_status);
/* DEVICE price / S0 / out / status, HOST tables strike[M], maturity[M], is_call[M]; scale_by_spot != 0 ->
 * K = strike[j]*S0/100 (so a dhj_price_grid_dev or dhj_generate_dev surface, flattened maturity-major to
 * M = nT*nK, is inverted without leaving HBM).  Asynchronous on `stream`. */
DHJ_API int dhj_implied_vol_dev(dhj_ctx* ctx, const double* d_price, int64_t P, const double* d_S0,
                                int64_t s0_stride, double r, double q, const double* strike, int32_t scale_by_spot,
                                const double* maturity, const int32_t* is_call, int32_t M, double* d_out_vol,
                                int32_t* d_out_status, void* stream);
/* Black-Scholes prices of vol[P][M] (vol quotes -> prices for dhj_market_create; the forward map of the above).
 * sigma = 0 gives the discounted intrinsic value; NaN for sigma < 0 or NaN and for invalid inputs. */
DHJ_API int dhj_bs_price(dhj_ctx* ctx, const double* vol, int64_t P, const double* S0, int64_t s0_stride, double r,
                         double q, const double* strike, int64_t strike_stride, const double* maturity,
                         const int32_t* is_call, int32_t M, double* out_price);

/* ---- Implied-volatility calibration objective ---------------------------------------------------
 * dhj_market_set_objective selects what dhj_loss_batch, dhj_loss_fd, dhj_loss_grad, dhj_lbfgs_minimize_fd and
 * dhj_lbfgs_minimize_grad compute on `market`:
 *   DHJ_OBJECTIVE_PRICE (the default): compute_loss, the mean squared relative price error + Feller penalty;
 *   DHJ_OBJECTIVE_IV:  f = (1/M_v) sum_{o valid} (sigma_o(x) - sigma^_o)^2 + Feller penalty, where sigma_o(x) is the
 *                      Black-Scholes implied vol (q = 0, the market's S0, K, T, r) of the model price, sigma^_o that of
 *                      the market price, and M_v the number of valid options of the market.
 * Setting DHJ_OBJECTIVE_IV inverts the stored market prices once on the device (dhj_implied_vol's solver); a quote
 * whose status is not 0 (below the lower bound, at or above the upper bound, invalid, not converged) has no implied
 * vol and is left out of the objective.  out_market_vol[n_markets][M] (sigma^, NaN where left out) and
 * out_status[n_markets][M] may be NULL (both are filled on failure too).  A market with no valid option makes the
 * call fail with DHJ_ERR_ARG; the object's objective and market vols are then left as they were.
 * On the IV objective f = 1e10 and g = 0 when a valid option has a model price NaN, inf or <= 0, a model-price
 * implied-vol status != 0 or a vega that is not a positive normal number.  dhj_loss_grad's g is exact with the
 * truncation range held fixed: (2/M_v) sum (sigma_o - sigma^_o) (dV_o/dp) / vega_o, chained to x as on the price
 * objective.  f has the same bits on every entry point.
 * dhj_market_implied_vols: model implied vols out_vol[B][M] and their status out_status[B][M] (may be NULL) at the
 * transformed x, every option of the selected market (reporting; any objective). */
#define DHJ_OBJECTIVE_PRICE 0
#define DHJ_OBJECTIVE_IV 1
DHJ_API int dhj_market_set_objective(dhj_ctx* ctx, dhj_market* market, int32_t objective, double* out_market_vol,
                                     int32_t* out_status);
DHJ_API int dhj_market_implied_vols(dhj_ctx* ctx, const dhj_market* market, const double* x,
                                    const int32_t* market_index, int64_t B, double* out_vol, int32_t* out_status);

/* Threads used by the library's host-side parallel loops (optimiser states in ask / tell, staging copies of pageable
 * buffers); 0 = all cores (default).  Several lock-step pipelines on one host divide the cores with this. */
DHJ_API int dhj_set_host_threads(int32_t n);

/* ---- synthetic generator: the host-side draw stream -------------------------------------------
 * Replaces the per-sample Python loop of generate_synthetic_calibrations
 * (/root/reference/src/data/synthetic_generator.py:98-142: 13 np.random.uniform, one np.random.normal(0.0003,
 * 0.01) for the spot return when i > 0, 15 np.random.normal(0, 0.02) of price noise, AR(1) smoothing :105-109,
 * spot walk :112-116) with the same arithmetic on NumPy's legacy MT19937 stream, bit for bit.  Host only, no
 * context.  State in: np.random.get_state() -> (key[624], pos, has_gauss, cached_gaussian); state out: the same
 * four values after the draws, for np.random.set_state().  Outputs: params[n][n_params], spots[n],
 * noise[n][n_noise] (the N(0, noise_sd) factors; market = model + noise * model, :141-142). */
DHJ_API int dhj_generator_draws(const uint32_t* mt_key, int32_t mt_pos, int32_t has_gauss, double cached_gauss,
                                int64_t n, int32_t n_params, const double* lo, const double* hi, double persistence,
                                double spot0, double ret_mean, double ret_sd, double noise_sd, int32_t n_noise,
                                double* params, double* spots, double* noise, uint32_t* out_key, int32_t* out_pos,
                                int32_t* out_has_gauss, double* out_cached_gauss);

/* ---- synthetic dataset sweep on the device (SURVEY "K3", BASELINE config 4) -------------------
 * Per-sample semantics of generate_synthetic_calibrations (/root/reference/src/data/synthetic_generator.py:98-157):
 * 13 uniform parameters in [lo, hi) (:100-102), AR(1) smoothing with `persistence` (:105-109), spot walk
 * spot * (1 + N(ret_mean, ret_sd)) from spot0 (:112-116), the nT x nK grid of calls at K = strikes_rel * spot / 100
 * priced with rate r and COS size N (:123-138), market = model + N(0, noise_sd) * model (:141-142) and
 * loss = mean(((model - market) / market)^2) (:154-157) — for samples [first, first + n) of the COUNTER STREAM
 * `seed`: every draw is a Philox4x32-10 function of (seed, sample index, slot), so any index range can be produced
 * on any GPU in any order and a sharded dataset does not depend on the number of shards.  Samples are grouped in
 * independent paths of `path_len` consecutive indices (index i: path i / path_len, step i % path_len); each path is
 * one history in the reference's sense (step 0: raw parameters and spot0; path_len = 1: i.i.d. samples).  The
 * exact stream definition is in csrc/dhj_generate.cuh and restated in oracle/cos_oracle.py (counter_*).
 * (The reference's own sequential NumPy stream is kept by dhj_generator_draws for seeded drop-in runs.)
 * Outputs, rows relative to `first`: params[n][13], spots[n], model[n][nT*nK] (maturity-major), market[n][nT*nK],
 * loss[n].  nT*nK <= 32.
 *   dhj_generate_dev: DEVICE pointers, asynchronous on `stream`; nothing leaves HBM.  market and loss may both be
 *                     NULL (parameters, spots and model prices only).
 *   dhj_generate:     HOST arrays (pinned or pageable); chunks are generated, priced and copied back double-buffered. */
DHJ_API int dhj_generate_dev(dhj_ctx* ctx, uint64_t seed, int64_t first, int64_t n, int32_t path_len, const double* lo,
                             const double* hi, double persistence, double spot0, double ret_mean, double ret_sd,
                             double noise_sd, const double* strikes_rel, int32_t nK, const double* maturities,
                             int32_t nT, double r, int32_t N, double L, double* d_params, double* d_spots,
                             double* d_model, double* d_market, double* d_loss, void* stream);
DHJ_API int dhj_generate(dhj_ctx* ctx, uint64_t seed, int64_t first, int64_t n, int32_t path_len, const double* lo,
                         const double* hi, double persistence, double spot0, double ret_mean, double ret_sd,
                         double noise_sd, const double* strikes_rel, int32_t nK, const double* maturities, int32_t nT,
                         double r, int32_t N, double L, double* params, double* spots, double* model, double* market,
                         double* loss);

/* ---- Monte Carlo pricing of path-dependent options ---------------------------------------------
 * dhj_mc_price: P parameter sets params[P][13] (calibrator order), one spot S0[0] (s0_stride 0) or S0[P] (1), one
 * maturity T, continuous rates r and q, and M <= DHJ_MC_MAX_OPTIONS options: kind[M] (DHJ_MC_*), is_call[M] (nonzero:
 * call), strike[M] (finite, >= 0) and barrier[M] (finite, > 0 for the barrier kinds; ignored otherwise; the whole
 * array may be NULL when no option has a barrier).  n_paths paths per set; out_price[P][M] = e^{-rT} x the mean payoff,
 * out_stderr[P][M] (may be NULL) = its standard error e^{-rT} sqrt(sample variance / n_paths) (NaN for n_paths = 1).
 *
 * Scheme: n_steps equal steps dt = T / n_steps, full-truncation Euler for the two variances (Lord, Koekkoek, van Dijk
 * 2010) and log-Euler for the spot with Poisson(lambda dt) Merton jumps per step; e^{-(r-q)t} S_t is an exact
 * martingale of the scheme, so the forward is unbiased, but the variance paths are discretised and the price is NOT an
 * unbiased estimate of the continuous-time price: the bias shrinks with dt (measured against the COS price in
 * DESIGN.md §6f) and barriers are monitored at the observation dates only (no continuity correction).  n_obs divides
 * n_steps; the observations are the ends of steps i n_steps / n_obs, i = 1..n_obs (S0 is not one):
 *   DHJ_MC_EUROPEAN  max(+-(S_T - K), 0)               DHJ_MC_ASIAN    max(+-(A - K), 0), A = mean of S at the dates
 *   DHJ_MC_UP_OUT    European payoff if max S < B      DHJ_MC_UP_IN    ... if max S >= B
 *   DHJ_MC_DOWN_OUT  ... if min S > B                  DHJ_MC_DOWN_IN  ... if min S <= B
 * Random numbers: Philox4x32-10 keyed by `seed`, a function of (seed, path, step) only (stream in csrc/dhj_mc.cuh):
 * every parameter set of a call sees the same numbers, and the outputs have the same bits from run to run and do not
 * depend on the other sets or options of the call.  Model parameters are not validated (a NaN gives NaN).
 * DHJ_ERR_ARG: P, M, n_steps, n_obs or n_paths < 1, n_steps > 2^28, n_steps not a multiple of n_obs, T not finite and
 * > 0, M > DHJ_MC_MAX_OPTIONS, an unknown kind, a strike not finite and >= 0, a barrier option without a finite
 * barrier > 0, a null array (other than barrier / out_stderr), s0_stride not 0 or 1.  Host arrays, synchronous. */
#define DHJ_MC_EUROPEAN 0
#define DHJ_MC_ASIAN 1
#define DHJ_MC_UP_OUT 2
#define DHJ_MC_UP_IN 3
#define DHJ_MC_DOWN_OUT 4
#define DHJ_MC_DOWN_IN 5
#define DHJ_MC_MAX_OPTIONS 64
DHJ_API int dhj_mc_price(dhj_ctx* ctx, const double* params, int64_t P, const double* S0, int64_t s0_stride,
                         double r, double q, double T, int32_t n_steps, int32_t n_obs, int32_t M,
                         const int32_t* kind, const int32_t* is_call, const double* strike, const double* barrier,
                         uint64_t seed, int64_t n_paths, double* out_price, double* out_stderr);

/* ---- checked build -----------------------------------------------------------------------------
 * lib/libdhj_checked.so is the same library compiled with -DDHJ_CHECKED: the kernels verify their own shared-memory
 * protocol (a stage of coefficients read before it was written / overwritten before it was consumed, an item record
 * used before it was prepared) and their shared / output indices, and count violations on the device (the substitute
 * for compute-sanitizer, which is closed on the B200 pool).  counts[8]: violations per kind since the library was
 * loaded (order: read-before-write, write-before-consumed, shared index, output index, item not prepared, 3 spare);
 * *enabled = 0 and all zeros in the product build. */
DHJ_API int dhj_debug_checks(dhj_ctx* ctx, int32_t* enabled, uint64_t* counts);

/* ---- measurement ---------------------------------------------------------------------------- */
/* Runs register-resident FP64 FMA-chain kernels on every SM (two operand forms: three vector registers, and one
 * multiplicand from a uniform register) and reports the best sustained DFMA rate (2 flop per FMA) — the
 * denominator of the FP64 roofline (MEASURED_PEAKS.json has no FP64 figure). */
DHJ_API int dhj_fp64_peak(dhj_ctx* ctx, int32_t iters, double* tflops, double* milliseconds);

#ifdef __cplusplus
}
#endif
#endif /* DHJ_H_ */
