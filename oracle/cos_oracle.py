"""CPU oracle for the COS pricing / calibration-loss hot path.  TEST INFRASTRUCTURE ONLY.

This module restates, in NumPy float64/complex128, the algorithm of the reference
(zenthepen/Option-Pricing-FFN-LBFGS) for the one path this repository accelerates.  It exists to
CHECK the CUDA path; it is never the thing shipped or measured.  Only `tests/`,
`__graft_entry__.smoke()` and the CPU-baseline / `--impl reference` legs of `bench.py` may import it.
The product package (`option-pricing-ffn-lbfgs_b200/`) must not, and does not.

Parity status: PINNED.  `tests/test_oracle_golden.py` checks every function here against fixtures
under `tests/golden/` that were produced by importing the unmodified reference in the build
container (`tests/golden/make_golden.py`); the literals of SURVEY.md §8c are checked as tripwires.

Two restatements are provided:

* `*_scalar`   one option at a time with NumPy scalars, operation for operation in the order the
               reference evaluates them (this is also what `bench.py --impl reference` times,
               because it reproduces the reference's execution model: Python loops over k);
* `price_batch` the same arithmetic vectorised over (parameter set, option, k) so that 1e5-price
               parity samples finish in seconds.

Reference citations are `/root/reference/<file>:<line>`.
Parameter vector order everywhere: (v01, kappa1, theta1, sigma1, rho1, v02, kappa2, theta2, sigma2,
rho2, lambda_j, mu_j, sigma_j) = src/calibration/lbfgs_calibrator.py:53-57.
"""
from __future__ import annotations

import numpy as np

N_PARAMS = 13
SENTINEL = 1e10           # src/calibration/lbfgs_calibrator.py:152-153
FD_STEP = 1e-8            # scipy L-BFGS-B default eps (scipy/optimize/_lbfgsb_py.py)

PARAM_NAMES = ("v1_0", "kappa1", "theta1", "sigma1", "rho1", "v2_0", "kappa2", "theta2", "sigma2",
               "rho2", "lambda_j", "mu_j", "sigma_j")           # lbfgs_calibrator.py:53-57

# src/data/synthetic_generator.py:75-89 (dict order = RNG draw order)
GENERATOR_RANGES = np.array([
    (0.025, 0.080), (1.5, 4.5), (0.025, 0.065), (0.20, 0.50), (-0.85, -0.40),
    (0.020, 0.070), (0.30, 1.20), (0.025, 0.070), (0.10, 0.35), (-0.70, -0.20),
    (0.05, 0.25), (-0.08, -0.01), (0.03, 0.12)])
GENERATOR_STRIKES_REL = np.array([90.0, 95.0, 100.0, 105.0, 110.0])   # synthetic_generator.py:91
GENERATOR_MATURITIES = np.array([0.25, 0.5, 1.0])                     # synthetic_generator.py:92
GENERATOR_RATE = 0.03                                                 # synthetic_generator.py:94


def is_call_flag(option_type) -> bool:
    """First letter, upper-cased, equal to 'C' (src/models/double_heston.py:172)."""
    return str(option_type).upper()[0] == "C"


# ----------------------------------------------------------------------------------------------
# scalar restatement
# ----------------------------------------------------------------------------------------------
def _heston_factor_scalar(u, tau, v0, kappa, theta, sigma, rho):
    """One variance factor of the CF: returns (A_j, B_j).  src/models/double_heston.py:64-71, 85-87."""
    i = 1j
    beta = kappa - rho * sigma * i * u
    d = np.sqrt(beta ** 2 + sigma ** 2 * u * (u + i))
    g = (beta - d) / (beta + d)
    B = ((beta - d) / sigma ** 2) * ((1 - np.exp(-d * tau)) / (1 - g * np.exp(-d * tau)))
    A = (kappa * theta / sigma ** 2) * ((beta - d) * tau - 2 * np.log((1 - g * np.exp(-d * tau)) / (1 - g)))
    return A, B


def cf_scalar(u, tau, p, r, q=0.0):
    """phi(u; tau) of the log-return.  src/models/double_heston.py:48-97."""
    v01, k1, t1, s1, rho1, v02, k2, t2, s2, rho2, lam, mu, sj = [np.float64(v) for v in p]
    i = 1j
    u = np.float64(u)
    with np.errstate(all="ignore"):
        A1, B1 = _heston_factor_scalar(u, tau, v01, k1, t1, s1, rho1)
        A2, B2 = _heston_factor_scalar(u, tau, v02, k2, t2, s2, rho2)
        compensator = np.exp(mu + 0.5 * sj ** 2) - 1                     # :82
        A = (r - q - lam * compensator) * i * u * tau                    # :83
        A += A1                                                          # :85-87
        A += A2                                                          # :89-91
        cf_jump = np.exp(lam * tau * (np.exp(i * u * mu - 0.5 * sj ** 2 * u ** 2) - 1))   # :93
        cf_heston = np.exp(A + B1 * v01 + B2 * v02)                      # :94
        return cf_heston * cf_jump                                       # :96


def _factor_cumulants(tau, r, v0, kappa, theta, sigma, rho):
    """c1, c2 of one factor.  src/models/double_heston.py:101-119 (r*tau enters once per factor)."""
    e = np.exp(-kappa * tau)
    c1 = r * tau + (1 - e) * (theta - v0) / (2 * kappa) - theta * tau / 2
    c2 = 1 / (8 * np.power(kappa, 3)) * (
        sigma * tau * kappa * e * (v0 - theta) * (8 * kappa * rho - 4 * sigma)
        + kappa * rho * sigma * (1 - e) * (16 * theta - 8 * v0)
        + 2 * theta * kappa * tau * (-4 * kappa * rho * sigma + np.power(sigma, 2) + 4 * np.power(kappa, 2))
        + np.power(sigma, 2) * ((theta - 2 * v0) * np.exp(-2 * kappa * tau) + theta * (6 * e - 7) + 2 * v0)
        + 8 * np.power(kappa, 2) * (v0 - theta) * (1 - e))
    return c1, c2


def truncation_range_scalar(p, S0, K, T, r, L=10):
    """(a, b).  src/models/double_heston.py:100-139.  Python min/max keep a NaN first argument."""
    v01, k1, t1, s1, rho1, v02, k2, t2, s2, rho2, lam, mu, sj = [np.float64(v) for v in p]
    with np.errstate(all="ignore"):
        c1a, c2a = _factor_cumulants(T, r, v01, k1, t1, s1, rho1)
        c1b, c2b = _factor_cumulants(T, r, v02, k2, t2, s2, rho2)
        c1 = c1a + c1b + lam * T * mu                                     # :123,127
        c2 = c2a + c2b + lam * T * (sj ** 2 + mu ** 2)                    # :124,128
        a = c1 - L * np.sqrt(np.abs(c2))
        b = c1 + L * np.sqrt(np.abs(c2))
        x = np.log(K / S0)
    a = min(a, x - 0.1)                                                   # :136
    b = max(b, x + 0.1)                                                   # :137
    return a, b


def _chi_psi_scalar(k, c, d, a, b):
    """(chi_k, psi_k).  src/models/double_heston.py:141-158."""
    if k == 0:
        return np.exp(d) - np.exp(c), d - c
    u = k * np.pi / (b - a)
    chi = (1.0 / (1 + u ** 2)) * (np.cos(u * (d - a)) * np.exp(d) - np.cos(u * (c - a)) * np.exp(c)
                                  + u * np.sin(u * (d - a)) * np.exp(d) - u * np.sin(u * (c - a)) * np.exp(c))
    psi = (1.0 / u) * (np.sin(u * (d - a)) - np.sin(u * (c - a)))
    return chi, psi


def price_scalar(p, S0, K, T, r, is_call=True, q=0.0, N=128, L=10):
    """One European option by the COS method.  src/models/double_heston.py:160-192."""
    with np.errstate(all="ignore"):
        x = np.log(K / S0)
        a, b = truncation_range_scalar(p, S0, K, T, r, L)
        u = np.arange(N) * np.pi / (b - a)                                # :165-166
        phi = np.array([cf_scalar(uk, T, p, r, q) for uk in u])           # :168
        V = np.zeros(N)
        for k in range(N):
            if is_call:
                chi, psi = _chi_psi_scalar(k, x, b, a, b)                 # :177-178
                V[k] = (2.0 / (b - a)) * (S0 * chi - K * psi)             # :179
            else:
                chi, psi = _chi_psi_scalar(k, a, x, a, b)                 # :183-184
                V[k] = (2.0 / (b - a)) * (K * psi - S0 * chi)             # :185
        terms = np.real(phi * np.exp(-1j * u * a)) * V                    # :187
        terms[0] *= 0.5                                                   # :188
        return float(np.exp(-r * T) * np.sum(terms))                      # :190


# ----------------------------------------------------------------------------------------------
# vectorised restatement (same arithmetic, arrays over (set, option, k))
# ----------------------------------------------------------------------------------------------
def _heston_factor_vec(u, tau, v0, kappa, theta, sigma, rho):
    i = 1j
    beta = kappa - rho * sigma * i * u
    d = np.sqrt(beta ** 2 + sigma ** 2 * u * (u + i))
    g = (beta - d) / (beta + d)
    E = np.exp(-d * tau)
    B = ((beta - d) / sigma ** 2) * ((1 - E) / (1 - g * E))
    A = (kappa * theta / sigma ** 2) * ((beta - d) * tau - 2 * np.log((1 - g * E) / (1 - g)))
    return A, B


def cf_vec(u, tau, params, r, q=0.0):
    """CF for broadcastable arrays: u[..., N], tau[..., 1], params[..., 13] (leading dims broadcast)."""
    P = [np.asarray(params)[..., j, None] for j in range(N_PARAMS)]
    v01, k1, t1, s1, rho1, v02, k2, t2, s2, rho2, lam, mu, sj = P
    i = 1j
    with np.errstate(all="ignore"):
        A1, B1 = _heston_factor_vec(u, tau, v01, k1, t1, s1, rho1)
        A2, B2 = _heston_factor_vec(u, tau, v02, k2, t2, s2, rho2)
        compensator = np.exp(mu + 0.5 * sj ** 2) - 1
        A = (r - q - lam * compensator) * i * u * tau
        A = A + A1
        A = A + A2
        cf_jump = np.exp(lam * tau * (np.exp(i * u * mu - 0.5 * sj ** 2 * u ** 2) - 1))
        return np.exp(A + B1 * v01 + B2 * v02) * cf_jump


def truncation_range_vec(params, S0, K, T, r, L=10):
    """(a, b) arrays, broadcasting params[..., 13] against S0, K, T."""
    P = [np.asarray(params)[..., j] for j in range(N_PARAMS)]
    v01, k1, t1, s1, rho1, v02, k2, t2, s2, rho2, lam, mu, sj = P
    with np.errstate(all="ignore"):
        c1a, c2a = _factor_cumulants(T, r, v01, k1, t1, s1, rho1)
        c1b, c2b = _factor_cumulants(T, r, v02, k2, t2, s2, rho2)
        c1 = c1a + c1b + lam * T * mu
        c2 = c2a + c2b + lam * T * (sj ** 2 + mu ** 2)
        a = c1 - L * np.sqrt(np.abs(c2))
        b = c1 + L * np.sqrt(np.abs(c2))
        x = np.log(K / S0)
        # Python min(a, y): y if y < a else a  -> a NaN `a` survives, a NaN `y` is dropped
        a = np.where((x - 0.1) < a, x - 0.1, a)
        b = np.where((x + 0.1) > b, x + 0.1, b)
    return a, b


def price_batch(params, S0, strike, maturity, is_call, r, q=0.0, N=128, L=10, chunk=2048,
                return_ab=False):
    """Prices for P parameter sets x M options -> float64[P, M].

    params[P,13]; S0 scalar or [P]; strike [M] or [P,M]; maturity [M]; is_call [M] (truthy = call).
    Like the reference, the CF is evaluated per option (no sharing across strikes), so the
    K-dependent widening of (a,b) (double_heston.py:135-137) is reproduced exactly.
    """
    params = np.asarray(params, dtype=np.float64).reshape(-1, N_PARAMS)
    P = params.shape[0]
    maturity = np.asarray(maturity, dtype=np.float64).reshape(-1)
    M = maturity.shape[0]
    S0 = np.broadcast_to(np.asarray(S0, dtype=np.float64), (P,))
    strike = np.broadcast_to(np.asarray(strike, dtype=np.float64), (P, M))
    call = np.broadcast_to(np.asarray(is_call).astype(bool), (M,))
    out = np.empty((P, M))
    ab = np.empty((P, M, 2))
    kk = np.arange(N)
    for lo in range(0, P, chunk):
        hi = min(P, lo + chunk)
        pr = params[lo:hi, None, :]                       # [p,1,13]
        s0 = S0[lo:hi, None]                              # [p,1]
        K = strike[lo:hi]                                 # [p,M]
        T = maturity[None, :]                             # [1,M]
        with np.errstate(all="ignore"):
            a, b = truncation_range_vec(pr, s0, K, T, r, L)                 # [p,M]
            x = np.log(K / s0)
            u = kk[None, None, :] * np.pi / (b - a)[..., None]              # [p,M,N]  (k*pi)/(b-a)
            phi = cf_vec(u, T[..., None], pr, r, q)                         # [p,M,N]
            c = np.where(call[None, :], x, a)[..., None]
            d = np.where(call[None, :], b, x)[..., None]
            a3 = a[..., None]
            ed, ec = np.exp(d), np.exp(c)
            chi = (1.0 / (1 + u ** 2)) * (np.cos(u * (d - a3)) * ed - np.cos(u * (c - a3)) * ec
                                          + u * np.sin(u * (d - a3)) * ed - u * np.sin(u * (c - a3)) * ec)
            psi = (1.0 / u) * (np.sin(u * (d - a3)) - np.sin(u * (c - a3)))
            chi[..., 0] = (ed - ec)[..., 0]
            psi[..., 0] = (d - c)[..., 0]
            sgn = np.where(call, 1.0, -1.0)[None, :, None]
            V = (2.0 / (b - a))[..., None] * (sgn * (s0[..., None] * chi - K[..., None] * psi))
            terms = np.real(phi * np.exp(-1j * u * a3)) * V
            terms[..., 0] *= 0.5
            out[lo:hi] = np.exp(-r * T) * np.sum(terms, axis=-1)
            ab[lo:hi, :, 0] = a
            ab[lo:hi, :, 1] = b
    return (out, ab) if return_ab else out


# ----------------------------------------------------------------------------------------------
# calibrator loss (src/calibration/lbfgs_calibrator.py)
# ----------------------------------------------------------------------------------------------
def transform_params(x):
    """Unconstrained x[...,13] -> model parameters.  lbfgs_calibrator.py:62-87."""
    x = np.asarray(x, dtype=np.float64)
    with np.errstate(all="ignore"):
        p = np.exp(x)
        p[..., 4] = np.tanh(x[..., 4])
        p[..., 9] = np.tanh(x[..., 9])
        p[..., 11] = x[..., 11]
    return p


def inverse_transform_params(p):
    """lbfgs_calibrator.py:89-109 (rho clipped to +-0.999 before arctanh)."""
    p = np.asarray(p, dtype=np.float64)
    with np.errstate(all="ignore"):
        x = np.log(p)
    x[..., 4] = np.arctanh(np.clip(p[..., 4], -0.999, 0.999))
    x[..., 9] = np.arctanh(np.clip(p[..., 9], -0.999, 0.999))
    x[..., 11] = p[..., 11]
    return x


def feller_penalty(p):
    """1000*(max(0,s1^2-2k1t1)+max(0,s2^2-2k2t2)).  lbfgs_calibrator.py:111-116."""
    p = np.asarray(p, dtype=np.float64)
    with np.errstate(all="ignore"):
        e1 = p[..., 3] ** 2 - 2 * p[..., 1] * p[..., 2]
        e2 = p[..., 8] ** 2 - 2 * p[..., 6] * p[..., 7]
    # Python max(0, e): e if e > 0 else 0  (a NaN e gives 0)
    pen1 = np.where(e1 > 0, e1, 0.0)
    pen2 = np.where(e2 > 0, e2, 0.0)
    return 1000.0 * (pen1 + pen2)


def loss_batch(x, spot, r, strike, maturity, is_call, market, N=128):
    """compute_loss for B unconstrained vectors x[B,13] -> float64[B].  lbfgs_calibrator.py:118-177."""
    x = np.asarray(x, dtype=np.float64).reshape(-1, N_PARAMS)
    p = transform_params(x)
    prices = price_batch(p, spot, strike, maturity, is_call, r, 0.0, N)      # q defaults to 0 (:131-149)
    market = np.asarray(market, dtype=np.float64)
    with np.errstate(all="ignore"):
        bad = np.any(~np.isfinite(prices) | (prices <= 0), axis=1)            # :152-153
        rel = (prices - market) / market                                      # :163
        mse = np.mean(rel ** 2, axis=1)                                       # :164
        total = mse + feller_penalty(p)                                       # :167-169
    return np.where(bad, SENTINEL, total)


def loss_scalar(x, spot, r, strike, maturity, is_call, market, N=128):
    """Scalar-path compute_loss (one option at a time, early exit on a bad price)."""
    p = transform_params(np.asarray(x, dtype=np.float64))
    prices = []
    for K, T, c in zip(strike, maturity, is_call):
        price = price_scalar(p, spot, K, T, r, bool(c), 0.0, N)
        if np.isnan(price) or np.isinf(price) or price <= 0:
            return SENTINEL
        prices.append(price)
    rel = (np.array(prices) - np.asarray(market)) / np.asarray(market)
    return float(np.mean(rel ** 2) + feller_penalty(p))


def fd_stencil(x, h=FD_STEP):
    """The 14 points scipy evaluates for one f,g request: x and x+h*e_i.  Returns (pts[14,13], dx[13]).

    scipy/optimize/_numdiff.py `_dense_difference`, method '2-point', abs_step=h, no bounds:
    x_i' = x_i + h ; dx_i = x_i' - x_i ; g_i = (f(x') - f(x)) / dx_i.
    """
    x = np.asarray(x, dtype=np.float64)
    pts = np.tile(x, (N_PARAMS + 1, 1))
    idx = np.arange(N_PARAMS)
    pts[1 + idx, idx] = x + h
    dx = pts[1 + idx, idx] - x
    return pts, dx


def loss_fd(x, spot, r, strike, maturity, is_call, market, N=128, h=FD_STEP):
    """(f, g[13]) exactly as scipy's L-BFGS-B obtains them from compute_loss with jac=None."""
    pts, dx = fd_stencil(x, h)
    f = loss_batch(pts, spot, r, strike, maturity, is_call, market, N)
    return float(f[0]), (f[1:] - f[0]) / dx


def initial_guess(kind, spot, strike, maturity, market, rng=np.random):
    """get_initial_guess(kind).  lbfgs_calibrator.py:179-234; kind 1 draws 13 uniforms from `rng`."""
    base = np.array([0.04, 2.5, 0.04, 0.3, -0.7, 0.04, 0.5, 0.04, 0.2, -0.5, 0.15, -0.04, 0.08])
    if kind == 0:
        p = base
    elif kind == 1:
        p = np.empty(13)
        for j in range(13):                                    # dict order (:202-206)
            w = 0.15 if j in (4, 9, 11) else 0.20
            p[j] = base[j] * (1 + rng.uniform(-w, w))
        p[4] = np.clip(p[4], -0.95, -0.3)                      # :209-210
        p[9] = np.clip(p[9], -0.95, -0.3)
    else:
        strike = np.asarray(strike, dtype=float); market = np.asarray(market, dtype=float)
        maturity = np.asarray(maturity, dtype=float)
        atm = (strike / spot > 0.95) & (strike / spot < 1.05)   # :214-215
        if atm.any():
            iv = (np.mean(market[atm]) / spot) / np.sqrt(np.mean(maturity[atm]))   # :218-221
            iv = max(0.01, min(0.1, iv))                        # :222
        else:
            iv = 0.04
        p = np.array([iv, 2.0, iv, 0.4, -0.6, iv, 0.7, iv, 0.25, -0.4, 0.12, -0.03, 0.07])
    return inverse_transform_params(p)


# ----------------------------------------------------------------------------------------------
# dataset generator inputs (src/data/synthetic_generator.py:98-142)
# ----------------------------------------------------------------------------------------------
def generator_draws(n, rng=np.random):
    """Host recurrence of the generator with the RNG draws hoisted out of the pricing loop.

    Per sample the reference draws: 13 uniforms (dict order, :100-102), [1 normal(0.0003, 0.01) if
    i>0, :115], then 15 normal(0, 0.02) (:141, maturity-major).  Returns params[n,13] after the
    AR(1) smoothing (:105-109), spots[n] (:112-116) and noise[n,15].
    """
    lo, hi = GENERATOR_RANGES[:, 0], GENERATOR_RANGES[:, 1]
    params = np.empty((n, N_PARAMS)); spots = np.empty(n); noise = np.empty((n, 15))
    for i in range(n):
        fresh = np.array([rng.uniform(lo[j], hi[j]) for j in range(N_PARAMS)])
        if i > 0:
            alpha = 0.9
            fresh = alpha * params[i - 1] + (1 - alpha) * fresh
            spots[i] = spots[i - 1] * (1 + rng.normal(0.0003, 0.01))
        else:
            spots[i] = 100.0
        params[i] = fresh
        noise[i] = [rng.normal(0, 0.02) for _ in range(15)]
    return params, spots, noise


# ----------------------------------------------------------------------------------------------
# counter stream of the device-resident dataset sweep (the product's definition: csrc/dhj_generate.cuh header;
# per-sample semantics of src/data/synthetic_generator.py:98-157 with draws that depend on the sample index only)
# ----------------------------------------------------------------------------------------------
_PHILOX_M0, _PHILOX_M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_PHILOX_W0, _PHILOX_W1 = 0x9E3779B9, 0xBB67AE85
COUNTER_STREAM_TAG = 0x44484A31
_MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(counter, key):
    """Philox4x32-10 (Salmon et al., SC'11; Random123).  counter[..., 4], key[..., 2] of uint32 -> uint32[..., 4]."""
    c = [np.asarray(counter[..., j], dtype=np.uint64) for j in range(4)]
    k0 = np.asarray(key[..., 0], dtype=np.uint64)
    k1 = np.asarray(key[..., 1], dtype=np.uint64)
    for _ in range(10):
        p0 = _PHILOX_M0 * c[0]
        p1 = _PHILOX_M1 * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _MASK32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _MASK32]
        k0 = (k0 + np.uint64(_PHILOX_W0)) & _MASK32
        k1 = (k1 + np.uint64(_PHILOX_W1)) & _MASK32
    return np.stack(c, axis=-1).astype(np.uint32)


def counter_words(seed, index, slot):
    """The two 64-bit words of (sample index, slot): w0 = x0 | x1 << 32, w1 = x2 | x3 << 32."""
    index = np.asarray(index, dtype=np.uint64)
    ctr = np.stack([index & _MASK32, index >> np.uint64(32), np.full(index.shape, slot, dtype=np.uint64),
                    np.full(index.shape, COUNTER_STREAM_TAG, dtype=np.uint64)], axis=-1)
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    key = np.broadcast_to(np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint64), index.shape + (2,))
    x = philox4x32_10(ctr, key).astype(np.uint64)
    return x[..., 0] | (x[..., 1] << np.uint64(32)), x[..., 2] | (x[..., 3] << np.uint64(32))


def counter_uniform(w):
    return (w >> np.uint64(11)).astype(np.float64) * 2.0 ** -53


def counter_normal_pair(seed, index, slot):
    """Box-Muller pair: u1 = ((w0 >> 11) + 1) 2^-53 in (0, 1], u2 = (w1 >> 11) 2^-53."""
    w0, w1 = counter_words(seed, index, slot)
    u1 = ((w0 >> np.uint64(11)) + np.uint64(1)).astype(np.float64) * 2.0 ** -53
    R = np.sqrt(-2.0 * np.log(u1))
    ang = 2.0 * np.pi * counter_uniform(w1)
    return R * np.cos(ang), R * np.sin(ang)


def counter_draws(seed, first, n, path_len, lo=None, hi=None, persistence=0.9, spot0=100.0, ret_mean=0.0003,
                  ret_sd=0.01, noise_sd=0.02, n_noise=15):
    """params[n,13], spots[n], noise[n,n_noise] for samples [first, first+n) of the counter stream.

    Sample i is step t = i % path_len of path i // path_len; per path the reference's recurrences
    (synthetic_generator.py:100-116): raw uniforms, AR(1) smoothing from step 1 on, spot walk from spot0.
    """
    lo = GENERATOR_RANGES[:, 0] if lo is None else np.asarray(lo, dtype=np.float64)
    hi = GENERATOR_RANGES[:, 1] if hi is None else np.asarray(hi, dtype=np.float64)
    first, n, path_len = int(first), int(n), int(path_len)
    start = (first // path_len) * path_len                    # head of the first path touched
    idx = np.arange(start, first + n, dtype=np.uint64)
    raw = np.empty((idx.size, N_PARAMS))
    for s in range(7):
        w0, w1 = counter_words(seed, idx, s)
        raw[:, 2 * s] = lo[2 * s] + (hi[2 * s] - lo[2 * s]) * counter_uniform(w0)
        if 2 * s + 1 < N_PARAMS:
            raw[:, 2 * s + 1] = lo[2 * s + 1] + (hi[2 * s + 1] - lo[2 * s + 1]) * counter_uniform(w1)
    z0, _ = counter_normal_pair(seed, idx, 7)
    ret = ret_mean + ret_sd * z0
    params = np.empty_like(raw)
    spots = np.empty(idx.size)
    t = (idx % np.uint64(path_len)).astype(np.int64)
    one_minus = 1.0 - persistence
    for r in range(idx.size):                                 # sequential inside a path, as in the reference
        if t[r] == 0:
            params[r] = raw[r]
            spots[r] = spot0
        else:
            params[r] = persistence * params[r - 1] + one_minus * raw[r]
            spots[r] = spots[r - 1] * (1.0 + ret[r])
    noise = np.empty((idx.size, n_noise))
    for c in range((n_noise + 1) // 2):
        za, zb = counter_normal_pair(seed, idx, 8 + c)
        noise[:, 2 * c] = noise_sd * za
        if 2 * c + 1 < n_noise:
            noise[:, 2 * c + 1] = noise_sd * zb
    cut = first - start
    return params[cut:], spots[cut:], noise[cut:]


def counter_generate(seed, first, n, path_len, r=GENERATOR_RATE, N=128, strikes_rel=None, maturities=None, L=10,
                     **kw):
    """Full restatement of the sweep: draws, C-oracle prices of calls on the nT x nK grid (maturity-major,
    K = K_rel * spot / 100, :123-138; the generator's 3 x 5 grid by default), market = price + noise * price
    (:141-142), loss = mean(((model - market) / market)^2) (:154-157).  One noise factor per option (slots
    8 .. 8 + (M - 1) / 2)."""
    strikes_rel = GENERATOR_STRIKES_REL if strikes_rel is None else np.asarray(strikes_rel, dtype=np.float64).ravel()
    maturities = GENERATOR_MATURITIES if maturities is None else np.asarray(maturities, dtype=np.float64).ravel()
    params, spots, noise = counter_draws(seed, first, n, path_len, n_noise=strikes_rel.size * maturities.size, **kw)
    K = np.tile(strikes_rel[None, :] * spots[:, None] / 100.0, (1, maturities.size))
    T = np.repeat(maturities, strikes_rel.size)
    model = c_price_batch(params, spots, K, T, np.ones(T.size), r, 0.0, N, L)
    market = model + noise * model
    loss = np.mean(((model - market) / market) ** 2, axis=1)
    return {"params": params, "spots": spots, "noise": noise, "model": model, "market": market, "loss": loss}


# ----------------------------------------------------------------------------------------------
# C restatement (oracle/cos_oracle.c), OpenMP over options: same arithmetic as the scalar port, ~1000x faster
# ----------------------------------------------------------------------------------------------
_C_LIB = None


def c_library(build=True):
    """ctypes handle of oracle/_build/liboracle.so (built on demand with `make -C oracle`)."""
    global _C_LIB
    if _C_LIB is not None:
        return _C_LIB
    import ctypes
    import os
    import subprocess
    from numpy.ctypeslib import ndpointer
    here = os.path.dirname(os.path.abspath(__file__))
    path = os.path.join(here, "_build", "liboracle.so")
    if build and (not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(os.path.join(here, "cos_oracle.c"))):
        subprocess.run(["make", "-C", here], check=True, capture_output=True)
    lib = ctypes.CDLL(path)
    D = ndpointer(np.float64, flags="C_CONTIGUOUS")
    I = ndpointer(np.int32, flags="C_CONTIGUOUS")
    lib.oracle_price_list.argtypes = [D, ctypes.c_int64, D, ctypes.c_int64, D, ctypes.c_int64, D, I, ctypes.c_int32,
                                      ctypes.c_double, ctypes.c_double, ctypes.c_int32, ctypes.c_double, D,
                                      ctypes.c_void_p]
    lib.oracle_loss_batch.argtypes = [D, ctypes.c_int64, ctypes.c_double, ctypes.c_double, D, D, I, D, ctypes.c_int32,
                                      ctypes.c_int32, D]
    lib.oracle_threads.restype = ctypes.c_int
    _C_LIB = lib
    return lib


def c_price_batch(params, S0, strike, maturity, is_call, r, q=0.0, N=128, L=10, return_ab=False):
    """price_batch through the C restatement: float64[P, M]."""
    lib = c_library()
    params = np.ascontiguousarray(params, dtype=np.float64).reshape(-1, N_PARAMS)
    P = params.shape[0]
    maturity = np.ascontiguousarray(maturity, dtype=np.float64).reshape(-1)
    M = maturity.size
    S0 = np.ascontiguousarray(np.broadcast_to(np.asarray(S0, dtype=np.float64), (P,)))
    strike = np.ascontiguousarray(np.broadcast_to(np.asarray(strike, dtype=np.float64), (P, M)))
    call = np.ascontiguousarray(np.broadcast_to(np.asarray(is_call), (M,)).astype(bool).astype(np.int32))
    out = np.empty((P, M))
    ab = np.empty((P, M, 2)) if return_ab else None
    lib.oracle_price_list(params, P, S0, 1, strike, M, maturity, call, M, float(r), float(q), int(N), float(L), out,
                          ab.ctypes.data if return_ab else None)
    return (out, ab) if return_ab else out


def c_loss_batch(x, spot, r, strike, maturity, is_call, market, N=128):
    lib = c_library()
    x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, N_PARAMS)
    maturity = np.ascontiguousarray(maturity, dtype=np.float64).reshape(-1)
    out = np.empty(x.shape[0])
    lib.oracle_loss_batch(x, x.shape[0], float(spot), float(r), np.ascontiguousarray(strike, dtype=np.float64),
                          maturity, np.ascontiguousarray(np.asarray(is_call).astype(bool).astype(np.int32)),
                          np.ascontiguousarray(market, dtype=np.float64), maturity.size, int(N), out)
    return out
