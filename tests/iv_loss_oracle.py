"""CPU oracle of the implied-volatility calibration objective (DESIGN.md §6e).  TEST INFRASTRUCTURE ONLY.

    f(x) = (1/M_v) sum_{o valid} (sigma_o(x) - sigma^_o)^2 + Feller(p(x))
    g    = (2/M_v) sum_{o valid} (sigma_o - sigma^_o) (dV_o/dp) / vega_o  dp/dx + dFeller/dp dp/dx

* prices and dV/dp: tests/jac_oracle.py's frozen-range price Jacobian (dual numbers through the reference's CF);
* sigma and vega: tests/iv_oracle.py (Black–Scholes in mpmath at 40 digits, every double input exact), q = 0;
* a quote is valid when its price lies strictly inside the no-arbitrage bounds (status 0); the others are left out;
* (1e10, 0) when a valid option's model price is NaN, inf or <= 0, lies outside the bounds, or has a vega that is not
  a positive normal double.
"""
from __future__ import annotations

import numpy as np

import iv_oracle as V
import jac_oracle as J
import oracle.cos_oracle as O

TINY = 2.2250738585072014e-308


def iv_status(price, S0, K, T, r, call):
    """0 inside the bounds (q = 0): D max(+-(F - K), 0) <= V < S0 (call) / K e^{-rT} (put); 1 below, 2 at or above,
    3 invalid — the status rule of dhj_implied_vol, on the same doubles."""
    if not np.isfinite(price):
        return 3
    KD = K * np.exp(-r * T)
    lower = max(S0 - KD, 0.0) if call else max(KD - S0, 0.0)
    upper = S0 if call else KD
    if price < lower:
        return 1
    if price >= upper:
        return 2
    return 0


def implied_vols(prices, S0, K, T, r, call, guess=None):
    """(sigma[M], vega[M], status[M]) of one row of prices; NaN where status != 0 (sigma = 0 at the lower bound)."""
    M = len(prices)
    sig, veg, st = np.full(M, np.nan), np.full(M, np.nan), np.zeros(M, dtype=np.int32)
    for o in range(M):
        st[o] = iv_status(prices[o], S0, K[o], T[o], r, bool(call[o]))
        if st[o]:
            continue
        if prices[o] == (max(S0 - K[o] * np.exp(-r * T[o]), 0.0) if call[o] else max(K[o] * np.exp(-r * T[o]) - S0, 0.0)):
            sig[o], veg[o] = 0.0, 0.0
            continue
        g = 0.3 if guess is None or not np.isfinite(guess[o]) else guess[o]
        s = V.implied_vol(prices[o], S0, K[o], T[o], r, 0.0, bool(call[o]), g)
        sig[o] = float(s)
        veg[o] = float(V.bs_vega(S0, K[o], T[o], r, 0.0, s))
    return sig, veg, st


def market_vols(spot, r, strike, maturity, is_call, market):
    """(sigma^[M], status[M]) of the market's quotes: NaN where the quote is left out (status != 0)."""
    s, _, st = implied_vols(np.asarray(market, dtype=np.float64), float(spot), np.asarray(strike, dtype=np.float64),
                            np.asarray(maturity, dtype=np.float64), r, np.asarray(is_call).astype(bool))
    return s, st


def _objective(sig, veg, mvol, prices):
    """(f_data, weights, bad) of one state: the data term, (sigma - sigma^) / vega per option and the sentinel flag."""
    valid = ~np.isnan(mvol)
    with np.errstate(all="ignore"):
        bad = bool(np.any(valid & (~np.isfinite(prices) | (prices <= 0) | np.isnan(sig) | ~(veg >= TINY)
                                   | np.isinf(veg))))
        d = np.where(valid, sig - mvol, 0.0)
        return np.sum(d * d) / valid.sum(), np.where(valid, d / veg, 0.0), bad


def iv_loss_grad_batch(x, spot, r, strike, maturity, is_call, market, N=128, mvol=None):
    """(f[B], g[B, 13]) of the IV objective and its exact gradient in the unconstrained x, frozen range; (1e10, 0) at
    the sentinel.  mvol: the market vols (market_vols(...)[0]) if already known."""
    x = np.asarray(x, dtype=np.float64).reshape(-1, O.N_PARAMS)
    K, T = np.asarray(strike, dtype=np.float64), np.asarray(maturity, dtype=np.float64)
    call = np.asarray(is_call).astype(bool)
    if mvol is None:
        mvol, _ = market_vols(spot, r, K, T, call, market)
    if not (~np.isnan(mvol)).any():
        raise ValueError("no quote has an implied vol")
    p = O.transform_params(x)
    prices, jac = J.price_jacobian_batch(p, spot, K, T, call, r, 0.0, N)
    f, g = np.empty(len(x)), np.zeros((len(x), O.N_PARAMS))
    Mv = (~np.isnan(mvol)).sum()
    for b in range(len(x)):
        with np.errstate(all="ignore"):
            sig, veg, _ = implied_vols(prices[b], float(spot), K, T, r, call, guess=mvol)
        data, w, bad = _objective(sig, veg, mvol, prices[b])
        if bad or not np.isfinite(p[b]).all():
            f[b] = O.SENTINEL
            continue
        f[b] = data + O.feller_penalty(p[b])
        gp = (2.0 / Mv) * (w @ jac[b]) + J.feller_gradient(p[b])
        g[b] = gp * J.transform_jacobian(x[b])
    return f, g


def iv_loss_frozen(x, spot, r, strike, maturity, is_call, mvol, ab, N=128, guess=None):
    """f[B] with the truncation range frozen at ab[M, 2] (the range of the state being differentiated)."""
    x = np.asarray(x, dtype=np.float64).reshape(-1, O.N_PARAMS)
    K, T = np.asarray(strike, dtype=np.float64), np.asarray(maturity, dtype=np.float64)
    call = np.asarray(is_call).astype(bool)
    p = O.transform_params(x)
    prices = J.price_batch_frozen(p, spot, K, T, call, r, np.broadcast_to(ab, (len(x),) + ab.shape), 0.0, N)
    out = np.empty(len(x))
    for b in range(len(x)):
        with np.errstate(all="ignore"):
            sig, veg, _ = implied_vols(prices[b], float(spot), K, T, r, call, guess=guess if guess is not None else mvol)
        data, _, bad = _objective(sig, veg, mvol, prices[b])
        out[b] = O.SENTINEL if bad else data + O.feller_penalty(p[b])
    return out
