"""Black–Scholes reference for the implied-volatility tests: price, vega and the implied-vol root in mpmath at 40
digits, with every double input taken as exact.

The accuracy measure of an implied vol sigma against the exact root sigma* of the same double price V is
    c = |sigma - sigma*| / (eps * (sigma* + V / vega)),   eps = 2^-52,
where V / vega is the option's own conditioning: a relative change of eps in V moves sigma* by eps * V / vega."""
import mpmath as mp
import numpy as np

EPS = 2.0 ** -52
mp.mp.dps = 40


def _mp(v):
    return v if isinstance(v, mp.mpf) else mp.mpf(float(v))


def _ncdf(z):
    return mp.erfc(-z / mp.sqrt(2)) / 2


def bs_price(S0, K, T, r, q, sigma, call):
    """Black–Scholes price (mpf) of a European option; sigma = 0 gives the discounted intrinsic value."""
    S0, K, T, r, q, sigma = (_mp(v) for v in (S0, K, T, r, q, sigma))
    F, D = S0 * mp.exp((r - q) * T), mp.exp(-r * T)
    if sigma == 0:
        return D * max((F - K) if call else (K - F), mp.mpf(0))
    s = sigma * mp.sqrt(T)
    d1 = (mp.log(F / K) + s * s / 2) / s
    d2 = d1 - s
    if call:
        return D * (F * _ncdf(d1) - K * _ncdf(d2))
    return D * (K * _ncdf(-d2) - F * _ncdf(-d1))


def bs_vega(S0, K, T, r, q, sigma):
    """dV/dsigma (mpf), the same for calls and puts."""
    S0, K, T, r, q, sigma = (_mp(v) for v in (S0, K, T, r, q, sigma))
    F, D = S0 * mp.exp((r - q) * T), mp.exp(-r * T)
    s = sigma * mp.sqrt(T)
    d1 = (mp.log(F / K) + s * s / 2) / s
    return D * F * mp.npdf(d1) * mp.sqrt(T)


def implied_vol(V, S0, K, T, r, q, call, guess):
    """sigma* (mpf) with bs_price(sigma*) == V exactly (V a double, taken as exact): Newton in sigma from `guess`
    with bisection safeguards, until the step is below 1e-28 (sigma + V / vega)."""
    V = mp.mpf(float(V))
    lo, hi = mp.mpf(0), mp.mpf("inf")
    x = mp.mpf(float(guess))
    for _ in range(200):
        f = bs_price(S0, K, T, r, q, x, call) - V
        if f == 0:
            return x
        if f > 0:
            hi = x
        else:
            lo = x
        vega = bs_vega(S0, K, T, r, q, x)
        xn = x - f / vega
        if not (lo < xn < hi):
            xn = (lo + hi) / 2 if hi < mp.inf else 2 * x
        if abs(xn - x) <= mp.mpf(10) ** -28 * (x + V / vega):
            return xn
        x = xn
    raise RuntimeError("implied_vol reference did not converge")


def c_measure(sigma, V, S0, K, T, r, q, call, sigma_true):
    """(c, sigma*) of a computed vol `sigma` for the double price V (module docstring)."""
    star = implied_vol(V, S0, K, T, r, q, call, sigma_true)
    vega = bs_vega(S0, K, T, r, q, star)
    c = abs(mp.mpf(float(sigma)) - star) / (EPS * (star + mp.mpf(float(V)) / vega))
    return float(c), float(star)


def domain_a(n, seed):
    """The round-trip domain: sigma log-uniform on [0.01, 3], T log-uniform on [1/365, 10], z = ln(F/K)/(sigma sqrt T)
    uniform on [-6, 6], r on [-0.02, 0.10], q on [0, 0.05], S0 in {1, 100, 1e4}, calls and puts.  Returns a dict of
    n float64 / int32 arrays with V = BS(sigma) evaluated in mpmath and rounded to a double.

    A deep in-the-money option whose time value is below 64 ulp of its price is redrawn: its double price carries
    no information about sigma (it may even round below the exact intrinsic value, where no root exists)."""
    rng = np.random.default_rng(seed)
    cols = {k: [] for k in ("sigma", "T", "r", "q", "S0", "K", "call", "V")}
    while len(cols["V"]) < n:
        sigma = float(np.exp(rng.uniform(np.log(0.01), np.log(3.0))))
        T = float(np.exp(rng.uniform(np.log(1 / 365), np.log(10.0))))
        z = rng.uniform(-6.0, 6.0)
        r, q = rng.uniform(-0.02, 0.10), rng.uniform(0.0, 0.05)
        S0 = float(rng.choice([1.0, 100.0, 1e4]))
        call = int(rng.integers(0, 2))
        K = float(S0 * np.exp((r - q) * T - z * sigma * np.sqrt(T)))
        Vm = bs_price(S0, K, T, r, q, sigma, call)
        V = float(Vm)
        if Vm - bs_price(S0, K, T, r, q, 0.0, call) <= 64 * np.spacing(V):
            continue
        for k, v in zip(cols, (sigma, T, r, q, S0, K, call, V)):
            cols[k].append(v)
    out = {k: np.array(v, dtype=np.float64) for k, v in cols.items()}
    out["call"] = out["call"].astype(np.int32)
    return out
