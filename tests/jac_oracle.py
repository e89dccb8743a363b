"""CPU oracle of the analytic parameter gradient.  TEST INFRASTRUCTURE ONLY.

Extends the pinned oracle (oracle/cos_oracle.py, left unchanged) with the derivatives the device computes:

* `price_batch_frozen`   COS prices with the truncation range [a, b] given (the reference formulas otherwise);
* `price_jacobian_batch` prices and d price / d(13 model parameters) with [a, b] held at its value for the
                         current parameters ("frozen range"), by forward-mode dual numbers through the reference's own
                         CF formula (with g = (beta - d)/(beta + d) and log((1 - gE)/(1 - g)), not the device's
                         rearranged algebra), contracted against the reference's chi/psi payoff basis;
* `loss_grad_batch`      compute_loss and its exact gradient in the unconstrained x (Feller term 0 at the kink,
                         (1e10, 0) at the sentinel).
"""
from __future__ import annotations

import numpy as np

import oracle.cos_oracle as O

N_PARAMS = O.N_PARAMS


class Dual:
    """value[...] and derivatives der[13, ...] (complex), propagated by the chain rule."""
    __slots__ = ("v", "d")

    def __init__(self, v, d):
        self.v, self.d = v, d

    @staticmethod
    def _lift(o):
        return o if isinstance(o, Dual) else Dual(o, 0.0)

    def __add__(self, o):
        o = Dual._lift(o)
        return Dual(self.v + o.v, self.d + o.d)
    __radd__ = __add__

    def __sub__(self, o):
        o = Dual._lift(o)
        return Dual(self.v - o.v, self.d - o.d)

    def __rsub__(self, o):
        return Dual._lift(o) - self

    def __neg__(self):
        return Dual(-self.v, -self.d)

    def __mul__(self, o):
        o = Dual._lift(o)
        return Dual(self.v * o.v, self.d * o.v + self.v * o.d)
    __rmul__ = __mul__

    def __truediv__(self, o):
        o = Dual._lift(o)
        q = self.v / o.v
        return Dual(q, (self.d - q * o.d) / o.v)

    def __rtruediv__(self, o):
        return Dual._lift(o) / self

    def exp(self):
        e = np.exp(self.v)
        return Dual(e, e * self.d)

    def log(self):
        return Dual(np.log(self.v), self.d / self.v)

    def sqrt(self):
        s = np.sqrt(self.v)
        return Dual(s, self.d / (2.0 * s))


def _params_dual(params):
    """params[..., 13] -> 13 Duals seeded with the unit tangents, shaped for broadcasting against [..., N]."""
    out = []
    for j in range(N_PARAMS):
        v = params[..., j, None]
        d = np.zeros((N_PARAMS,) + v.shape)
        d[j] = 1.0
        out.append(Dual(v, d))
    return out


def _heston_factor_dual(u, tau, v0, kappa, theta, sigma, rho):
    """_heston_factor_vec (double_heston.py:64-71, 85-87) in dual numbers."""
    i = 1j
    beta = kappa - rho * sigma * (i * u)
    d = (beta * beta + sigma * sigma * (u * (u + i))).sqrt()
    g = (beta - d) / (beta + d)
    E = (-(d * tau)).exp()
    B = ((beta - d) / (sigma * sigma)) * ((1 - E) / (1 - g * E))
    A = (kappa * theta / (sigma * sigma)) * ((beta - d) * tau - 2 * ((1 - g * E) / (1 - g)).log())
    return A, B


def cf_dual(u, tau, params, r, q=0.0):
    """cf_vec (double_heston.py:48-97) with d phi / d params: a Dual of shape u.shape, der[13, ...]."""
    v01, k1, t1, s1, rho1, v02, k2, t2, s2, rho2, lam, mu, sj = _params_dual(params)
    i = 1j
    A1, B1 = _heston_factor_dual(u, tau, v01, k1, t1, s1, rho1)
    A2, B2 = _heston_factor_dual(u, tau, v02, k2, t2, s2, rho2)
    compensator = (mu + 0.5 * (sj * sj)).exp() - 1
    A = (r - q - lam * compensator) * (i * u * tau)
    A = A + A1
    A = A + A2
    jump = (lam * tau) * ((mu * (i * u) - 0.5 * (sj * sj) * (u ** 2)).exp() - 1)
    return (A + B1 * v01 + B2 * v02 + jump).exp()


def _basis(S0, K, T, call, a, b, r, N):
    """u[p,M,N] and the discounted payoff basis exp(-rT) (2/(b-a)) V_k with the k = 0 weight 1/2 (price_batch)."""
    kk = np.arange(N)
    x = np.log(K / S0)
    u = kk[None, None, :] * np.pi / (b - a)[..., None]
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
    V = (2.0 / (b - a))[..., None] * (sgn * (S0[..., None] * chi - K[..., None] * psi))
    V[..., 0] *= 0.5
    return u, np.exp(-r * T)[..., None] * V


def _prepare(params, S0, strike, maturity, is_call):
    params = np.asarray(params, dtype=np.float64).reshape(-1, N_PARAMS)
    P = params.shape[0]
    maturity = np.asarray(maturity, dtype=np.float64).reshape(-1)
    M = maturity.shape[0]
    S0 = np.broadcast_to(np.asarray(S0, dtype=np.float64), (P,))
    strike = np.broadcast_to(np.asarray(strike, dtype=np.float64), (P, M))
    call = np.broadcast_to(np.asarray(is_call).astype(bool), (M,))
    return params, P, S0, strike, maturity, M, call


def price_batch_frozen(params, S0, strike, maturity, is_call, r, ab, q=0.0, N=128):
    """COS prices float64[P, M] with the truncation range given: ab[P, M, 2]."""
    params, P, S0, strike, maturity, M, call = _prepare(params, S0, strike, maturity, is_call)
    ab = np.broadcast_to(np.asarray(ab, dtype=np.float64), (P, M, 2))
    with np.errstate(all="ignore"):
        a, b = ab[..., 0], ab[..., 1]
        u, W = _basis(S0[:, None], strike, maturity[None, :], call, a, b, r, N)
        phi = O.cf_vec(u, maturity[None, :, None], params[:, None, :], r, q)
        return np.sum(np.real(phi * np.exp(-1j * u * a[..., None])) * W, axis=-1)


def price_jacobian_batch(params, S0, strike, maturity, is_call, r, q=0.0, N=128, L=10, chunk=8):
    """(prices[P, M], jac[P, M, 13]): COS prices and their exact derivatives in the 13 model parameters with the
    truncation range frozen at its value for `params`."""
    params, P, S0, strike, maturity, M, call = _prepare(params, S0, strike, maturity, is_call)
    prices, jac = np.empty((P, M)), np.empty((P, M, N_PARAMS))
    for lo in range(0, P, chunk):
        hi = min(P, lo + chunk)
        pr = params[lo:hi, None, :]
        s0 = S0[lo:hi, None]
        K = strike[lo:hi]
        T = maturity[None, :]
        with np.errstate(all="ignore"):
            a, b = O.truncation_range_vec(pr, s0, K, T, r, L)
            u, W = _basis(s0, K, T, call, a, b, r, N)
            phi = cf_dual(u, T[..., None], pr, r, q)
            rot = np.exp(-1j * u * a[..., None])
            prices[lo:hi] = np.sum(np.real(phi.v * rot) * W, axis=-1)
            jac[lo:hi] = np.moveaxis(np.sum(np.real(phi.d * rot) * W, axis=-1), 0, -1)
    return prices, jac


def transform_jacobian(x):
    """d p / d x of the calibrator's transform (diagonal): p for exp parameters, 1 - rho^2 for tanh, 1 for mu_j."""
    p = O.transform_params(x)
    dp = p.copy()
    dp[..., 4] = 1.0 - p[..., 4] ** 2
    dp[..., 9] = 1.0 - p[..., 9] ** 2
    dp[..., 11] = 1.0
    return dp


def feller_gradient(p):
    """d Feller / d p: 1000 (2 sigma, -2 theta, -2 kappa) per factor whose excess is > 0 (0 at and below the kink)."""
    p = np.asarray(p, dtype=np.float64)
    g = np.zeros_like(p)
    for f in range(2):
        k, t, s = p[..., 5 * f + 1], p[..., 5 * f + 2], p[..., 5 * f + 3]
        with np.errstate(all="ignore"):
            on = (s * s - 2 * k * t) > 0
        g[..., 5 * f + 3] = np.where(on, 2000.0 * s, 0.0)
        g[..., 5 * f + 1] = np.where(on, -2000.0 * t, 0.0)
        g[..., 5 * f + 2] = np.where(on, -2000.0 * k, 0.0)
    return g


def loss_grad_batch(x, spot, r, strike, maturity, is_call, market, N=128):
    """(f[B], g[B, 13]): compute_loss (loss_batch) and its exact gradient in the unconstrained x, frozen range;
    (1e10, 0) where the loss is the sentinel."""
    x = np.asarray(x, dtype=np.float64).reshape(-1, N_PARAMS)
    p = O.transform_params(x)
    prices, jac = price_jacobian_batch(p, spot, strike, maturity, is_call, r, 0.0, N)
    market = np.broadcast_to(np.asarray(market, dtype=np.float64), prices.shape)
    M = prices.shape[1]
    with np.errstate(all="ignore"):
        bad = np.any(~np.isfinite(prices) | (prices <= 0), axis=1)
        rel = (prices - market) / market
        f = np.mean(rel ** 2, axis=1) + O.feller_penalty(p)
        gp = (2.0 / M) * np.einsum("bm,bmi->bi", rel / market, jac) + feller_gradient(p)
        g = gp * transform_jacobian(x)
    return np.where(bad, O.SENTINEL, f), np.where(bad[:, None], 0.0, g)
