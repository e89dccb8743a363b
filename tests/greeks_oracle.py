"""CPU oracle of the Greeks (dhj_price_greeks).  TEST INFRASTRUCTURE ONLY.

Builds on tests/jac_oracle.py (left unchanged) and the pinned oracle:

* theta, rho, rho_q: forward-mode dual numbers seeded in (T, r, q) through the reference's own CF formula, the
  truncation range [a, b] held at its value for the current inputs (the frozen range), the discount exp(-rT)
  differentiated with it;
* delta, gamma: the analytic S0-derivatives of the payoff basis (jac_oracle._basis): with x = log(K/S0)
      d/dS0 [S0 chi_k(x, b) - K psi_k(x, b)] = chi_k(x, b)         (call; put: -chi_k(a, x))
      d/dS0 chi_k(x, b) = (K / S0^2) cos(u_k (x - a))              (put: the same)
  because the payoff integrand (S0 e^y - K) cos(u_k (y - a)) is 0 at y = x.

`greeks_batch` returns (prices[P, M], greeks[P, M, 5]) in the library's order: delta, gamma, theta, rho, rho_q.
"""
from __future__ import annotations

import numpy as np

import oracle.cos_oracle as O
from jac_oracle import Dual, _basis, _heston_factor_dual, _prepare

N_PARAMS = O.N_PARAMS
GREEKS = ("delta", "gamma", "theta", "rho", "rho_q")


def cf_time_dual(u, tau, params, r, q):
    """cf_vec (double_heston.py:48-97) with tau, r, q Duals (derivatives der[3, ...] in T, r, q); params plain."""
    v01, k1, t1, s1, rho1, v02, k2, t2, s2, rho2, lam, mu, sj = [Dual(params[..., j, None], 0.0)
                                                                   for j in range(N_PARAMS)]
    A1, B1 = _heston_factor_dual(u, tau, v01, k1, t1, s1, rho1)
    A2, B2 = _heston_factor_dual(u, tau, v02, k2, t2, s2, rho2)
    compensator = (mu + 0.5 * (sj * sj)).exp() - 1
    A = (r - q - lam * compensator) * (tau * (1j * u))
    A = A + A1
    A = A + A2
    jump = (lam * tau) * ((mu * (1j * u) - 0.5 * (sj * sj) * (u ** 2)).exp() - 1)
    return (A + B1 * v01 + B2 * v02 + jump).exp()


def _spot_basis(S0, K, call, a, b, N):
    """(2/(b-a)) w_k d V_k / dS0 and (2/(b-a)) w_k d^2 V_k / dS0^2 of the undiscounted payoff basis, [p, M, N]."""
    kk = np.arange(N)
    x = np.log(K / S0)
    u = kk[None, None, :] * np.pi / (b - a)[..., None]
    c = np.where(call[None, :], x, a)[..., None]
    d = np.where(call[None, :], b, x)[..., None]
    a3 = a[..., None]
    ed, ec = np.exp(d), np.exp(c)
    chi = (1.0 / (1 + u ** 2)) * (np.cos(u * (d - a3)) * ed - np.cos(u * (c - a3)) * ec
                                  + u * np.sin(u * (d - a3)) * ed - u * np.sin(u * (c - a3)) * ec)
    chi[..., 0] = (ed - ec)[..., 0]
    tw = (2.0 / (b - a))[..., None]
    sgn = np.where(call, 1.0, -1.0)[None, :, None]
    D1 = tw * sgn * chi
    D2 = tw * (K / S0 ** 2)[..., None] * np.cos(u * (x[..., None] - a3))
    D1[..., 0] *= 0.5
    D2[..., 0] *= 0.5
    return D1, D2


def greeks_batch(params, S0, strike, maturity, is_call, r, q=0.0, N=128, L=10, chunk=8):
    """(prices[P, M], greeks[P, M, 5]) with the truncation range frozen at its value for the inputs."""
    params, P, S0, strike, maturity, M, call = _prepare(params, S0, strike, maturity, is_call)
    prices, greeks = np.empty((P, M)), np.empty((P, M, 5))
    seed = np.eye(3).reshape(3, 3, 1, 1, 1)                     # seed[i]: unit tangent in T, r or q
    for lo in range(0, P, chunk):
        hi = min(P, lo + chunk)
        pr = params[lo:hi, None, :]
        s0 = S0[lo:hi, None]
        K = strike[lo:hi]
        T = maturity[None, :]
        with np.errstate(all="ignore"):
            a, b = O.truncation_range_vec(pr, s0, K, T, r, L)
            u, W = _basis(s0, K, T, call, a, b, 0.0, N)            # undiscounted (exp(-0 T) = 1)
            D1, D2 = _spot_basis(s0, K, call, a, b, N)
            tau = Dual(np.broadcast_to(T[..., None], (1, M, 1)), seed[0])
            phi = cf_time_dual(u, tau, pr, Dual(r, seed[1]), Dual(q, seed[2]))
            rot = np.exp(-1j * u * a[..., None])
            g = np.real(phi.v * rot)
            s = np.sum(g * W, axis=-1)
            ds = np.sum(np.real(phi.d * rot) * W, axis=-1)            # [3, p, M]: d/dT, d/dr, d/dq at fixed disc
            disc = np.exp(-r * T)
            V = disc * s
            prices[lo:hi] = V
            greeks[lo:hi, :, 0] = disc * np.sum(g * D1, axis=-1)
            greeks[lo:hi, :, 1] = disc * np.sum(g * D2, axis=-1)
            greeks[lo:hi, :, 2] = -(disc * ds[0] - r * V)
            greeks[lo:hi, :, 3] = disc * ds[1] - T * V
            greeks[lo:hi, :, 4] = disc * ds[2]
    return prices, greeks


def binding(params, S0, strike, maturity, r, L=10):
    """[P, M] True where the strike's +-0.1 widening sets a or b (its own range then moves with S0)."""
    params, P, S0, strike, maturity, M, _ = _prepare(params, S0, strike, maturity, np.ones(1))
    with np.errstate(all="ignore"):
        a, b = O.truncation_range_vec(params[:, None, :], S0[:, None], strike, maturity[None, :], r, L)
        x = np.log(strike / S0[:, None])
        return (a == x - 0.1) | (b == x + 0.1)
