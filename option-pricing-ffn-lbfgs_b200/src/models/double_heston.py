"""Drop-in replacement for the reference's `src/models/double_heston.py`, computed on a B200.

Same class, constructor signature, attribute names and method names as the reference
(/root/reference/src/models/double_heston.py:8-192).  Every method evaluates on the GPU through
libdhj.so (ctypes, include/dhj.h); there is no NumPy re-implementation here and no CPU fallback: if
the library or the device is missing, construction of the first object raises `dhj.NativeError`.

`monte_carlo` (extension) prices the same option's path-dependent variants (Asian, discretely monitored barriers) by
simulation on the device.

One object still prices ONE option, as in the reference; batches should use `dhj.Context.price_grid`
/ `price_list` (or the calibrator / generator drop-ins, which batch internally).
"""
import os
import sys

import numpy as np

_PKG_ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if _PKG_ROOT not in sys.path:
    sys.path.insert(0, _PKG_ROOT)

from dhj import GREEKS, default_context  # noqa: E402


class DoubleHeston():
    """Double Heston + Merton-jump European option pricer (COS method) — GPU-backed drop-in.

    Parameters follow the reference (double_heston.py:26-27):
    S0, K, T, r, v01, kappa1, theta1, sigma1, rho1, v02, kappa2, theta2, sigma2, rho2,
    lambda_j, mu_j, sigma_j, option_type="C", q=0.0
    """

    def __init__(self, S0, K, T, r, v01, kappa1, theta1, sigma1, rho1,
                 v02, kappa2, theta2, sigma2, rho2, lambda_j, mu_j, sigma_j, option_type="C", q=0.0):
        self.S0 = S0
        self.K = K
        self.T = T
        self.r = r
        self.q = q
        self.v01 = v01
        self.kappa1 = kappa1
        self.theta1 = theta1
        self.sigma1 = sigma1
        self.rho1 = rho1
        self.v02 = v02
        self.kappa2 = kappa2
        self.theta2 = theta2
        self.sigma2 = sigma2
        self.rho2 = rho2
        self.option_type = option_type
        self.lambda_j = lambda_j
        self.mu_j = mu_j
        self.sigma_j = sigma_j
        self._ctx = default_context()

    # -- helpers ----------------------------------------------------------------------------------
    def _params(self):
        return np.array([self.v01, self.kappa1, self.theta1, self.sigma1, self.rho1,
                         self.v02, self.kappa2, self.theta2, self.sigma2, self.rho2,
                         self.lambda_j, self.mu_j, self.sigma_j], dtype=np.float64)

    def _is_call(self):
        # any string whose first letter upper-cases to 'C' is a call, everything else a put
        # (double_heston.py:172)
        return self.option_type.upper()[0] == 'C'

    # -- reference API ----------------------------------------------------------------------------
    def characteristic_function(self, phi, tau):
        """phi(u; tau) of the log-return (double_heston.py:48-97); scalar or array `phi`, real or complex."""
        arr = np.asarray(phi)
        arr = arr.astype(np.complex128) if np.iscomplexobj(arr) else arr.astype(np.float64)
        cf = self._ctx.cf(self._params(), self.r, self.q, tau, arr)
        return cf if np.ndim(phi) else np.complex128(cf)

    def truncationRange(self, L=10):
        """(a, b) = c1 -+ L sqrt|c2|, widened to cover log(K/S0) +- 0.1 (double_heston.py:100-139)."""
        ab = self._ctx.truncation_range(self._params(), self.S0, [self.K], [self.T], self.r, L)[0, 0]
        return np.float64(ab[0]), np.float64(ab[1])

    def chi_k(self, k, c, d, a, b):
        """double_heston.py:141-151"""
        chi, _ = self._ctx.chi_psi([k], c, d, a, b)
        return np.float64(chi[0])

    def psi_k(self, k, c, d, a, b):
        """double_heston.py:153-158"""
        _, psi = self._ctx.chi_psi([k], c, d, a, b)
        return np.float64(psi[0])

    def pricing(self, N=128):
        """COS price with N cosine terms (double_heston.py:160-192) — one kernel launch."""
        price = self._ctx.price_list(self._params(), self.S0, [self.K], [self.T], [self._is_call()],
                                     self.r, self.q, N)
        return np.float64(price[0, 0])

    def pricing_gradient(self, N=128):
        """float64[13]: d pricing(N) / d(v01, kappa1, theta1, sigma1, rho1, v02, kappa2, theta2, sigma2, rho2,
        lambda_j, mu_j, sigma_j), exact with the truncation range held at its value for the current parameters
        (extension, not in the reference) — one kernel launch."""
        _, jac = self._ctx.price_jacobian(self._params(), self.S0, [self.K], [self.T], [self._is_call()], self.r,
                                          self.q, N)
        return jac[0, 0].copy()

    def greeks(self, N=128):
        """{"delta", "gamma", "theta", "rho", "rho_q"}: dV/dS0, d2V/dS0^2, -dV/dT (per year), dV/dr and dV/dq of
        pricing(N), exact with the truncation range held at its value for the current inputs (extension, not in the
        reference) — one kernel launch."""
        _, g = self._ctx.price_greeks(self._params(), self.S0, [self.K], [self.T], [self._is_call()], self.r, self.q,
                                      N)
        return {name: np.float64(g[0, 0, i]) for i, name in enumerate(GREEKS)}

    def implied_volatility(self, N=128):
        """Black–Scholes implied volatility of pricing(N) at the same S0, K, T, r, q and option type (extension, not
        in the reference): NaN where the COS price lies outside the no-arbitrage bounds — two kernel launches."""
        price = self._ctx.price_list(self._params(), self.S0, [self.K], [self.T], [self._is_call()], self.r, self.q, N)
        vol = self._ctx.implied_vol(price, self.S0, [self.K], [self.T], [self._is_call()], self.r, self.q)
        return np.float64(vol[0, 0])

    def monte_carlo(self, kind="european", barrier=None, n_paths=1 << 20, n_steps=None, n_obs=None, seed=0):
        """(price, stderr): Monte Carlo price of a path-dependent option at the same S0, K, T, r, q and option type
        (extension, not in the reference).  kind: one of dhj.MC_KINDS ("european", "asian", "up-and-out",
        "up-and-in", "down-and-out", "down-and-in"); barrier B for the barrier kinds; n_steps equal steps of the
        full-truncation Euler scheme (default ceil(252 T)); n_obs observation dates for the average and the barrier
        (default every step; must divide n_steps).  The scheme is discrete: see dhj.Context.mc_price."""
        if n_steps is None:
            n_steps = max(1, int(np.ceil(252 * self.T)))
        price, err = self._ctx.mc_price(self._params(), self.S0, self.T, [kind], [self._is_call()], [self.K], self.r,
                                        self.q, None if barrier is None else [barrier], n_paths, n_steps, n_obs, seed)
        return np.float64(price[0, 0]), np.float64(err[0, 0])
