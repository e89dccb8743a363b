"""Drop-in replacement for the reference's `src/calibration/lbfgs_calibrator.py`, with the loss and the
finite-difference gradient evaluated on a B200.

Same public surface as the reference (/root/reference/src/calibration/lbfgs_calibrator.py):
`CalibrationResult` (:21-41) and `DoubleHestonJumpCalibrator(spot, risk_free_rate, market_options)` with
`transform_params`, `inverse_transform_params`, `compute_feller_penalty`, `compute_loss`,
`get_initial_guess`, `calibrate(maxiter=300, multi_start=3)` and the attributes `param_names`,
`market_prices`, `n_calls`, `best_loss` (:47-60).

What changes underneath:
  * `compute_loss(x)` is one kernel launch that prices every market option (libdhj `dhj_loss_batch`);
  * L-BFGS-B stays scipy's, on the host, but instead of letting scipy call `compute_loss` 14 times per
    step for its forward differences, `calibrate` hands it `jac=True` and one launch returns f and
    g_i = (f(x+h e_i) - f(x)) / ((x_i+h) - x_i), h = 1e-8 — the arithmetic scipy itself does
    (`dhj_loss_fd`; scipy/optimize/_numdiff.py `_dense_difference`).  `n_calls` still advances by 14
    per step and `best_loss` still sees all 14 values;
  * the `multi_start` optimisers run in lock-step: each round's requests (one per still-running start)
    are evaluated by ONE launch.  The global NumPy RNG is consumed in the reference's order (the three
    initial guesses are drawn in start order before any optimiser runs), so seeded runs start from the
    same points.
There is no CPU path: without libdhj.so / a B200 the constructor raises `dhj.NativeError`.
"""
import sys
import threading
import time
from dataclasses import dataclass
from pathlib import Path
from typing import Dict, List

import numpy as np
from scipy.optimize import minimize
import warnings
warnings.filterwarnings('ignore')          # the reference silences warnings process-wide at import (:13-14)

sys.path.insert(0, str(Path(__file__).parent.parent / 'models'))
sys.path.insert(0, str(Path(__file__).parent.parent.parent))

from double_heston import DoubleHeston  # noqa: E402,F401  (re-exported like the reference does)
from dhj import default_context  # noqa: E402

_SENTINEL = 1e10       # :152-153
_FD_STEP = 1e-8        # scipy's L-BFGS-B `eps` default, what jac=None uses
# scipy's default maxfun = 15000 counts LOSS evaluations; with jac=None every (f, g) request costs 14 of them
# (1 + 13 forward points), so the reference stops after 1072 requests (14 * 1072 > 15000).  The drop-in answers a
# request with one call (jac=True), which scipy counts as 1: the same limit is 15000 // 14 = 1071 requests.
_MAXFUN_REQUESTS = 15000 // 14


@dataclass
class CalibrationResult:
    """Container for calibration results (field-for-field the reference's dataclass, :21-41).

    calibration_time and iterations are None for synthetic data that was not actually calibrated.
    """
    date: str
    spot: float
    risk_free: float
    parameters: Dict[str, float]
    market_prices: np.ndarray
    model_prices: np.ndarray
    market_options: List[Dict]
    final_loss: float
    calibration_time: float = None
    success: bool = True
    iterations: int = None
    message: str = ""


class _LockstepEvaluator:
    """Collects one (f, g) request per running optimiser thread and answers them with one launch."""

    def __init__(self, market, n_workers):
        self._market = market
        self._cv = threading.Condition()
        self._active = n_workers
        self._pending = {}
        self._answers = {}
        self._error = None
        self.launches = 0

    def _flush_locked(self):
        order = sorted(self._pending)
        xs = np.stack([self._pending[i] for i in order])
        self._pending.clear()
        try:
            f, g, f_all = self._market.loss_fd(xs, _FD_STEP, want_all=True)
            self.launches += 1
            for row, i in enumerate(order):
                self._answers[i] = (f[row], g[row].copy(), f_all[row].copy())
        except Exception as exc:              # a device error must surface in every waiting thread
            self._error = exc
        self._cv.notify_all()

    def request(self, worker, x):
        with self._cv:
            self._pending[worker] = np.array(x, dtype=np.float64)
            if len(self._pending) == self._active:
                self._flush_locked()
            while worker not in self._answers and self._error is None:
                self._cv.wait()
            if self._error is not None:
                raise self._error
            return self._answers.pop(worker)

    def retire(self, worker):
        with self._cv:
            self._active -= 1
            if self._pending and len(self._pending) == self._active:
                self._flush_locked()


class DoubleHestonJumpCalibrator:

    #: run the multi_start optimisers in lock-step, one launch per round (False: one after another)
    batch_starts = True

    def __init__(self, spot: float, risk_free_rate: float, market_options: List[Dict]):
        self.spot = spot
        self.risk_free_rate = risk_free_rate
        self.market_options = market_options
        self.market_prices = np.array([opt['price'] for opt in market_options])

        self.param_names = [
            'v1_0', 'kappa1', 'theta1', 'sigma1', 'rho1',
            'v2_0', 'kappa2', 'theta2', 'sigma2', 'rho2',
            'lambda_j', 'mu_j', 'sigma_j'
        ]

        self.n_calls = 0
        self.best_loss = np.inf

        self._ctx = default_context()        # created once per process, before any timed region
        self._market = None
        self._iv_market = None               # the same options on the implied-vol objective (objective="iv")

    # -- device-side market ------------------------------------------------------------------------
    def _device_market(self, objective: str = "price"):
        if objective == "iv":
            if self._iv_market is None:
                opts = self.market_options
                is_call = [str(o['option_type']).upper()[0] == 'C' for o in opts]
                mk = self._ctx.market(
                    float(self.spot), float(self.risk_free_rate),
                    [float(o['strike']) for o in opts], [float(o['maturity']) for o in opts], is_call,
                    [float(o['price']) for o in opts], N=128)
                mk.set_objective("iv")
                self._iv_market = mk
            return self._iv_market
        if objective != "price":
            raise ValueError(f"objective must be 'price' or 'iv' (got {objective!r})")
        if self._market is None:
            opts = self.market_options
            is_call = [str(o['option_type']).upper()[0] == 'C' for o in opts]     # double_heston.py:172
            self._market = self._ctx.market(
                float(self.spot), float(self.risk_free_rate),
                [float(o['strike']) for o in opts], [float(o['maturity']) for o in opts], is_call,
                [float(o['price']) for o in opts], N=128)                           # default N (:150)
        return self._market

    # -- parameter maps (host, identical to the reference) ----------------------------------------
    def transform_params(self, x: np.ndarray) -> Dict[str, float]:
        """Unconstrained optimisation variables -> model parameters (:62-87): exp, tanh for rho, mu_j as is."""
        values = np.exp(np.asarray(x, dtype=np.float64))
        values[4] = np.tanh(x[4])
        values[9] = np.tanh(x[9])
        values[11] = x[11]
        return {name: values[i] for i, name in enumerate(self.param_names)}

    def inverse_transform_params(self, params: Dict[str, float]) -> np.ndarray:
        """Model parameters -> unconstrained variables (:89-109)."""
        x = np.zeros(13)
        for i, name in enumerate(self.param_names):
            if name in ('rho1', 'rho2'):
                x[i] = np.arctanh(np.clip(params[name], -0.999, 0.999))
            elif name == 'mu_j':
                x[i] = params[name]
            else:
                x[i] = np.log(params[name])
        return x

    def compute_feller_penalty(self, params: Dict[str, float]) -> float:
        """1000 * (max(0, s1^2 - 2 k1 t1) + max(0, s2^2 - 2 k2 t2))  (:111-116)."""
        penalty1 = max(0, params['sigma1']**2 - 2*params['kappa1']*params['theta1'])
        penalty2 = max(0, params['sigma2']**2 - 2*params['kappa2']*params['theta2'])
        return 1000.0 * (penalty1 + penalty2)

    # -- loss ---------------------------------------------------------------------------------------
    def _track(self, loss):
        # the reference returns the sentinel before it reaches its best_loss update (:152-153, :171-172)
        if loss != _SENTINEL and loss < self.best_loss:
            self.best_loss = loss

    def compute_loss(self, x: np.ndarray) -> float:
        """Relative MSE + Feller penalty, 1e10 on a NaN/inf/non-positive price (:118-177). One launch."""
        self.n_calls += 1
        try:
            xv = np.ascontiguousarray(x, dtype=np.float64).reshape(13)
        except Exception:
            return _SENTINEL                 # the reference swallows malformed input the same way (:176-177)
        loss = self._device_market().loss_batch(xv)[0]
        if loss == _SENTINEL:
            return _SENTINEL
        self._track(loss)
        return loss

    def compute_loss_and_grad(self, x: np.ndarray, gradient: str = "fd", objective: str = "price"):
        """f(x) and scipy's 2-point forward-difference gradient (h = 1e-8) in ONE launch.  gradient="analytic": the
        exact gradient instead (truncation range held fixed, g = 0 at the 1e10 sentinel); `n_calls` advances by 1.
        objective="iv": f is the implied-vol objective (mean squared error of the model's Black–Scholes implied vols
        against the quotes' over the quotes that have one, + Feller; DESIGN.md §6e) instead of compute_loss."""
        market = self._device_market(objective)
        if gradient == "analytic":
            f, g = market.loss_grad(np.asarray(x, dtype=np.float64).reshape(1, 13))
            self.n_calls += 1
            self._track(f[0])
            return f[0], g[0]
        if gradient != "fd":
            raise ValueError(f"gradient must be 'fd' or 'analytic' (got {gradient!r})")
        f, g, f_all = market.loss_fd(np.asarray(x, dtype=np.float64).reshape(1, 13), _FD_STEP, want_all=True)
        self.n_calls += 14
        for v in f_all[0]:
            self._track(v)
        return f[0], g[0]

    # -- initial guesses (:179-234) -----------------------------------------------------------------
    def get_initial_guess(self, guess_type: int = 0) -> np.ndarray:
        """0: literature values; 1: the same perturbed (13 draws from the global NumPy RNG); 2: ATM-implied."""
        literature = {
            'v1_0': 0.04, 'kappa1': 2.5, 'theta1': 0.04, 'sigma1': 0.3, 'rho1': -0.7,
            'v2_0': 0.04, 'kappa2': 0.5, 'theta2': 0.04, 'sigma2': 0.2, 'rho2': -0.5,
            'lambda_j': 0.15, 'mu_j': -0.04, 'sigma_j': 0.08
        }
        if guess_type == 0:
            params = literature
        elif guess_type == 1:
            params = {}
            for name, value in literature.items():
                width = 0.15 if name in ('rho1', 'rho2', 'mu_j') else 0.20
                params[name] = value * (1 + np.random.uniform(-width, width))
            params['rho1'] = np.clip(params['rho1'], -0.95, -0.3)
            params['rho2'] = np.clip(params['rho2'], -0.95, -0.3)
        else:
            atm = [opt for opt in self.market_options if 0.95 < opt['strike']/self.spot < 1.05]
            if atm:
                avg_price = np.mean([opt['price'] for opt in atm])
                avg_maturity = np.mean([opt['maturity'] for opt in atm])
                implied_var = (avg_price / self.spot) / np.sqrt(avg_maturity)
                implied_var = max(0.01, min(0.1, implied_var))
            else:
                implied_var = 0.04
            params = {
                'v1_0': implied_var, 'kappa1': 2.0, 'theta1': implied_var, 'sigma1': 0.4, 'rho1': -0.6,
                'v2_0': implied_var, 'kappa2': 0.7, 'theta2': implied_var, 'sigma2': 0.25, 'rho2': -0.4,
                'lambda_j': 0.12, 'mu_j': -0.03, 'sigma_j': 0.07
            }
        return self.inverse_transform_params(params)

    # -- optimiser driver (:236-336) ----------------------------------------------------------------
    @staticmethod
    def _minimize(fun_and_grad, x0, maxiter, maxfun=_MAXFUN_REQUESTS):
        return minimize(fun=fun_and_grad, x0=x0, jac=True, method='L-BFGS-B',
                        options={'maxiter': maxiter, 'ftol': 1e-9, 'gtol': 1e-6, 'maxfun': maxfun})

    def calibrate(self, maxiter: int = 300, multi_start: int = 3, *, x0=None, gradient: str = "fd",
                  objective: str = "price") -> CalibrationResult:
        """Calibrate to the market prices with `multi_start` L-BFGS-B runs; the best (lowest loss) wins.

        `x0` (keyword-only extension, not in the reference): optional unconstrained starting points
        [multi_start, 13] replacing the built-in guesses — the warm-start hook for an FFN predictor
        (docs/METHODOLOGY.md:112-134 of the reference describes that pipeline; its code is not in the repo).

        `gradient` (keyword-only extension): "fd" (default) is the reference's forward difference; "analytic" answers
        each scipy request with the exact gradient of the loss (one evaluation, `n_calls` + 1 per request, scipy's
        default maxfun = 15000 requests).

        `objective` (keyword-only extension): "price" (default) is the reference's loss; "iv" fits the Black–Scholes
        implied vols of the quotes instead: f = mean over the quotes that have an implied vol (status 0) of
        (sigma_model - sigma_market)^2 + the Feller penalty (DESIGN.md §6e).  It works with both gradients.  With
        objective="iv", `final_loss` (and `best_loss`) are values of that objective, not of compute_loss; the fields of
        the result are otherwise the same (model_prices are the model's prices at the optimum).
        """
        if gradient not in ("fd", "analytic"):
            raise ValueError(f"gradient must be 'fd' or 'analytic' (got {gradient!r})")
        if objective not in ("price", "iv"):
            raise ValueError(f"objective must be 'price' or 'iv' (got {objective!r})")
        start_time = time.time()
        market = self._device_market(objective)

        # initial points in start order: keeps the reference's global-RNG consumption (:252-256)
        if x0 is None:
            x0s = [self.get_initial_guess(guess_type=i % 3) for i in range(multi_start)]
        else:
            x0s = [np.array(v, dtype=np.float64) for v in np.asarray(x0, dtype=np.float64).reshape(multi_start, 13)]
        results = [None] * multi_start
        finished_at = [None] * multi_start
        counters = [[0, np.inf] for _ in range(multi_start)]          # per-start n_calls, best_loss

        def track(i, f_all):
            counters[i][0] += 14
            for v in f_all:
                if v != _SENTINEL and v < counters[i][1]:
                    counters[i][1] = v

        if gradient == "analytic":
            for i in range(multi_start):
                def fg(x, i=i):
                    f, g = market.loss_grad(np.asarray(x, dtype=np.float64).reshape(1, 13))
                    counters[i][0] += 1
                    if f[0] != _SENTINEL and f[0] < counters[i][1]:
                        counters[i][1] = f[0]
                    return f[0], g[0]
                try:
                    results[i] = self._minimize(fg, x0s[i], maxiter, maxfun=15000)
                except Exception as exc:
                    results[i] = exc
                finished_at[i] = time.time()
        elif self.batch_starts and multi_start > 1:
            evaluator = _LockstepEvaluator(market, multi_start)

            def worker(i):
                def fg(x):
                    f, g, f_all = evaluator.request(i, x)
                    track(i, f_all)
                    return f, g
                try:
                    results[i] = self._minimize(fg, x0s[i], maxiter)
                except Exception as exc:                                # reference: `except: continue` (:316-317)
                    results[i] = exc
                finally:
                    finished_at[i] = time.time()
                    evaluator.retire(i)

            threads = [threading.Thread(target=worker, args=(i,), daemon=True) for i in range(multi_start)]
            for t in threads:
                t.start()
            for t in threads:
                t.join()
        else:
            for i in range(multi_start):
                def fg(x, i=i):
                    f, g, f_all = market.loss_fd(np.asarray(x, dtype=np.float64).reshape(1, 13), _FD_STEP,
                                                 want_all=True)
                    track(i, f_all[0])
                    return f[0], g[0]
                try:
                    results[i] = self._minimize(fg, x0s[i], maxiter)
                except Exception as exc:
                    results[i] = exc
                finished_at[i] = time.time()

        from dhj import NativeError
        for res in results:
            if isinstance(res, NativeError):       # a device failure is not an "optimisation start failed"
                raise res
        if multi_start > 0:
            self.n_calls, self.best_loss = counters[-1]                # the reference resets per start (:253-254)

        best_idx, best_loss = None, np.inf
        for i, res in enumerate(results):
            if res is None or isinstance(res, Exception):
                continue
            if res.fun < best_loss:                                    # strict: first start wins ties (:271)
                best_loss, best_idx = res.fun, i

        if best_idx is None:                                           # :320-334
            return CalibrationResult(
                date='', spot=self.spot, risk_free=self.risk_free_rate,
                parameters={name: 0.0 for name in self.param_names},
                market_prices=self.market_prices, model_prices=np.zeros_like(self.market_prices),
                market_options=self.market_options, final_loss=np.inf,
                calibration_time=time.time() - start_time, success=False, iterations=0,
                message="All optimization starts failed")

        res = results[best_idx]
        model_prices = market.prices(res.x)[0]                         # re-pricing at the optimum (:276-299)
        return CalibrationResult(
            date='', spot=self.spot, risk_free=self.risk_free_rate,
            parameters=self.transform_params(res.x),
            market_prices=self.market_prices, model_prices=model_prices,
            market_options=self.market_options, final_loss=res.fun,
            calibration_time=finished_at[best_idx] - start_time,
            success=res.success, iterations=res.nit, message=res.message)


if __name__ == "__main__":
    print("Double Heston + jump L-BFGS-B calibrator (B200 build). See tests/ for usage.")
