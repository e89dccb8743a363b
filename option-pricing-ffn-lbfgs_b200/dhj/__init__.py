"""dhj — host-side Python over libdhj.so: B200 COS pricing of the Double-Heston + Merton-jump model.

    from dhj import default_context
    ctx = default_context()
    prices = ctx.price_grid(params, S0, strikes, maturities, r)      # float64[P, nT, nK]

The drop-in replacements for the reference's modules live beside this package under `src/`
(src/models/double_heston.py, src/calibration/lbfgs_calibrator.py, src/data/synthetic_generator.py).
"""
from ._native import (BatchLBFGS, Context, Market, NativeError, default_context, generator_draws, load_library, set_host_threads, EXPORTS,
                      LIB_PATH, N_PARAMS, N_GREEKS, GREEKS, IV_STATUS, FD_POINTS, MC_KINDS)

__all__ = ["BatchLBFGS", "Context", "Market", "NativeError", "default_context", "generator_draws", "load_library", "set_host_threads",
           "EXPORTS", "LIB_PATH", "N_PARAMS", "N_GREEKS", "GREEKS", "IV_STATUS", "FD_POINTS", "MC_KINDS"]
from .calibrate_many import calibrate_many, calibrate_many_sharded, initial_guesses  # noqa: E402

__all__ += ["calibrate_many", "calibrate_many_sharded", "initial_guesses"]
