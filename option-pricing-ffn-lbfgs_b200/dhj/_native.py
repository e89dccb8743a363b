"""ctypes binding of libdhj.so (include/dhj.h).  The only native entry into the product.

There is NO CPU fallback: if the shared library has not been built, or no sm_100 device is present,
the first use raises `NativeError` with the reason.  PyTorch is not needed here; the `*_dev` entry
points accept raw device pointers / stream handles (ints) so that a torch caller can pass
`tensor.data_ptr()` and `torch.cuda.current_stream().cuda_stream`.
"""
from __future__ import annotations

import ctypes
import os
import threading

import numpy as np
from numpy.ctypeslib import ndpointer

N_PARAMS = 13
N_GREEKS = 5
GREEKS = ("delta", "gamma", "theta", "rho", "rho_q")
# status codes of implied_vol (include/dhj.h)
IV_STATUS = ("ok", "below_lower_bound", "above_upper_bound", "invalid_input", "not_converged")
FD_POINTS = 14
LIB_PATH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "lib", "libdhj.so")

# every symbol include/dhj.h declares (tests/test_abi.py checks the header against this list)
EXPORTS = (
    "dhj_abi_version", "dhj_device_count", "dhj_init", "dhj_destroy", "dhj_last_error", "dhj_launch_count",
    "dhj_price_list", "dhj_price_grid", "dhj_price_grid_dev",
    "dhj_market_create", "dhj_market_destroy", "dhj_loss_batch", "dhj_loss_fd", "dhj_market_prices",
    "dhj_cf", "dhj_cf_complex", "dhj_truncation_range", "dhj_chi_psi", "dhj_fp64_peak",
    "dhj_lbfgs_create", "dhj_lbfgs_destroy", "dhj_lbfgs_ask", "dhj_lbfgs_tell", "dhj_lbfgs_result", "dhj_lbfgs_minimize_fd",
    "dhj_generator_draws", "dhj_generate_dev", "dhj_generate", "dhj_set_host_threads", "dhj_debug_checks",
    "dhj_price_jacobian", "dhj_loss_grad", "dhj_lbfgs_minimize_grad", "dhj_price_greeks",
    "dhj_implied_vol", "dhj_implied_vol_dev", "dhj_bs_price",
    "dhj_market_set_objective", "dhj_market_implied_vols", "dhj_mc_price",
)
# calibration objectives of a Market (dhj_market_set_objective)
OBJECTIVES = {"price": 0, "iv": 1}
# option kinds of mc_price, in the order of their codes (DHJ_MC_* in include/dhj.h)
MC_KINDS = ("european", "asian", "up-and-out", "up-and-in", "down-and-out", "down-and-in")


class NativeError(RuntimeError):
    """libdhj.so is missing, failed to load, or a call returned an error code."""


_F64 = ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_I32 = ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_c_i64, _c_i32, _c_f64, _c_vp = ctypes.c_int64, ctypes.c_int32, ctypes.c_double, ctypes.c_void_p

_lib = None
_lib_lock = threading.Lock()


def load_library(path: str | None = None) -> ctypes.CDLL:
    """dlopen libdhj.so and declare the argument types.  Does not touch the GPU."""
    global _lib
    with _lib_lock:
        if _lib is not None and path is None:
            return _lib
        p = path or os.environ.get("DHJ_LIBRARY", LIB_PATH)
        if not os.path.exists(p):
            raise NativeError(
                f"{p} not found: build it with `python __graft_entry__.py build` (or `make -C "
                f"option-pricing-ffn-lbfgs_b200/csrc`).  This package has no CPU fallback.")
        try:
            lib = ctypes.CDLL(p)
        except OSError as e:
            raise NativeError(f"cannot load {p}: {e}") from e
        missing = [s for s in EXPORTS if not hasattr(lib, s)]
        if missing:
            raise NativeError(f"{p} does not export {missing}")
        lib.dhj_abi_version.restype = ctypes.c_int
        lib.dhj_device_count.argtypes = [ctypes.POINTER(ctypes.c_int)]
        lib.dhj_init.argtypes = [ctypes.c_int, ctypes.POINTER(_c_vp)]
        lib.dhj_destroy.argtypes = [_c_vp]
        lib.dhj_last_error.argtypes = [_c_vp]
        lib.dhj_last_error.restype = ctypes.c_char_p
        lib.dhj_launch_count.argtypes = [_c_vp, ctypes.POINTER(_c_i64)]
        lib.dhj_price_list.argtypes = [_c_vp, _F64, _c_i64, _F64, _c_i64, _c_f64, _c_f64, _F64, _c_i64, _F64, _I32,
                                       _c_i32, _c_i32, _c_f64, _c_vp]
        lib.dhj_price_grid.argtypes = [_c_vp, _c_vp, _c_i64, _c_vp, _c_i64, _c_f64, _c_f64, _F64, _c_i32, _F64,
                                       _c_i32, _c_i32, _c_i32, _c_i32, _c_f64, _c_vp]
        lib.dhj_price_grid_dev.argtypes = [_c_vp, _c_vp, _c_i64, _c_vp, _c_i64, _c_f64, _c_f64, _F64, _c_i32, _F64,
                                           _c_i32, _c_i32, _c_i32, _c_i32, _c_f64, _c_vp, _c_vp]
        lib.dhj_market_create.argtypes = [_c_vp, _c_i32, _c_i32, _F64, _c_f64, _F64, _c_i64, _F64, _I32, _F64,
                                          _c_i32, ctypes.POINTER(_c_vp)]
        lib.dhj_market_destroy.argtypes = [_c_vp]
        lib.dhj_loss_batch.argtypes = [_c_vp, _c_vp, _F64, _c_vp, _c_i64, _F64]
        lib.dhj_loss_fd.argtypes = [_c_vp, _c_vp, _F64, _c_vp, _c_i64, _c_f64, _F64, _F64, _c_vp]
        lib.dhj_market_prices.argtypes = [_c_vp, _c_vp, _F64, _c_vp, _c_i64, _F64]
        lib.dhj_cf.argtypes = [_c_vp, _F64, _c_f64, _c_f64, _c_f64, _F64, _c_i32, _F64, _F64]
        lib.dhj_cf_complex.argtypes = [_c_vp, _F64, _c_f64, _c_f64, _c_f64, _F64, _F64, _c_i32, _F64, _F64]
        lib.dhj_truncation_range.argtypes = [_c_vp, _F64, _c_i64, _F64, _c_i64, _c_f64, _F64, _F64, _c_i32, _c_f64,
                                             _F64]
        lib.dhj_chi_psi.argtypes = [_c_vp, _I32, _c_i32, _c_f64, _c_f64, _c_f64, _c_f64, _F64, _F64]
        lib.dhj_fp64_peak.argtypes = [_c_vp, _c_i32, ctypes.POINTER(_c_f64), ctypes.POINTER(_c_f64)]
        _I64 = ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")
        lib.dhj_lbfgs_create.argtypes = [_c_i64, _c_i32, _c_i32, _c_i32, _c_i32, _c_i32, _c_f64, _c_f64, _F64,
                                         ctypes.POINTER(_c_vp)]
        lib.dhj_lbfgs_destroy.argtypes = [_c_vp]
        lib.dhj_lbfgs_ask.argtypes = [_c_vp, ctypes.POINTER(_c_i64), _I64, _F64]
        lib.dhj_lbfgs_tell.argtypes = [_c_vp, _c_i64, _F64, _F64]
        lib.dhj_lbfgs_result.argtypes = [_c_vp, _c_vp, _c_vp, _c_vp, _c_vp, _c_vp]
        lib.dhj_lbfgs_minimize_fd.argtypes = [_c_vp, _c_vp, _c_vp, _c_vp, _c_i64, _c_f64, ctypes.POINTER(_c_i64),
                                              ctypes.POINTER(_c_i64), _F64]
        lib.dhj_price_jacobian.argtypes = [_c_vp, _F64, _c_i64, _F64, _c_i64, _c_f64, _c_f64, _F64, _c_i64, _F64,
                                           _I32, _c_i32, _c_i32, _c_f64, _c_vp, _c_vp]
        lib.dhj_price_greeks.argtypes = lib.dhj_price_jacobian.argtypes
        lib.dhj_implied_vol.argtypes = [_c_vp, _F64, _c_i64, _F64, _c_i64, _c_f64, _c_f64, _F64, _c_i64, _F64, _I32,
                                        _c_i32, _c_vp, _c_vp]
        lib.dhj_implied_vol_dev.argtypes = [_c_vp, _c_vp, _c_i64, _c_vp, _c_i64, _c_f64, _c_f64, _F64, _c_i32, _F64,
                                            _I32, _c_i32, _c_vp, _c_vp, _c_vp]
        lib.dhj_bs_price.argtypes = [_c_vp, _F64, _c_i64, _F64, _c_i64, _c_f64, _c_f64, _F64, _c_i64, _F64, _I32,
                                     _c_i32, _c_vp]
        lib.dhj_loss_grad.argtypes = [_c_vp, _c_vp, _F64, _c_vp, _c_i64, _F64, _F64]
        lib.dhj_market_set_objective.argtypes = [_c_vp, _c_vp, _c_i32, _c_vp, _c_vp]
        lib.dhj_market_implied_vols.argtypes = [_c_vp, _c_vp, _F64, _c_vp, _c_i64, _F64, _c_vp]
        lib.dhj_lbfgs_minimize_grad.argtypes = [_c_vp, _c_vp, _c_vp, _c_vp, _c_i64, ctypes.POINTER(_c_i64),
                                                ctypes.POINTER(_c_i64), _F64]
        _U32 = ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")
        lib.dhj_generator_draws.argtypes = [_U32, _c_i32, _c_i32, _c_f64, _c_i64, _c_i32, _F64, _F64, _c_f64, _c_f64,
                                            _c_f64, _c_f64, _c_f64, _c_i32, _F64, _F64, _F64, _U32,
                                            ctypes.POINTER(_c_i32), ctypes.POINTER(_c_i32), ctypes.POINTER(_c_f64)]
        _c_u64 = ctypes.c_uint64
        gen_head = [_c_vp, _c_u64, _c_i64, _c_i64, _c_i32, _F64, _F64, _c_f64, _c_f64, _c_f64, _c_f64, _c_f64, _F64,
                    _c_i32, _F64, _c_i32, _c_f64, _c_i32, _c_f64]
        lib.dhj_generate_dev.argtypes = gen_head + [_c_vp] * 6
        lib.dhj_generate.argtypes = gen_head + [_c_vp] * 5
        lib.dhj_set_host_threads.argtypes = [_c_i32]
        lib.dhj_mc_price.argtypes = [_c_vp, _F64, _c_i64, _F64, _c_i64, _c_f64, _c_f64, _c_f64, _c_i32, _c_i32, _c_i32,
                                     _I32, _I32, _F64, _c_vp, _c_u64, _c_i64, _F64, _c_vp]
        lib.dhj_debug_checks.argtypes = [_c_vp, ctypes.POINTER(_c_i32), ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")]
        for name in EXPORTS:
            if name not in ("dhj_last_error",):
                getattr(lib, name).restype = ctypes.c_int
        if lib.dhj_abi_version() != 1:
            raise NativeError(f"{p}: ABI version {lib.dhj_abi_version()} != 1")
        if path is None:
            _lib = lib
        return lib


def _f64(a, shape=None):
    a = np.ascontiguousarray(a, dtype=np.float64)
    if shape is not None:
        a = a.reshape(shape)
    return a


def _ptr(a: np.ndarray) -> int:
    return a.ctypes.data


def _is_call(is_call, M):
    return np.ascontiguousarray(np.broadcast_to(np.asarray(is_call), (M,)).astype(bool).astype(np.int32))


def _strikes(strike, is_call, rows, M, what="P"):
    """(strike, strike_stride, is_call) of an option list: strike [M] (stride 0) or [rows, M] (stride M), is_call
    broadcast to int32[M]."""
    strike = _f64(strike)
    if strike.size == M:
        strike, k_stride = strike.reshape(M), 0
    elif strike.size == rows * M:
        strike, k_stride = strike.reshape(rows, M), M
    else:
        raise ValueError(f"strike must be [M] or [{what}, M]")
    return strike, k_stride, _is_call(is_call, M)


def _option_list(values, S0, strike, maturity, is_call, per_option=False):
    """(values, P, S0, s0_stride, strike, strike_stride, maturity, M, is_call) of an option list in dhj_price_list's
    layout: values are parameter sets [P, 13] or, per_option, one value per option ([M] or [P, M]); S0 a scalar or
    [P]; strike [M] or [P, M]."""
    maturity = _f64(maturity).reshape(-1)
    M = maturity.shape[0]
    values = _f64(values)
    if not per_option:
        values = values.reshape(-1, N_PARAMS)
    elif values.ndim == 2 and values.shape[1] == M:
        pass
    elif M and values.size % M == 0:
        values = values.reshape(-1, M)
    else:
        raise ValueError("values must be [M] or [P, M]")
    P = values.shape[0]
    S0 = _f64(S0).reshape(-1)
    if S0.size not in (1, P):
        raise ValueError("S0 must be a scalar or have one entry per row")
    strike, k_stride, call = _strikes(strike, is_call, P, M)
    return values, P, S0, 0 if S0.size == 1 else 1, strike, k_stride, maturity, M, call


class Context:
    """One libdhj context = one CUDA device.  Calls are serialised with a lock (the C side is not re-entrant)."""

    def __init__(self, device: int = 0, library: str | None = None):
        """`library`: path of another build of libdhj (the checked build of tests/test_gpu_checked.py); default the
        product library."""
        self._lib = load_library(library)
        self._h = _c_vp()
        self._lock = threading.RLock()
        rc = self._lib.dhj_init(int(device), ctypes.byref(self._h))
        if rc != 0:
            msg = self._lib.dhj_last_error(None).decode()
            self._h = None
            raise NativeError(f"dhj_init(device={device}) failed ({rc}): {msg}")
        self.device = int(device)

    # -- plumbing ---------------------------------------------------------------------------------
    def _check(self, rc: int, what: str):
        if rc != 0:
            raise NativeError(f"{what} failed ({rc}): {self._lib.dhj_last_error(self._h).decode()}")

    def close(self):
        if getattr(self, "_h", None):
            self._lib.dhj_destroy(self._h)
            self._h = None

    def __del__(self):  # pragma: no cover - interpreter shutdown order
        try:
            self.close()
        except Exception:
            pass

    def debug_checks(self):
        """(enabled, counts[8]) of the checked build's device-side self-checks (dhj_debug_checks)."""
        en, counts = _c_i32(), np.zeros(8, dtype=np.uint64)
        with self._lock:
            self._check(self._lib.dhj_debug_checks(self._h, ctypes.byref(en), counts), "dhj_debug_checks")
        return bool(en.value), counts

    @property
    def launch_count(self) -> int:
        n = _c_i64()
        self._check(self._lib.dhj_launch_count(self._h, ctypes.byref(n)), "dhj_launch_count")
        return n.value

    # -- pricing ----------------------------------------------------------------------------------
    def price_jacobian(self, params, S0, strike, maturity, is_call, r, q=0.0, N=128, L=10.0):
        """(prices float64[P, M], jac float64[P, M, 13]) of P parameter sets on an option list: jac[p, o, i] =
        d price / d param_i with the truncation range held at its value for the current parameters
        (dhj_price_jacobian)."""
        params, P, S0, s0_stride, strike, k_stride, maturity, M, call = _option_list(params, S0, strike, maturity,
                                                                                   is_call)
        prices, jac = np.empty((P, M)), np.empty((P, M, N_PARAMS))
        with self._lock:
            self._check(self._lib.dhj_price_jacobian(self._h, params, P, S0, s0_stride, float(r), float(q), strike,
                                                     k_stride, maturity, call, M, int(N), float(L), _ptr(prices),
                                                     _ptr(jac)), "dhj_price_jacobian")
        return prices, jac

    def price_greeks(self, params, S0, strike, maturity, is_call, r, q=0.0, N=128, L=10.0):
        """(prices float64[P, M], greeks float64[P, M, 5]) of P parameter sets on an option list: greeks[p, o] =
        (delta, gamma, theta, rho, rho_q) = (dV/dS0, d2V/dS0^2, -dV/dT, dV/dr, dV/dq), exact with the truncation
        range held at its value for the current inputs (dhj_price_greeks)."""
        params, P, S0, s0_stride, strike, k_stride, maturity, M, call = _option_list(params, S0, strike, maturity,
                                                                                   is_call)
        prices, greeks = np.empty((P, M)), np.empty((P, M, N_GREEKS))
        with self._lock:
            self._check(self._lib.dhj_price_greeks(self._h, params, P, S0, s0_stride, float(r), float(q), strike,
                                                   k_stride, maturity, call, M, int(N), float(L), _ptr(prices),
                                                   _ptr(greeks)), "dhj_price_greeks")
        return prices, greeks

    # -- implied volatility -----------------------------------------------------------------------
    def implied_vol(self, price, S0, strike, maturity, is_call, r, q=0.0, return_status=False):
        """Black–Scholes implied vols float64[P, M] of prices [P, M] (or [M]) on an option list in price_list's layout:
        S0 scalar or [P], strike [M] or [P, M] (dhj_implied_vol).  NaN outside the no-arbitrage bounds; with
        return_status also the int32[P, M] status codes (IV_STATUS names them)."""
        price, P, S0, s0_stride, strike, k_stride, maturity, M, call = _option_list(price, S0, strike, maturity,
                                                                                    is_call, per_option=True)
        vol, status = np.empty((P, M)), np.empty((P, M), dtype=np.int32)
        with self._lock:
            self._check(self._lib.dhj_implied_vol(self._h, price, P, S0, s0_stride, float(r), float(q), strike,
                                                  k_stride, maturity, call, M, _ptr(vol), _ptr(status)),
                        "dhj_implied_vol")
        return (vol, status) if return_status else vol

    def implied_vol_dev(self, d_price: int, P: int, d_S0: int, s0_stride: int, strike, maturity, is_call, r, q,
                        d_out_vol: int, d_out_status: int = 0, scale_by_spot=False, stream: int = 0):
        """Asynchronous device-pointer variant (dhj_implied_vol_dev): pointers and the stream are ints, the tables
        strike[M], maturity[M], is_call[M] host arrays; scale_by_spot: K = strike * S0 / 100."""
        strike, maturity = _f64(strike).reshape(-1), _f64(maturity).reshape(-1)
        M = maturity.size
        if strike.size != M:
            raise ValueError("strike must be [M]")
        call = _is_call(is_call, M)
        with self._lock:
            self._check(self._lib.dhj_implied_vol_dev(self._h, d_price, int(P), d_S0, int(s0_stride), float(r),
                                                      float(q), strike, int(bool(scale_by_spot)), maturity, call, M,
                                                      d_out_vol, d_out_status or None, stream or None),
                        "dhj_implied_vol_dev")

    def bs_price(self, vol, S0, strike, maturity, is_call, r, q=0.0):
        """Black–Scholes prices float64[P, M] of vols [P, M] (or [M]) in implied_vol's layout (dhj_bs_price)."""
        vol, P, S0, s0_stride, strike, k_stride, maturity, M, call = _option_list(vol, S0, strike, maturity, is_call,
                                                                                  per_option=True)
        out = np.empty((P, M))
        with self._lock:
            self._check(self._lib.dhj_bs_price(self._h, vol, P, S0, s0_stride, float(r), float(q), strike, k_stride,
                                               maturity, call, M, _ptr(out)), "dhj_bs_price")
        return out

    def price_list(self, params, S0, strike, maturity, is_call, r, q=0.0, N=128, L=10.0) -> np.ndarray:
        """Prices float64[P, M] of P parameter sets on an option list (dhj_price_list)."""
        params, P, S0, s0_stride, strike, k_stride, maturity, M, call = _option_list(params, S0, strike, maturity,
                                                                                   is_call)
        out = np.empty((P, M), dtype=np.float64)
        with self._lock:
            self._check(self._lib.dhj_price_list(self._h, params, P, S0, s0_stride, float(r), float(q), strike,
                                                 k_stride, maturity, call, M, int(N), float(L), _ptr(out)),
                        "dhj_price_list")
        return out

    def price_grid(self, params, S0, strikes, maturities, r, q=0.0, N=128, L=10.0, scale_by_spot=False,
                   is_call=True, out=None) -> np.ndarray:
        """Prices float64[P, nT, nK] on a strike x maturity grid, maturity-major (dhj_price_grid).

        `params`, `S0` and `out` may be pinned host arrays (e.g. views of pinned torch tensors): the
        library then copies to/from them directly instead of staging.
        """
        params = _f64(params).reshape(-1, N_PARAMS)
        P = params.shape[0]
        S0 = _f64(S0).reshape(-1)
        if S0.size not in (1, P):
            raise ValueError("S0 must be a scalar or have one entry per parameter set")
        strikes, maturities = _f64(strikes).reshape(-1), _f64(maturities).reshape(-1)
        nK, nT = strikes.size, maturities.size
        if out is None:
            out = np.empty((P, nT, nK), dtype=np.float64)
        elif out.dtype != np.float64 or out.size != P * nT * nK or not out.flags.c_contiguous:
            raise ValueError("out must be C-contiguous float64[P, nT, nK]")
        with self._lock:
            self._check(self._lib.dhj_price_grid(self._h, _ptr(params), P, _ptr(S0), 0 if S0.size == 1 else 1,
                                                 float(r), float(q), strikes, nK, maturities, nT,
                                                 int(bool(scale_by_spot)), int(bool(is_call)), int(N), float(L),
                                                 _ptr(out)), "dhj_price_grid")
        return out.reshape(P, nT, nK)

    def price_grid_dev(self, d_params: int, P: int, d_S0: int, s0_stride: int, strikes, maturities, r, q, N, L,
                       scale_by_spot, is_call, d_out: int, stream: int = 0):
        """Asynchronous device-pointer variant (dhj_price_grid_dev); pointers/stream are ints."""
        strikes, maturities = _f64(strikes).reshape(-1), _f64(maturities).reshape(-1)
        with self._lock:
            self._check(self._lib.dhj_price_grid_dev(self._h, d_params, int(P), d_S0, int(s0_stride), float(r),
                                                     float(q), strikes, strikes.size, maturities, maturities.size,
                                                     int(bool(scale_by_spot)), int(bool(is_call)), int(N), float(L),
                                                     d_out, stream or None), "dhj_price_grid_dev")

    # -- Monte Carlo pricing of path-dependent options -------------------------------------------
    def mc_price(self, params, S0, T, kind, is_call, strike, r, q=0.0, barrier=None, n_paths=1 << 20, n_steps=252,
                 n_obs=None, seed=0):
        """(price float64[P, M], stderr float64[P, M]): Monte Carlo prices of M options of one maturity T under P
        parameter sets (dhj_mc_price).  kind[M]: names from MC_KINDS or their codes; is_call[M], strike[M] and
        barrier[M] (needed for the barrier kinds; NaN or anything elsewhere) broadcast to M; S0 a scalar or [P].
        n_steps equal time steps, n_obs equally spaced observation dates (None: every step; must divide n_steps).
        The draws depend on (seed, path, step) only, so all sets share them and the result is reproducible."""
        params = _f64(params).reshape(-1, N_PARAMS)
        P = params.shape[0]
        S0 = _f64(S0).reshape(-1)
        if S0.size not in (1, P):
            raise ValueError("S0 must be a scalar or have one entry per parameter set")
        kinds = np.atleast_1d(np.asarray(kind, dtype=object))
        strike = np.atleast_1d(_f64(strike))
        M = max(kinds.size, strike.size, np.size(is_call), 1 if barrier is None else np.size(barrier))
        codes = np.empty(kinds.size, dtype=np.int32)
        for i, k in enumerate(kinds):
            if isinstance(k, str):
                if k not in MC_KINDS:
                    raise ValueError(f"unknown option kind {k!r}: expected one of {MC_KINDS}")
                codes[i] = MC_KINDS.index(k)
            else:
                codes[i] = int(k)
        codes = np.ascontiguousarray(np.broadcast_to(codes, (M,)))
        strike = np.ascontiguousarray(np.broadcast_to(strike, (M,)))
        call = _is_call(is_call, M)
        bar = None if barrier is None else np.ascontiguousarray(np.broadcast_to(_f64(barrier), (M,)))
        n_steps = int(n_steps)
        n_obs = n_steps if n_obs is None else int(n_obs)
        price, err = np.empty((P, M)), np.empty((P, M))
        with self._lock:
            self._check(self._lib.dhj_mc_price(self._h, params, P, S0, 0 if S0.size == 1 else 1, float(r), float(q),
                                               float(T), n_steps, n_obs, M, codes, call, strike,
                                               None if bar is None else _ptr(bar), int(seed) & 0xFFFFFFFFFFFFFFFF,
                                               int(n_paths), price, _ptr(err)), "dhj_mc_price")
        return price, err

    # -- synthetic dataset sweep (counter stream) ------------------------------------------------
    @staticmethod
    def _gen_args(seed, first, n, path_len, lo, hi, persistence, spot0, ret_mean, ret_sd, noise_sd, strikes_rel,
                  maturities, r, N, L):
        lo, hi = _f64(lo).reshape(N_PARAMS), _f64(hi).reshape(N_PARAMS)
        strikes_rel, maturities = _f64(strikes_rel).reshape(-1), _f64(maturities).reshape(-1)
        return (int(seed) & 0xFFFFFFFFFFFFFFFF, int(first), int(n), int(path_len), lo, hi, float(persistence),
                float(spot0), float(ret_mean), float(ret_sd), float(noise_sd), strikes_rel, strikes_rel.size,
                maturities, maturities.size, float(r), int(N), float(L))

    def generate_dev(self, seed, first, n, path_len, lo, hi, persistence, spot0, ret_mean, ret_sd, noise_sd,
                     strikes_rel, maturities, r, d_params: int, d_spots: int, d_model: int, d_market: int = 0,
                     d_loss: int = 0, stream: int = 0, N=128, L=10.0):
        """Samples [first, first+n) of the counter stream, drawn, priced and noised on the device into DEVICE
        buffers (ints: pointers / stream handle); asynchronous (dhj_generate_dev)."""
        args = self._gen_args(seed, first, n, path_len, lo, hi, persistence, spot0, ret_mean, ret_sd, noise_sd,
                              strikes_rel, maturities, r, N, L)
        with self._lock:
            self._check(self._lib.dhj_generate_dev(self._h, *args, d_params, d_spots, d_model, d_market or None,
                                                   d_loss or None, stream or None), "dhj_generate_dev")

    def generate(self, seed, first, n, path_len, lo, hi, persistence, spot0, ret_mean, ret_sd, noise_sd, strikes_rel,
                 maturities, r, N=128, L=10.0, out=None):
        """Same into HOST arrays (dhj_generate): dict of params[n,13], spots[n], model[n,M], market[n,M], loss[n].
        `out` may hold preallocated (e.g. pinned) arrays under those keys."""
        args = self._gen_args(seed, first, n, path_len, lo, hi, persistence, spot0, ret_mean, ret_sd, noise_sd,
                              strikes_rel, maturities, r, N, L)
        n, M = int(n), args[12] * args[14]
        shapes = {"params": (n, N_PARAMS), "spots": (n,), "model": (n, M), "market": (n, M), "loss": (n,)}
        res = {}
        for key, shp in shapes.items():
            a = None if out is None else out.get(key)
            if a is None:
                a = np.empty(shp, dtype=np.float64)
            elif a.dtype != np.float64 or a.size != int(np.prod(shp)) or not a.flags.c_contiguous:
                raise ValueError(f"out[{key!r}] must be C-contiguous float64{list(shp)}")
            res[key] = a
        with self._lock:
            self._check(self._lib.dhj_generate(self._h, *args, *[_ptr(res[k]) for k in shapes]), "dhj_generate")
        return {k: res[k].reshape(shapes[k]) for k in shapes}

    # -- the remaining DoubleHeston methods -------------------------------------------------------
    def cf(self, params, r, q, tau, u) -> np.ndarray:
        """characteristic_function at real (dhj_cf) or complex (dhj_cf_complex) frequencies `u`."""
        u = np.asarray(u)
        if np.iscomplexobj(u):
            flat = np.ascontiguousarray(u, dtype=np.complex128).reshape(-1)
            ur, ui = np.ascontiguousarray(flat.real), np.ascontiguousarray(flat.imag)
            re, im = np.empty_like(ur), np.empty_like(ur)
            with self._lock:
                self._check(self._lib.dhj_cf_complex(self._h, _f64(params, (N_PARAMS,)), float(r), float(q),
                                                     float(tau), ur, ui, ur.size, re, im), "dhj_cf_complex")
            return (re + 1j * im).reshape(u.shape)
        u = _f64(u)
        flat = u.reshape(-1)
        re, im = np.empty_like(flat), np.empty_like(flat)
        with self._lock:
            self._check(self._lib.dhj_cf(self._h, _f64(params, (N_PARAMS,)), float(r), float(q), float(tau), flat,
                                         flat.size, re, im), "dhj_cf")
        return (re + 1j * im).reshape(u.shape)

    def truncation_range(self, params, S0, strike, maturity, r, L=10.0) -> np.ndarray:
        params = _f64(params).reshape(-1, N_PARAMS)
        P = params.shape[0]
        S0 = _f64(S0).reshape(-1)
        strike, maturity = _f64(strike).reshape(-1), _f64(maturity).reshape(-1)
        out = np.empty((P, maturity.size, 2))
        with self._lock:
            self._check(self._lib.dhj_truncation_range(self._h, params, P, S0, 0 if S0.size == 1 else 1, float(r),
                                                       strike, maturity, maturity.size, float(L), out),
                        "dhj_truncation_range")
        return out

    def chi_psi(self, k, c, d, a, b):
        k = np.ascontiguousarray(np.asarray(k, dtype=np.int32).reshape(-1))
        chi, psi = np.empty(k.size), np.empty(k.size)
        with self._lock:
            self._check(self._lib.dhj_chi_psi(self._h, k, k.size, float(c), float(d), float(a), float(b), chi, psi),
                        "dhj_chi_psi")
        return chi, psi

    def fp64_peak(self, iters: int = 4096):
        t, ms = _c_f64(), _c_f64()
        with self._lock:
            self._check(self._lib.dhj_fp64_peak(self._h, int(iters), ctypes.byref(t), ctypes.byref(ms)),
                        "dhj_fp64_peak")
        return t.value, ms.value

    def market(self, S0, r, strike, maturity, is_call, price, N=128) -> "Market":
        return Market(self, S0, r, strike, maturity, is_call, price, N)


class Market:
    """Device-resident market(s): what DoubleHestonJumpCalibrator.__init__ stores (dhj_market_create)."""

    def __init__(self, ctx: Context, S0, r, strike, maturity, is_call, price, N=128):
        self.ctx = ctx
        maturity = _f64(maturity).reshape(-1)
        M = maturity.size
        S0 = _f64(S0).reshape(-1)
        n = S0.size
        price = _f64(price).reshape(n, M)
        strike, k_stride, call = _strikes(strike, is_call, n, M, "n_markets")
        self.n_markets, self.M, self.N = n, M, int(N)
        self.objective = "price"
        self._h = _c_vp()
        with ctx._lock:
            ctx._check(ctx._lib.dhj_market_create(ctx._h, n, M, S0, float(r), strike, k_stride, maturity, call, price,
                                                  int(N), ctypes.byref(self._h)), "dhj_market_create")

    def close(self):
        if getattr(self, "_h", None) and getattr(self.ctx, "_h", None):
            self.ctx._lib.dhj_market_destroy(self._h)
        self._h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _batch(x, market_index):
        """(x float64[B, 13], B, market index int32[B] or None, its pointer or None)"""
        x = _f64(x).reshape(-1, N_PARAMS)
        B = x.shape[0]
        if market_index is None:
            return x, B, None, None
        idx = np.ascontiguousarray(np.asarray(market_index, dtype=np.int32).reshape(B))
        return x, B, idx, idx.ctypes.data

    def loss_batch(self, x, market_index=None) -> np.ndarray:
        x, B, idx, pidx = self._batch(x, market_index)
        out = np.empty(B)
        c = self.ctx
        with c._lock:
            c._check(c._lib.dhj_loss_batch(c._h, self._h, x, pidx, B, out), "dhj_loss_batch")
        return out

    def loss_fd(self, x, h=1e-8, market_index=None, want_all=False):
        """(f[C], g[C,13][, f_all[C,14]]) in one launch (dhj_loss_fd)."""
        x, C, idx, pidx = self._batch(x, market_index)
        f, g = np.empty(C), np.empty((C, N_PARAMS))
        f_all = np.empty((C, FD_POINTS)) if want_all else None
        c = self.ctx
        with c._lock:
            c._check(c._lib.dhj_loss_fd(c._h, self._h, x, pidx, C, float(h), f, g,
                                        f_all.ctypes.data if want_all else None), "dhj_loss_fd")
        return (f, g, f_all) if want_all else (f, g)

    def loss_grad(self, x, market_index=None):
        """(f[C], g[C,13]): the loss and its exact gradient in the unconstrained x (dhj_loss_grad; truncation range
        held fixed, g = 0 where f is the 1e10 sentinel)."""
        x, C, idx, pidx = self._batch(x, market_index)
        f, g = np.empty(C), np.empty((C, N_PARAMS))
        c = self.ctx
        with c._lock:
            c._check(c._lib.dhj_loss_grad(c._h, self._h, x, pidx, C, f, g), "dhj_loss_grad")
        return f, g

    def set_objective(self, objective: str):
        """Select what loss_batch, loss_fd, loss_grad and the BatchLBFGS loops compute on this market: "price" (the
        default: relative price error + Feller) or "iv" (mean squared implied-vol error over the quotes that have an
        implied vol + Feller; dhj_market_set_objective).  Returns (market_vols[n_markets, M], status[n_markets, M]):
        the quotes' Black–Scholes implied vols (q = 0; NaN where status != 0: left out of the objective) and their
        IV_STATUS codes ((None, None) for "price").  A market without any valid quote raises NativeError and the
        market keeps its objective."""
        if objective not in OBJECTIVES:
            raise ValueError(f"objective must be 'price' or 'iv' (got {objective!r})")
        vol = np.empty((self.n_markets, self.M)) if objective == "iv" else None
        status = np.empty((self.n_markets, self.M), dtype=np.int32) if objective == "iv" else None
        c = self.ctx
        with c._lock:
            c._check(c._lib.dhj_market_set_objective(c._h, self._h, OBJECTIVES[objective],
                                                     _ptr(vol) if vol is not None else None,
                                                     _ptr(status) if status is not None else None),
                     "dhj_market_set_objective")
        self.objective = objective
        return vol, status

    def implied_vols(self, x, market_index=None):
        """(vol[B, M], status[B, M]): Black–Scholes implied vols (q = 0) of the model prices at the unconstrained x
        and their IV_STATUS codes, every option (dhj_market_implied_vols)."""
        x, B, idx, pidx = self._batch(x, market_index)
        vol, status = np.empty((B, self.M)), np.empty((B, self.M), dtype=np.int32)
        c = self.ctx
        with c._lock:
            c._check(c._lib.dhj_market_implied_vols(c._h, self._h, x, pidx, B, vol, _ptr(status)),
                     "dhj_market_implied_vols")
        return vol, status

    def prices(self, x, market_index=None) -> np.ndarray:
        x, B, idx, pidx = self._batch(x, market_index)
        out = np.empty((B, self.M))
        c = self.ctx
        with c._lock:
            c._check(c._lib.dhj_market_prices(c._h, self._h, x, pidx, B, out), "dhj_market_prices")
        return out


class BatchLBFGS:
    """Lock-step batch of unconstrained L-BFGS-B instances (dhj_lbfgs_*): host-only, no device needed.

        opt = BatchLBFGS(x0)                      # x0[n, dim]
        while True:
            idx, x = opt.ask()
            if idx.size == 0: break
            f, g = evaluate(x, idx)               # e.g. Market.loss_fd(x, market_index=...)
            opt.tell(f, g)
        x, f, nit, nfev, status = opt.result()

    `maxfun` counts (f, g) requests.  The reference lets scipy difference the loss itself (jac=None), where each
    request costs 14 loss evaluations against scipy's default maxfun = 15000: the equivalent request limit is
    15000 // 14 = 1071, the default here (and what the drop-in `calibrate` passes to scipy).
    """

    MESSAGES = ("CONVERGENCE: NORM OF PROJECTED GRADIENT <= PGTOL",
                "CONVERGENCE: RELATIVE REDUCTION OF F <= FACTR*EPSMCH",
                "STOP: TOTAL NO. OF ITERATIONS REACHED LIMIT",
                "STOP: TOTAL NO. OF F,G EVALUATIONS EXCEEDS LIMIT",
                "ABNORMAL: ")

    def __init__(self, x0, maxiter=300, ftol=1e-9, gtol=1e-6, m=10, maxfun=15000 // 14, maxls=20):
        self._lib = load_library()
        x0 = _f64(x0)
        if x0.ndim != 2:
            raise ValueError("x0 must be [n_states, dim]")
        self.n, self.dim = x0.shape
        self._h = _c_vp()
        rc = self._lib.dhj_lbfgs_create(self.n, self.dim, int(m), int(maxiter), int(maxfun), int(maxls), float(ftol),
                                        float(gtol), x0, ctypes.byref(self._h))
        if rc != 0:
            raise NativeError(f"dhj_lbfgs_create failed ({rc})")
        self._idx = np.empty(self.n, dtype=np.int64)
        self._x = np.empty((self.n, self.dim))
        self._n_active = 0

    def ask(self):
        n = _c_i64()
        rc = self._lib.dhj_lbfgs_ask(self._h, ctypes.byref(n), self._idx, self._x)
        if rc != 0:
            raise NativeError(f"dhj_lbfgs_ask failed ({rc})")
        self._n_active = n.value
        return self._idx[:n.value].copy(), self._x[:n.value].copy()

    def tell(self, f, g):
        f, g = _f64(f).reshape(-1), _f64(g).reshape(-1, self.dim)
        if f.size != self._n_active or g.shape[0] != self._n_active:
            raise ValueError("tell() needs one f and one g per point of the last ask()")
        rc = self._lib.dhj_lbfgs_tell(self._h, self._n_active, f, g)
        if rc != 0:
            raise NativeError(f"dhj_lbfgs_tell failed ({rc})")

    def minimize_fd(self, market: "Market", state_market=None, h=1e-8):
        """Run the whole lock-step loop natively (dhj_lbfgs_minimize_fd): every round one `dhj_loss_fd` launch on
        `market` over all states that wait for an evaluation (state i uses market `state_market[i]`), until every
        optimiser has stopped.  Returns (rounds, state_rounds, (seconds in ask, loss, tell)).  The GIL is released for
        the whole call."""
        return self._minimize("dhj_lbfgs_minimize_fd", market, state_market, float(h))

    def minimize_grad(self, market: "Market", state_market=None):
        """minimize_fd with the analytic gradient (dhj_lbfgs_minimize_grad): every round one `dhj_loss_grad` call,
        one loss evaluation per request.  Returns (rounds, state_rounds, (seconds in ask, loss, tell))."""
        return self._minimize("dhj_lbfgs_minimize_grad", market, state_market)

    def _minimize(self, name, market, state_market, *args):
        sm = None if state_market is None else np.ascontiguousarray(np.asarray(state_market, dtype=np.int32).reshape(self.n))
        rounds, state_rounds, secs = _c_i64(), _c_i64(), np.zeros(3)
        c = market.ctx
        with c._lock:
            c._check(getattr(self._lib, name)(self._h, c._h, market._h, None if sm is None else sm.ctypes.data, self.n,
                                              *args, ctypes.byref(rounds), ctypes.byref(state_rounds), secs), name)
        return rounds.value, state_rounds.value, tuple(secs)

    def result(self):
        x, f = np.empty((self.n, self.dim)), np.empty(self.n)
        nit, nfev, status = (np.empty(self.n, dtype=np.int32) for _ in range(3))
        rc = self._lib.dhj_lbfgs_result(self._h, x.ctypes.data, f.ctypes.data, nit.ctypes.data, nfev.ctypes.data,
                                        status.ctypes.data)
        if rc != 0:
            raise NativeError(f"dhj_lbfgs_result failed ({rc})")
        return x, f, nit, nfev, status

    def close(self):
        if getattr(self, "_h", None):
            self._lib.dhj_lbfgs_destroy(self._h)
            self._h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass


_default_ctx: Context | None = None
_default_lock = threading.Lock()


def generator_draws(n, lo, hi, persistence, spot0, ret_mean, ret_sd, noise_sd, n_noise):
    """The synthetic generator's draw stream (dhj_generator_draws) on NumPy's GLOBAL legacy RandomState: reads
    `np.random.get_state()`, produces params[n, len(lo)], spots[n], noise[n, n_noise] exactly as the reference's
    per-sample `np.random.uniform` / `np.random.normal` calls would (synthetic_generator.py:98-142), and writes
    the advanced state back with `np.random.set_state()`.  Host only: needs the library, not a GPU."""
    lib = load_library()
    kind, key, pos, has_gauss, cached = np.random.get_state()
    if kind != "MT19937":
        raise NativeError(f"np.random global state is {kind}, expected the legacy MT19937")
    lo, hi = _f64(lo), _f64(hi)
    n = int(n)
    params, spots, noise = np.empty((n, lo.size)), np.empty(n), np.empty((n, int(n_noise)))
    key_in = np.ascontiguousarray(key, dtype=np.uint32)
    key_out = np.empty(624, dtype=np.uint32)
    pos_out, hg_out, cached_out = _c_i32(), _c_i32(), _c_f64()
    rc = lib.dhj_generator_draws(key_in, int(pos), int(has_gauss), float(cached), n, lo.size, lo, hi,
                                 float(persistence), float(spot0), float(ret_mean), float(ret_sd), float(noise_sd),
                                 int(n_noise), params, spots, noise, key_out, ctypes.byref(pos_out),
                                 ctypes.byref(hg_out), ctypes.byref(cached_out))
    if rc != 0:
        raise NativeError(f"dhj_generator_draws failed ({rc})")
    np.random.set_state(("MT19937", key_out, pos_out.value, hg_out.value, cached_out.value))
    return params, spots, noise


def set_host_threads(n: int) -> None:
    """Threads of the library's host-side parallel loops (dhj_set_host_threads); 0 = all cores."""
    if load_library().dhj_set_host_threads(int(n)) != 0:
        raise NativeError("dhj_set_host_threads failed")


def default_context() -> Context:
    """Process-wide context on the device named by DHJ_DEVICE / LOCAL_RANK (default 0), created once."""
    global _default_ctx
    with _default_lock:
        if _default_ctx is None:
            dev = int(os.environ.get("DHJ_DEVICE", os.environ.get("LOCAL_RANK", "0")))
            _default_ctx = Context(dev)
        return _default_ctx
