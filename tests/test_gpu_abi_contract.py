"""The host side of the C ABI on the device: the lock-step loops' shape check, the argument checks shared by the
option-list entry points, the number of launches of each entry point, and the chunking of the synchronous staged
calls."""
import ctypes
import math

import numpy as np
import pytest

from oracle import cos_oracle as O

pytestmark = pytest.mark.gpu

DHJ_ERR_ARG = -1
K5, T5 = np.tile(O.GENERATOR_STRIKES_REL, 3), np.repeat(O.GENERATOR_MATURITIES, 5)   # 15 options, 3 maturities


@pytest.fixture(scope="module")
def ctx():
    import dhj
    c = dhj.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def raw():
    """The library without the binding's argument types, so that null pointers can be passed."""
    import dhj
    return ctypes.CDLL(dhj._native.LIB_PATH)


def _params(n, seed):
    rng = np.random.default_rng(seed)
    lo, hi = O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1]
    return lo + (hi - lo) * rng.random((n, 13))


@pytest.fixture(scope="module")
def market(ctx):
    """A 15-option, 3-maturity market of 2 % noisy model prices, and the unconstrained x of its parameters."""
    p = _params(1, 3)[0]
    rng = np.random.default_rng(4)
    price = ctx.price_list(p, 100.0, K5, T5, True, 0.03)[0] * (1 + 0.02 * rng.standard_normal(15))
    mk = ctx.market(100.0, 0.03, K5, T5, np.ones(15), price)
    yield mk, O.inverse_transform_params(p)
    mk.close()


# ---- the lock-step loops reject an optimiser of another shape before the first ask -------------------------------
def _x0(x, n, seed):
    return x + 0.05 * np.random.default_rng(seed).standard_normal((n, 13))


@pytest.mark.parametrize("method", ["minimize_fd", "minimize_grad"])
def test_minimize_rejects_dimension(ctx, market, method):
    import dhj
    mk, x = market
    opt = dhj.BatchLBFGS(np.zeros((4, 14)))
    with pytest.raises(dhj.NativeError, match="dimension is 14, not 13"):
        getattr(opt, method)(mk)
    opt.close()


@pytest.mark.parametrize("method", ["minimize_fd", "minimize_grad"])
def test_minimize_rejects_state_count_then_converges(ctx, raw, market, method):
    import dhj
    mk, x = market
    x0 = _x0(x, 4, 5)
    opt = dhj.BatchLBFGS(x0)
    name = "dhj_lbfgs_" + method
    fn = getattr(raw, name)
    h = [ctypes.c_double(1e-8)] if method == "minimize_fd" else []
    rc = fn(ctypes.c_void_p(opt._h.value), ctypes.c_void_p(ctx._h.value), ctypes.c_void_p(mk._h.value), None,
            ctypes.c_int64(opt.n - 1), *h, None, None, None)
    assert rc == DHJ_ERR_ARG
    msg = dhj.load_library().dhj_last_error(ctx._h).decode()
    assert "n_states (3) != the optimiser's state count (4)" in msg
    # nothing of the rejected call is left: the optimiser runs to its stop exactly as a fresh one does, and lowers the
    # loss of every state.  (Which stop it reports is the optimiser's business: on this 2 % noisy market the
    # forward-difference line search ends "ABNORMAL" at the noise floor.)
    rounds, _, _ = getattr(opt, method)(mk)
    fresh = dhj.BatchLBFGS(x0)
    getattr(fresh, method)(mk)
    got, want = opt.result(), fresh.result()
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    assert rounds > 0 and np.all(got[2] > 0)
    assert np.all(got[1] < mk.loss_batch(x0))
    opt.close()
    fresh.close()


# ---- the argument checks of the option-list entry points ------------------------------------------------------
_I64 = ("P", "s0_stride", "strike_stride")
_I32 = ("M", "N")
_F = ("r", "q", "L")
_SIGNATURES = {
    "dhj_price_list": ("in", "P", "S0", "s0_stride", "r", "q", "strike", "strike_stride", "maturity", "is_call", "M",
                       "N", "L", "out"),
    "dhj_price_jacobian": ("in", "P", "S0", "s0_stride", "r", "q", "strike", "strike_stride", "maturity", "is_call",
                           "M", "N", "L", "out", "out2"),
    "dhj_price_greeks": ("in", "P", "S0", "s0_stride", "r", "q", "strike", "strike_stride", "maturity", "is_call",
                         "M", "N", "L", "out", "out2"),
    "dhj_implied_vol": ("in", "P", "S0", "s0_stride", "r", "q", "strike", "strike_stride", "maturity", "is_call", "M",
                        "out", "out2"),
    "dhj_bs_price": ("in", "P", "S0", "s0_stride", "r", "q", "strike", "strike_stride", "maturity", "is_call", "M",
                     "out"),
}
# (case, overrides, message, entry points that take N and L only)
_CASES = [
    ("s0_stride", {"s0_stride": 2}, "s0_stride must be 0 or 1", False),
    ("strike_stride", {"strike_stride": 3}, "strike_stride must be 0 or M", False),
    ("null_strike", {"strike": None}, "null option table", False),
    ("null_maturity", {"maturity": None}, "null option table", False),
    ("null_is_call", {"is_call": None}, "null option table", False),
    ("N", {"N": 0}, "N must be >= 1 (got 0)", True),
    ("L_nan", {"L": math.nan}, "L is NaN", True),
    ("P", {"P": -1}, "P must be >= 0 (got -1)", False),
]


@pytest.mark.parametrize("case,overrides,message,needs_n", _CASES, ids=[c[0] for c in _CASES])
@pytest.mark.parametrize("name", list(_SIGNATURES))
def test_option_list_checks(ctx, raw, name, case, overrides, message, needs_n):
    import dhj
    sig = _SIGNATURES[name]
    if needs_n and "N" not in sig:
        pytest.skip(f"{name} has no {case} argument")
    P, M = 2, 15
    arrays = {"in": np.full((P, M), 0.2), "S0": np.full(P, 100.0), "strike": K5.copy(), "maturity": T5.copy(),
              "is_call": np.ones(M, dtype=np.int32), "out": np.empty((P, M, 13)), "out2": np.empty((P, M, 13))}
    scalars = {"P": P, "s0_stride": 1, "strike_stride": 0, "r": 0.03, "q": 0.0, "M": M, "N": 128, "L": 10.0}
    args = [ctypes.c_void_p(ctx._h.value)]
    for key in sig:
        v = overrides.get(key, arrays.get(key, scalars.get(key)))
        if key in _I64:
            args.append(ctypes.c_int64(v))
        elif key in _I32:
            args.append(ctypes.c_int32(v))
        elif key in _F:
            args.append(ctypes.c_double(v))
        else:
            args.append(None if v is None else ctypes.c_void_p(v.ctypes.data))
    assert getattr(raw, name)(*args) == DHJ_ERR_ARG
    assert dhj.load_library().dhj_last_error(ctx._h).decode() == message


# ---- launches per entry point ---------------------------------------------------------------------------------------
def _launches(ctx, call):
    n0 = ctx.launch_count
    call()
    return ctx.launch_count - n0


def test_launch_counts(ctx, market):
    mk, x = market
    p = _params(8, 6)
    V = ctx.price_list(p, 100.0, K5, T5, True, 0.03)
    xs = _x0(x, 4, 7)
    assert _launches(ctx, lambda: ctx.price_list(p, 100.0, K5, T5, True, 0.03)) == 1
    assert _launches(ctx, lambda: ctx.price_jacobian(p, 100.0, K5, T5, True, 0.03)) == 1
    assert _launches(ctx, lambda: ctx.price_greeks(p, 100.0, K5, T5, True, 0.03)) == 1
    assert _launches(ctx, lambda: ctx.implied_vol(V, 100.0, K5, T5, True, 0.03)) == 1
    assert _launches(ctx, lambda: ctx.bs_price(np.full_like(V, 0.2), 100.0, K5, T5, True, 0.03)) == 1
    assert _launches(ctx, lambda: ctx.cf(p[0], 0.03, 0.0, 0.5, np.linspace(0.1, 50, 64))) == 1
    assert _launches(ctx, lambda: ctx.cf(p[0], 0.03, 0.0, 0.5, np.linspace(0.1, 50, 64) - 0.5j)) == 1
    assert _launches(ctx, lambda: ctx.truncation_range(p, 100.0, K5, T5, 0.03)) == 1
    assert _launches(ctx, lambda: ctx.chi_psi(np.arange(64), -0.1, 0.2, -1.0, 1.0)) == 1
    assert _launches(ctx, lambda: mk.prices(xs)) == 1
    assert _launches(ctx, lambda: mk.loss_batch(xs)) == 1
    assert _launches(ctx, lambda: mk.loss_fd(xs)) == 1
    # 600 states x 14 stencil points >= 8 192 units: expand -> pricing kernel -> reduction
    assert _launches(ctx, lambda: mk.loss_fd(_x0(x, 600, 8))) == 3
    assert _launches(ctx, lambda: mk.loss_grad(xs)) == 1 + 3   # expand, then per chunk price, Jacobian, reduction
    assert _launches(ctx, lambda: mk.implied_vols(xs)) == 3


def test_launch_counts_iv_objective(ctx, market):
    mk, x = market
    iv = ctx.market(100.0, 0.03, K5, T5, np.ones(15), mk.prices(x)[0])
    try:
        assert _launches(ctx, lambda: iv.set_objective("iv")) == 1
        xs = _x0(x, 4, 9)
        assert _launches(ctx, lambda: iv.loss_grad(xs)) == 1 + 4   # + the IV residual per chunk
    finally:
        iv.close()


# ---- chunks of the synchronous staged calls ---------------------------------------------------------------------
def test_staged_chunks_bitwise(ctx):
    """price_jacobian over 3 000 sets of a 200-option list is cut into chunks of at most 32 MiB of staged rows (params
    in, prices and Jacobian out): its rows equal those of the same sets priced one chunk at a time, bit for bit, with
    one launch per chunk."""
    M, P = 200, 3000
    K = np.tile(np.linspace(80.0, 120.0, 20), 10)
    T = np.repeat(np.linspace(0.1, 2.0, 10), 20)
    call = np.arange(M) % 3 != 0
    p = _params(P, 10)
    per_row = 8 * (13 + M + 13 * M)
    chunk = (32 << 20) // per_row
    n_chunks = -(-P // chunk)
    assert n_chunks == 3
    n0 = ctx.launch_count
    prices, jac = ctx.price_jacobian(p, 100.0, K, T, call, 0.03, 0.01)
    assert ctx.launch_count - n0 == n_chunks
    for lo in range(0, P, chunk):
        pc, jc = ctx.price_jacobian(p[lo:lo + chunk], 100.0, K, T, call, 0.03, 0.01)
        assert np.array_equal(prices[lo:lo + chunk], pc, equal_nan=True)
        assert np.array_equal(jac[lo:lo + chunk], jc, equal_nan=True)
