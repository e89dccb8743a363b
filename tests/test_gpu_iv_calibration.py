"""The implied-volatility calibration objective on the device (DESIGN.md §6e): f and the exact gradient against the
CPU oracle (tests/iv_loss_oracle.py), the three entry points against each other, the FD gradient against the device's
own loss, the sentinel and exclusion rules, independence of the batch, the checked build, and calibrations."""
import os

import numpy as np
import pytest

import iv_loss_oracle as IL
from conftest import PKG
from oracle import cos_oracle as O
from test_iv_loss_cpu import iv_markets

pytestmark = pytest.mark.gpu

CHECKED = os.path.join(PKG, "lib", "libdhj_checked.so")
F_TOL = 1e-11            # |f - oracle| / f; measured worst 9.8e-13 on one NVIDIA B200 (ragged4)
G_TOL = 3e-11            # |g - oracle| / |g|inf; measured worst 2.7e-12 on one NVIDIA B200 (ragged4)
# IV RMSE of the noise-free fits (analytic gradient): measured 0.88e-4 to 2.44e-4 over the four markets on one NVIDIA
# B200, not the 1e-5 an exact fit would give: L-BFGS-B stops on ftol = 1e-9 of max(|f|, 1), and the IV objective is
# ~1e-8 there.  The price-objective fits from the same starts measured 0.33e-4 to 1.28e-4 (median ratio 1.61).
RMSE_PIN = 5e-4
P_LIT = np.array([0.04, 2.5, 0.04, 0.3, -0.7, 0.04, 0.5, 0.04, 0.2, -0.5, 0.15, -0.04, 0.08])


@pytest.fixture(scope="module")
def ctx():
    import dhj
    c = dhj.Context(0)
    yield c
    c.close()


def _ragged4():
    """4 maturities with 9 to 12 strikes each (the dense pricing path), calls and puts, 1 % noise."""
    Ks = [np.linspace(80.0, 120.0, n) for n in (9, 10, 11, 12)]
    K = np.concatenate(Ks)
    T = np.concatenate([np.full(len(k), t) for k, t in zip(Ks, (0.1, 0.4, 1.0, 2.0))])
    call = np.arange(len(K)) % 3 != 0
    mk = O.price_batch(P_LIT, 100.0, K, T, call, 0.02)[0] * (1 + 0.01 * np.random.default_rng(8).standard_normal(len(K)))
    x = O.inverse_transform_params(P_LIT)[None, :] + 0.1 * np.random.default_rng(9).standard_normal((3, 13))
    return ("ragged4", 100.0, 0.02, K, T, call, mk, x)


def _markets():
    return iv_markets() + [_ragged4()]


def _sentinel_states():
    """A NaN parameter; a tiny-variance state whose COS prices go below 0 (v = 1e-6) and one whose prices stay
    positive but fall below the intrinsic value (v = 1e-8) on the C1 market's options."""
    out = []
    for v in (1e-6, 1e-8):
        out.append(O.inverse_transform_params(np.array([v, 2.5, v, 1e-3, -0.7, v, 0.5, v, 1e-3, -0.5, 1e-6, -0.04,
                                                        0.01])))
    nan = O.inverse_transform_params(P_LIT)
    nan[2] = np.nan
    return np.vstack(out + [nan])


@pytest.mark.parametrize("m", range(4))
def test_iv_loss_and_grad_vs_oracle(ctx, m):
    tag, S0, r, K, T, call, mk, x = _markets()[m]
    market = ctx.market(S0, r, K, T, call, mk)
    mvol, st = market.set_objective("iv")
    want_mvol, want_st = IL.market_vols(S0, r, K, T, call, mk)
    assert np.array_equal(st[0], want_st) and (st == 0).any()         # ragged4: noise excludes a few quotes
    ok = want_st == 0
    assert np.isnan(mvol[0, ~ok]).all() and np.abs(mvol[0, ok] - want_mvol[ok]).max() <= 1e-12 * want_mvol[ok].max()
    fb = market.loss_batch(x)
    ffd, _ = market.loss_fd(x)
    fg, g = market.loss_grad(x)
    assert np.array_equal(fb, ffd) and np.array_equal(fb, fg)          # one f, whatever the entry point
    want_f, want_g = IL.iv_loss_grad_batch(x, S0, r, K, T, call, mk, mvol=want_mvol)
    ferr = np.abs(fb / want_f - 1).max()
    gerr = (np.abs(g - want_g).max(axis=1) / np.abs(want_g).max(axis=1)).max()
    print(f"{tag}: |f - oracle| / f {ferr:.2e}, |g - oracle| / |g|inf {gerr:.2e}")
    assert ferr <= F_TOL and gerr <= G_TOL


@pytest.mark.parametrize("m", [0, 3])
def test_iv_fd_gradient_is_scipys_difference(ctx, m):
    """loss_fd's g is scipy's forward difference of the device f: the 14 stencil losses from loss_batch give the same
    bits, and f_all holds them."""
    tag, S0, r, K, T, call, mk, x = _markets()[m]
    market = ctx.market(S0, r, K, T, call, mk)
    market.set_objective("iv")
    h = 1e-8
    f, g, f_all = market.loss_fd(x, h, want_all=True)
    for c in range(len(x)):
        pts = np.repeat(x[c][None, :], 14, axis=0)
        for i in range(13):
            pts[1 + i, i] = x[c, i] + h
        fv = market.loss_batch(pts)
        assert np.array_equal(fv, f_all[c])
        assert np.array_equal((fv[1:] - fv[0]) / ((x[c] + h) - x[c]), g[c])


def test_iv_sentinel(ctx):
    tag, S0, r, K, T, call, mk, x = _markets()[2]
    market = ctx.market(S0, r, K, T, call, mk)
    market.set_objective("iv")
    xs = _sentinel_states()
    prices = market.prices(xs[:2])
    low = np.maximum(S0 - K * np.exp(-r * T), 0.0)
    assert (prices[0] <= 0).any() and (prices[1] > 0).all() and (prices[1] < low).any()
    fb = market.loss_batch(xs)
    ffd, gfd = market.loss_fd(xs)
    fg, g = market.loss_grad(xs)
    for f in (fb, ffd, fg):
        assert (f == O.SENTINEL).all(), f
    assert (g == 0).all()
    want_f, want_g = IL.iv_loss_grad_batch(xs, S0, r, K, T, call, mk)
    assert (want_f == O.SENTINEL).all() and (want_g == 0).all()


def test_iv_exclusion(ctx):
    """A quote noised below its intrinsic value is left out (status 1) and f is that of the market without it; a
    market without any valid quote cannot be set to the IV objective and stays on the price objective."""
    import dhj
    tag, S0, r, K, T, call, mk, x = _markets()[2]
    mk = mk.copy()
    mk[0] = 0.98 * max(S0 - K[0] * np.exp(-r * T[0]), 0.0)
    market = ctx.market(S0, r, K, T, call, mk)
    mvol, st = market.set_objective("iv")
    assert st[0, 0] == 1 and np.isnan(mvol[0, 0]) and (st[0, 1:] == 0).all()
    keep = np.arange(len(K)) != 0
    without = ctx.market(S0, r, K[keep], T[keep], call[keep], mk[keep])
    without.set_objective("iv")
    f1, g1 = market.loss_grad(x)
    f2, g2 = without.loss_grad(x)
    assert np.array_equal(market.loss_batch(x), without.loss_batch(x)) and np.array_equal(f1, f2)
    assert np.allclose(g1, g2, rtol=1e-13, atol=1e-15)
    # no valid quote: every price below its intrinsic value (or at or above the spot)
    bad = np.where(K < S0, 0.5 * (S0 - K * np.exp(-r * T)), S0)
    none = ctx.market(S0, r, K, T, call, bad)
    ref = ctx.market(S0, r, K, T, call, bad)
    with pytest.raises(dhj.NativeError, match="no option with an implied vol"):
        none.set_objective("iv")
    assert none.objective == "price"
    assert np.array_equal(none.loss_batch(x), ref.loss_batch(x))
    assert np.array_equal(none.loss_grad(x)[1], ref.loss_grad(x)[1])


def test_iv_independence_and_determinism(ctx):
    """A state's (f, g) is bit-identical alone, among 64 states and among 30 000 states, on repeated calls, on the
    analytic and the FD path."""
    tag, S0, r, K, T, call, mk, x = _markets()[0]
    market = ctx.market(S0, r, K, T, call, mk)
    market.set_objective("iv")
    rng = np.random.default_rng(9)
    big = x[rng.integers(0, len(x), 30000)] + 1e-2 * rng.standard_normal((30000, 13))
    probe = big[12345].copy()
    mid = np.vstack([big[:40], probe[None, :], big[40:63]])
    f1, g1 = market.loss_grad(probe[None, :])
    f64, g64 = market.loss_grad(mid)
    fb, gb = market.loss_grad(big)
    assert f1[0] == f64[40] == fb[12345]
    assert np.array_equal(g1[0], g64[40]) and np.array_equal(g1[0], gb[12345])
    f2, g2 = market.loss_grad(big)
    assert np.array_equal(fb, f2) and np.array_equal(gb, g2)
    d1, e1 = market.loss_fd(probe[None, :])
    d64, e64 = market.loss_fd(mid)
    db, eb = market.loss_fd(big)
    assert d1[0] == d64[40] == db[12345] == f1[0]
    assert np.array_equal(e1[0], e64[40]) and np.array_equal(e1[0], eb[12345])
    assert np.array_equal(market.loss_batch(big), fb)
    assert np.array_equal(market.loss_fd(big)[1], eb)


def test_checked_build_iv():
    import dhj
    tag, S0, r, K, T, call, mk, x = _markets()[3]
    xs = np.vstack([x, _sentinel_states()[:2]])
    outs = []
    for lib in (None, CHECKED):
        c = dhj.Context(0, library=lib)
        m = c.market(S0, r, K, T, call, mk)
        mv = m.set_objective("iv")[0]
        outs.append((mv, m.loss_batch(xs), m.loss_fd(xs), m.loss_grad(xs), m.implied_vols(xs)))
        if lib:
            enabled, counts = c.debug_checks()
            assert enabled and not counts.any(), counts
        m.close()
        c.close()
    a, b = outs
    assert np.array_equal(a[0], b[0], equal_nan=True) and np.array_equal(a[1], b[1])
    for u, v in zip(a[2] + a[3] + a[4], b[2] + b[3] + b[4]):
        assert np.array_equal(u, v, equal_nan=True)


def test_implied_vols_report(ctx):
    tag, S0, r, K, T, call, mk, x = _markets()[1]
    market = ctx.market(S0, r, K, T, call, mk)
    vol, st = market.implied_vols(x)
    want = ctx.implied_vol(market.prices(x), S0, K, T, call, r, 0.0, return_status=True)
    assert np.array_equal(vol, want[0], equal_nan=True) and np.array_equal(st, want[1])


# ---- calibrations --------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def cal():
    import sys
    p = os.path.join(PKG, "src", "calibration")
    if p not in sys.path:
        sys.path.insert(0, p)
    import lbfgs_calibrator
    return lbfgs_calibrator


def _noise_free_market(seed):
    rng = np.random.default_rng(seed)
    p = P_LIT * (1 + 0.2 * rng.uniform(-1, 1, 13))
    p[3], p[4], p[8], p[9] = 0.3, -0.6, 0.1, -0.4       # both Feller conditions hold: the true x has f = 0
    K, T = np.tile(O.GENERATOR_STRIKES_REL, 3), np.repeat(O.GENERATOR_MATURITIES, 5)
    return p, K, T


def test_calibrate_iv_noise_free(ctx, cal):
    """Noise-free markets (model prices at known parameters) calibrated on the IV objective from the three built-in
    starts reach the pinned IV RMSE (analytic gradient); the FD gradient runs and ends in the same basin.  Prints the
    median IV RMSE ratio against the price-objective fit from the same starts."""
    ratios, rmse_an, rmse_fd = [], [], []
    for seed in range(4):
        p, K, T = _noise_free_market(seed)
        prices = ctx.price_list(p, 100.0, K, T, np.ones(15, bool), 0.03)[0]
        opts = [{"strike": float(K[j]), "maturity": float(T[j]), "price": float(prices[j]), "option_type": "call"}
                for j in range(15)]
        c = cal.DoubleHestonJumpCalibrator(100.0, 0.03, opts)
        mvol = c._device_market("iv").set_objective("iv")[0][0]
        out = {}
        for obj, grad in (("iv", "analytic"), ("iv", "fd"), ("price", "analytic")):
            np.random.seed(seed)
            res = c.calibrate(maxiter=300, multi_start=3, gradient=grad, objective=obj)
            vol = c._device_market("iv").implied_vols(c.inverse_transform_params(res.parameters))[0][0]
            out[(obj, grad)] = (res, np.sqrt(np.mean((vol - mvol) ** 2)))
        rmse = out[("iv", "analytic")][1]
        rmse_an.append(rmse)
        rmse_fd.append(out[("iv", "fd")][1])
        ratios.append(rmse / out[("price", "analytic")][1])
        f_an, f_fd = out[("iv", "analytic")][0].final_loss, out[("iv", "fd")][0].final_loss
        print(f"seed {seed}: IV RMSE iv/analytic {rmse:.2e}, iv/fd {out[('iv', 'fd')][1]:.2e}, "
              f"price/analytic {out[('price', 'analytic')][1]:.2e}; final IV loss analytic {f_an:.3e} fd {f_fd:.3e}")
    print(f"median IV RMSE ratio (IV objective / price objective): {np.median(ratios):.3f}")
    assert max(rmse_an) <= RMSE_PIN
    assert max(rmse_fd) <= 1e-3                                         # same basin: a fit, not a different surface


def _c5(n, seed=7):
    import dhj
    ctx = dhj.default_context()
    lo, hi = O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1]
    data = ctx.generate(seed, 0, n, 500, lo, hi, 0.9, 100.0, 0.0003, 0.01, 0.02, O.GENERATOR_STRIKES_REL,
                        O.GENERATOR_MATURITIES, 0.03)
    spots, market = data["spots"], data["market"]
    K = np.tile(O.GENERATOR_STRIKES_REL[None, :] * spots[:, None] / 100.0, (1, 3))
    T = np.repeat(O.GENERATOR_MATURITIES, 5)
    return spots, K, T, market


def test_calibrate_many_iv_c5(monkeypatch):
    """calibrate_many(objective="iv") on 200 C5 markets: pipelines=1 and pipelines=4 give the same bits, both
    gradients converge, and the count of excluded quotes (noise below the intrinsic value) is reported."""
    import dhj
    spots, K, T, market = _c5(10000)
    sub = np.arange(200)
    x0 = dhj.initial_guesses(spots, K, T, market, 3)
    kw = dict(maxiter=300, multi_start=3, objective="iv")
    one = dhj.calibrate_many(spots[sub], 0.03, K[sub], T, np.ones(15), market[sub], x0=x0[sub], pipelines=1,
                             gradient="analytic", **kw)
    import sys
    monkeypatch.setattr(sys.modules["dhj.calibrate_many"], "_PIPELINE_MIN_MARKETS", 1)   # pipeline 200 markets too
    four = dhj.calibrate_many(spots[sub], 0.03, K[sub], T, np.ones(15), market[sub], x0=x0[sub], pipelines=4,
                              gradient="analytic", **kw)
    for key in ("x", "final_loss", "status", "model_prices", "market_vols", "model_vols", "excluded_quotes"):
        assert np.array_equal(one[key], four[key], equal_nan=True), key
    fd = dhj.calibrate_many(spots[sub], 0.03, K[sub], T, np.ones(15), market[sub], x0=x0[sub], pipelines=1,
                            gradient="fd", **kw)
    assert np.isfinite(one["final_loss"]).all() and np.isfinite(fd["final_loss"]).all()
    rmse = np.sqrt(np.nanmean((one["model_vols"] - one["market_vols"]) ** 2, axis=1))
    # the quotes carry 2 % multiplicative price noise: the fit sits at the noise level, not at 0
    assert np.median(rmse) < 0.05
    # all 10 000 markets: how many quotes have no implied vol
    _, st = dhj.default_context().implied_vol(market, spots, K, T, np.ones(15), 0.03, 0.0, return_status=True)
    print(f"C5 (10 000 markets x 15 quotes): {(st != 0).sum()} quotes excluded, in {(st != 0).any(axis=1).sum()} "
          f"markets; 200-market IV RMSE median {np.median(rmse):.3e}; analytic / FD final loss median "
          f"{np.median(one['final_loss'] / fd['final_loss']):.4f}")
    assert np.array_equal(one["excluded_quotes"], (st[sub] != 0).sum(axis=1))


def test_calibrate_many_iv_drops_markets_without_quotes():
    import dhj
    spots, K, T, market = _c5(20)
    market = market.copy()
    market[3] = 2.0 * spots[3]                          # every quote at or above the upper bound
    np.random.seed(0)
    res = dhj.calibrate_many(spots, 0.03, K, T, np.ones(15), market, maxiter=50, multi_start=3, objective="iv",
                             pipelines=1, gradient="analytic", return_all_starts=True)
    assert res["status"][3] == 4 and not res["success"][3] and np.isnan(res["final_loss"][3])
    assert np.isnan(res["x"][3]).all() and res["excluded_quotes"][3] == 15
    others = np.arange(20) != 3
    assert np.isfinite(res["final_loss"][others]).all()
    # the other markets are what they are without the dropped one
    np.random.seed(0)
    x0 = dhj.initial_guesses(spots, K, T, market, 3)
    ref = dhj.calibrate_many(spots[others], 0.03, K[others], T, np.ones(15), market[others], maxiter=50,
                             multi_start=3, objective="iv", pipelines=1, gradient="analytic", x0=x0[others])
    assert np.array_equal(res["final_loss"][others], ref["final_loss"])


def test_calibrate_many_sharded_iv_single_rank():
    """calibrate_many_sharded forwards objective="iv" to calibrate_many through **kwargs and returns the IV outputs;
    without a process group it is one rank holding every market, with calibrate_many's results."""
    import dhj
    spots, K, T, market = _c5(30)
    np.random.seed(0)
    sh = dhj.calibrate_many_sharded(spots, 0.03, K, T, np.ones(15), market, maxiter=50, multi_start=3,
                                    objective="iv", gradient="analytic", pipelines=1)
    np.random.seed(0)
    ref = dhj.calibrate_many(spots, 0.03, K, T, np.ones(15), market, maxiter=50, multi_start=3, objective="iv",
                             gradient="analytic", pipelines=1)
    for key in ("x", "final_loss", "status", "model_prices", "market_vols", "model_vols", "excluded_quotes"):
        assert np.array_equal(sh[key], ref[key], equal_nan=True), key
    assert sh["market_vols"].shape == (30, 15) and np.isfinite(sh["model_vols"]).any()
