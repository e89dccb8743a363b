"""The analytic parameter gradient on the device: k_price_jac's price Jacobian and k_loss_grad_reduce's (f, g) against
the dual-number oracle (tests/jac_oracle.py), against the device's own prices / losses, determinism over launch
compositions, the checked build, and calibrations driven by the analytic gradient.

Every derivative is defined with the truncation range held at its value for the current parameters (frozen range)."""
import os

import numpy as np
import pytest

import jac_oracle as J
from conftest import PKG
from test_jacobian_cpu import _off_kink
from oracle import cos_oracle as O

pytestmark = pytest.mark.gpu

JAC_TOL = 1e-10          # of the column's largest |entry|, as the host emulation
CHECKED = os.path.join(PKG, "lib", "libdhj_checked.so")


@pytest.fixture(scope="module")
def ctx():
    import dhj
    c = dhj.Context(0)
    yield c
    c.close()


def _families():
    """(name, params, S0, K, T, call, r): generator-range sets on the C1 / C5 grid with calls and puts, the C3 edge
    strikes (binding widening), and a dense slice of 40 strikes per maturity."""
    rng = np.random.default_rng(11)
    lo, hi = O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1]
    params = lo + (hi - lo) * rng.random((24, 13))
    K5, T5 = np.tile(O.GENERATOR_STRIKES_REL, 3), np.repeat(O.GENERATOR_MATURITIES, 5)
    out = [("grid_calls", params, 100.0, K5, T5, np.ones(15, bool), 0.03),
           ("grid_mixed", params, 100.0, K5, T5, np.arange(15) % 2 == 0, 0.03)]
    Ke, Te = np.linspace(50.0, 150.0, 9), np.array([0.02, 0.1, 1.0])
    out.append(("edge", params[:8], 100.0, np.tile(Ke, 3), np.repeat(Te, 9), np.arange(27) % 3 != 0, 0.03))
    Kd, Td = np.linspace(80.0, 120.0, 40), np.array([0.25, 1.5])
    out.append(("dense", params[:6], 100.0, np.tile(Kd, 2), np.repeat(Td, 40), np.arange(80) % 5 != 0, 0.03))
    return out


@pytest.mark.parametrize("N", [128, 256])
@pytest.mark.parametrize("fam", range(4))
def test_price_jacobian_vs_oracle(ctx, fam, N):
    name, params, S0, K, T, call, r = _families()[fam]
    prices, jac = ctx.price_jacobian(params, S0, K, T, call, r, N=N)
    want_p, want_j = J.price_jacobian_batch(params, S0, K, T, call, r, N=N)
    scale = np.abs(want_j).max(axis=1, keepdims=True)
    err = np.abs(jac - want_j) / scale
    print(f"{name} N={N}: worst |jac - oracle| / column scale {err.max():.2e}")
    assert err.max() <= JAC_TOL, (name, err.max(axis=(0, 1)))
    # the prices that come with the Jacobian are the pricing kernel's to 1e-12 where the price is not tiny
    ref = ctx.price_list(params, S0, K, T, call, r, N=N)
    big = ref >= 1e-3 * S0
    assert (np.abs(prices - ref)[big] <= 1e-12 * ref[big]).all(), np.abs(prices / ref - 1)[big].max()
    assert (np.abs(prices - want_p) <= 1e-10 * S0).all()


def _markets():
    import dhj
    g = np.load(os.path.join(PKG, "..", "tests", "golden", "loss_cases.npz"))
    out = []
    for tag in ("c1", "ragged"):
        out.append((tag, float(g[f"{tag}_spot"]), float(g[f"{tag}_r"]), g[f"{tag}_strike"], g[f"{tag}_maturity"],
                    g[f"{tag}_is_call"].astype(bool), g[f"{tag}_market"], g[f"{tag}_x"]))
    # more than 8 strikes per maturity (the dense pricing path of the FD loss)
    Kd, Td = np.linspace(85.0, 115.0, 12), np.array([0.3, 1.2])
    K, T, call = np.tile(Kd, 2), np.repeat(Td, 12), np.arange(24) % 4 != 0
    p_true = np.array([0.04, 2.5, 0.04, 0.3, -0.7, 0.04, 0.5, 0.04, 0.2, -0.5, 0.15, -0.04, 0.08])
    mk = O.price_batch(p_true, 100.0, K, T, call, 0.02)[0] * (1 + 0.02 * np.random.default_rng(5).standard_normal(24))
    x = O.inverse_transform_params(p_true)[None, :] + 0.2 * np.random.default_rng(6).standard_normal((12, 13))
    out.append(("dense12", 100.0, 0.02, K, T, call, mk, x))
    res = []
    for tag, S0, r, K, T, call, mk, x in out:
        x = np.array(x, dtype=np.float64)
        feller = O.inverse_transform_params(p_true).copy()
        feller[3] = np.log(0.6)                       # sigma1^2 > 2 kappa1 theta1: Feller term active
        feller[6] = np.log(0.6)                       # (the literature values sit exactly on factor 2's kink)
        bad = x[0].copy()
        bad[2] = np.nan                               # NaN parameter -> sentinel
        res.append((tag, S0, r, K, T, call, mk, np.vstack([x, feller, bad])))
    return res


@pytest.mark.parametrize("m", range(3))
def test_loss_grad(ctx, m):
    tag, S0, r, K, T, call, mk, x = _markets()[m]
    market = ctx.market(S0, r, K, T, call, mk)
    f, g = market.loss_grad(x)
    want_f, want_g = J.loss_grad_batch(x, S0, r, K, T, call, mk)
    assert np.array_equal(f == O.SENTINEL, want_f == O.SENTINEL) and (f[-1] == O.SENTINEL) and (g[-1] == 0).all()
    assert (O.feller_penalty(O.transform_params(x[-2])) > 0)
    ok = f != O.SENTINEL
    # at an exact fit (f ~ 1e-28) the residuals, hence g, are rounding noise: only its size is checked there
    fit = ok & (f < 1e-20)
    assert (np.abs(g[fit]) <= 1e-10).all() and (np.abs(want_g[fit]) <= 1e-10).all()
    gscale = np.maximum(np.abs(want_g).max(axis=1), 1e-12)
    gerr = np.where(fit, 0.0, np.abs(g - want_g).max(axis=1) / gscale)
    print(f"{tag}: worst |g - oracle| / |g|inf {gerr.max():.2e}")
    assert (gerr <= 1e-9).all(), gerr
    # f is the device loss
    fl = market.loss_batch(x)
    assert np.array_equal(f == O.SENTINEL, fl == O.SENTINEL)
    # f is formed from the pricing kernel's prices in the loss path's order: the loss itself
    assert (np.abs(f - fl)[ok] <= 1e-12 * np.abs(fl[ok])).all(), np.abs(f / fl - 1)[ok].max()
    # g against a central difference of the device loss.  The difference also moves [a, b]; on the C1 and dense markets
    # that term is below 1e-6 of |g|inf, on the ragged market (K 80-120, T 0.25-1.5) it was measured at 4.1e-5 of
    # |g|inf on one B200 (the oracle, which freezes [a, b] the same way, agrees with the device to 1.5e-12 there)
    cd_tol = 1e-4 if tag == "ragged" else 1e-6
    h = 1e-5
    for c in np.flatnonzero(ok & (f > 1e-20) & _off_kink(x))[:6]:
        pts = np.repeat(x[c][None, :], 26, axis=0)
        for i in range(13):
            pts[2 * i, i] += h
            pts[2 * i + 1, i] -= h
        fv = market.loss_batch(pts)
        cd = (fv[0::2] - fv[1::2]) / (2 * h)
        assert np.abs(cd - g[c]).max() <= cd_tol * np.abs(g[c]).max(), (c, cd, g[c])


def test_loss_grad_deterministic(ctx):
    """A state's (f, g) is bit-identical alone, among 64 states, among 30 000 states, and on repeated calls."""
    tag, S0, r, K, T, call, mk, x = _markets()[0]
    market = ctx.market(S0, r, K, T, call, mk)
    rng = np.random.default_rng(9)
    big = x[rng.integers(0, len(x), 30000)] + 1e-3 * rng.standard_normal((30000, 13))
    probe = big[12345].copy()
    f1, g1 = market.loss_grad(probe[None, :])
    f64, g64 = market.loss_grad(np.vstack([big[:40], probe[None, :], big[40:63]]))
    fb, gb = market.loss_grad(big)
    assert f1[0] == f64[40] == fb[12345]
    assert np.array_equal(g1[0], g64[40]) and np.array_equal(g1[0], gb[12345])
    f2, g2 = market.loss_grad(big)
    assert np.array_equal(fb, f2) and np.array_equal(gb, g2)


def test_checked_build_jacobian():
    """Zero violations and the product build's bits on: the binding family, the multi-chunk slices of
    test_gpu_derivative_edges (129 strikes with binding strikes at the chunk boundary, every strike binding, 200
    strikes, ragged N, per-set rows, and the reversed and one-option compositions), the dense market's loss_grad and
    loss_grad over 16 markets with a shuffled market_index."""
    import dhj
    import test_gpu_derivative_edges as E
    name, params, S0, K, T, call, r = _families()[2]
    tag, S0m, rm, Km, Tm, callm, mk, x = _markets()[2]
    edge_cases = [E._jac_case(n)[:9] for n in ("bind_edges-128", "bind_edges-33", "all_bind", "n200", "per_set_L12")]
    pe, Se, Ke, Te, ce, re, qe, Ne, Le = edge_cases[0]
    edge_cases.append((pe, Se, Ke[::-1], Te[::-1], ce[::-1], re, qe, Ne, Le))
    edge_cases.append((pe, Se, Ke[64:65], Te[64:65], ce[64:65], re, qe, Ne, Le))
    many = None
    outs = []
    for lib in (None, CHECKED):
        c = dhj.Context(0, library=lib)
        if many is None:
            many = E._multi_market(c, 16, 3)
        Sm, rmm, Kmm, Tmm, cm, mkm, xm, im = many
        res = [c.price_jacobian(params, S0, K, T, call, r), c.market(S0m, rm, Km, Tm, callm, mk).loss_grad(x),
               c.market(Sm, rmm, Kmm, Tmm, cm, mkm).loss_grad(xm, im)]
        res += [c.price_jacobian(p, s, k, t, cc, rr, qq, N=n, L=l) for p, s, k, t, cc, rr, qq, n, l in edge_cases]
        if lib:
            enabled, counts = c.debug_checks()
            assert enabled and not counts.any(), counts
        outs.append(res)
        c.close()
    for a, b in zip(*outs):
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


# ---- calibrations driven by the analytic gradient ---------------------------------------------------------------
@pytest.fixture(scope="module")
def cal():
    import sys
    p = os.path.join(PKG, "src", "calibration")
    if p not in sys.path:
        sys.path.insert(0, p)
    import lbfgs_calibrator
    return lbfgs_calibrator


def test_calibrate_analytic_c1(cal, golden):
    """calibrate(gradient="analytic") on the C1 market (seed 0, three starts) converges, at a final loss no worse than
    the worst the reference reaches in its basin A (calib_ensemble.npz: 7.97e-7)."""
    gi = golden("initial_guess.npz")
    opts = [{"strike": float(gi["strike"][j]), "maturity": float(gi["maturity"][j]), "price": float(gi["market"][j]),
             "option_type": "call"} for j in range(15)]
    c = cal.DoubleHestonJumpCalibrator(float(gi["spot"]), float(gi["r"]), opts)
    np.random.seed(0)
    res = c.calibrate(maxiter=300, multi_start=3, gradient="analytic")
    ens = golden("calib_ensemble.npz")
    basin_a = ens["fun"][ens["nit"] == 17]
    print(f"C1 analytic: final loss {res.final_loss:.6e}, n_calls {c.n_calls}; reference basin A worst "
          f"{basin_a.max():.6e}")
    assert res.success and res.final_loss <= basin_a.max()
    f, g = c.compute_loss_and_grad(c.inverse_transform_params(res.parameters), gradient="analytic")
    assert np.isfinite(g).all()


def test_calibrate_many_analytic_c5():
    """calibrate_many(gradient="analytic") on the C5 inputs (10 000 markets x 3 starts) fits to the noise level like
    the FD path; on a 200-market sub-sample the final losses match the FD path's (median ratio <= 1.02)."""
    import time

    import dhj
    ctx = dhj.default_context()
    n = 10000
    lo, hi = O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1]
    data = ctx.generate(7, 0, n, 500, lo, hi, 0.9, 100.0, 0.0003, 0.01, 0.02, O.GENERATOR_STRIKES_REL,
                        O.GENERATOR_MATURITIES, 0.03)
    spots, market = data["spots"], data["market"]
    K = np.tile(O.GENERATOR_STRIKES_REL[None, :] * spots[:, None] / 100.0, (1, 3))
    T = np.repeat(O.GENERATOR_MATURITIES, 5)
    x0 = dhj.initial_guesses(spots, K, T, market, 3)
    t0 = time.perf_counter()
    res = dhj.calibrate_many(spots, 0.03, K, T, np.ones(15), market, maxiter=300, multi_start=3, x0=x0,
                             gradient="analytic")
    wall = time.perf_counter() - t0
    print(f"C5 analytic: {wall:.3f} s, {res['rounds']} rounds, {res['evaluations']} evaluations, median final loss "
          f"{np.median(res['final_loss']):.3e}")
    assert res["x"].shape == (n, 13) and np.isfinite(res["final_loss"]).all()
    assert np.quantile(res["final_loss"] / data["loss"], 0.99) < 5.0 and (res["final_loss"] < 0.1).all()
    sub = np.random.default_rng(3).choice(n, size=200, replace=False)
    fd = dhj.calibrate_many(spots[sub], 0.03, K[sub], T, np.ones(15), market[sub], maxiter=300, multi_start=3,
                            x0=x0[sub])
    an = dhj.calibrate_many(spots[sub], 0.03, K[sub], T, np.ones(15), market[sub], maxiter=300, multi_start=3,
                            x0=x0[sub], gradient="analytic")
    ratio = an["final_loss"] / fd["final_loss"]
    q5, q50, q95 = np.quantile(ratio, [0.05, 0.5, 0.95])
    print(f"analytic / FD final loss on 200 markets: 5% {q5:.4f}, median {q50:.4f}, 95% {q95:.4f}")
    assert q50 <= 1.02 and q5 >= 0.8 and q95 <= 1.15       # measured on one B200: 0.910 / 0.999 / 1.021
    assert np.array_equal(an["final_loss"], res["final_loss"][sub])    # a state does not depend on its batch
