"""The implied-volatility calibration objective on the CPU (tests/iv_loss_oracle.py): its exact gradient against
Richardson central differences of its own frozen-range objective, and the rule that leaves out quotes without an
implied vol."""
import os

import numpy as np
import pytest

import iv_loss_oracle as IL
from conftest import ROOT
from oracle import cos_oracle as O

# worst |g - Richardson| / |g|inf measured 2.3e-11 over the states below (c1 1.0e-11, ragged 1.6e-13, C1 market
# 2.3e-11); pinned with 10x headroom
GRAD_TOL = 2.5e-10
H = 1e-3                 # difference step in x: Richardson's O(h^6) error term is far below the tolerance


def iv_markets():
    """(tag, S0, r, K, T, call, market, x[3]): the two loss_cases.npz markets and the C1 market (initial_guess.npz),
    each with three states away from an exact fit and from the Feller kink."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "loss_cases.npz"))
    gi = np.load(os.path.join(ROOT, "tests", "golden", "initial_guess.npz"))
    out = []
    for tag in ("c1", "ragged"):
        out.append((tag, float(g[f"{tag}_spot"]), float(g[f"{tag}_r"]), g[f"{tag}_strike"], g[f"{tag}_maturity"],
                    g[f"{tag}_is_call"].astype(bool), g[f"{tag}_market"]))
    out.append(("c1_guess", float(gi["spot"]), float(gi["r"]), gi["strike"], gi["maturity"], np.ones(15, bool),
                gi["market"]))
    p_lit = np.array([0.04, 2.5, 0.04, 0.3, -0.7, 0.04, 0.5, 0.04, 0.2, -0.5, 0.15, -0.04, 0.08])
    x_lit = O.inverse_transform_params(p_lit)
    rng = np.random.default_rng(21)
    res = []
    for tag, S0, r, K, T, call, mk in out:
        xs = [x_lit + 0.1 * rng.standard_normal(13) for _ in range(2)]
        feller = x_lit.copy()
        feller[3] = np.log(0.6)                         # Feller term active on both factors
        feller[6] = np.log(0.6) - 1.0
        res.append((tag, S0, r, np.asarray(K, float), np.asarray(T, float), call, np.asarray(mk, float),
                    np.vstack(xs + [feller])))
    return res


def _far_from_kink(x, steps):
    p = O.transform_params(np.vstack([x + s * np.eye(13)[i] for i in range(13) for s in (-steps, steps)]))
    e = np.stack([p[:, 3] ** 2 - 2 * p[:, 1] * p[:, 2], p[:, 8] ** 2 - 2 * p[:, 6] * p[:, 7]], axis=1)
    e0 = O.transform_params(x[None, :])
    e0 = np.array([e0[0, 3] ** 2 - 2 * e0[0, 1] * e0[0, 2], e0[0, 8] ** 2 - 2 * e0[0, 6] * e0[0, 7]])
    return (np.sign(e) == np.sign(e0)).all()


@pytest.mark.parametrize("m", range(3))
def test_iv_gradient_vs_richardson(m):
    tag, S0, r, K, T, call, mk, x = iv_markets()[m]
    mvol, st = IL.market_vols(S0, r, K, T, call, mk)
    assert (st == 0).all()
    f, g = IL.iv_loss_grad_batch(x, S0, r, K, T, call, mk, mvol=mvol)
    assert (f != O.SENTINEL).all()
    worst = 0.0
    for c in range(len(x)):
        assert _far_from_kink(x[c], 4 * H)
        _, ab = O.price_batch(O.transform_params(x[c])[None, :], S0, K, T, call, r, return_ab=True)
        sig0 = IL.implied_vols(O.price_batch(O.transform_params(x[c])[None, :], S0, K, T, call, r)[0], S0, K, T, r,
                               call, guess=mvol)[0]
        pts = []
        for i in range(13):
            for s in (1, -1, 2, -2, 4, -4):
                v = x[c].copy()
                v[i] += s * H
                pts.append(v)
        fv = IL.iv_loss_frozen(np.array(pts), S0, r, K, T, call, mvol, ab[0], guess=sig0).reshape(13, 6)
        d1, d2, d4 = ((fv[:, 2 * k] - fv[:, 2 * k + 1]) / (2 * (1 << k) * H) for k in range(3))
        r1, r2 = (4 * d1 - d2) / 3, (4 * d2 - d4) / 3
        rich = (16 * r1 - r2) / 15
        err = np.abs(rich - g[c]).max() / np.abs(g[c]).max()
        worst = max(worst, err)
        # f at the state itself: the frozen objective at its own range is the objective
        assert IL.iv_loss_frozen(x[c][None, :], S0, r, K, T, call, mvol, ab[0])[0] == pytest.approx(f[c], rel=1e-13)
    print(f"{tag}: worst |g - Richardson| / |g|inf {worst:.2e}")
    assert worst <= GRAD_TOL


def test_iv_sentinel_on_oracle():
    tag, S0, r, K, T, call, mk, x = iv_markets()[0]
    bad = x[0].copy()
    bad[2] = np.nan
    f, g = IL.iv_loss_grad_batch(np.vstack([x[0], bad]), S0, r, K, T, call, mk)
    assert f[0] != O.SENTINEL and f[1] == O.SENTINEL and (g[1] == 0).all()


def test_iv_exclusion_on_oracle():
    """A quote pushed below its intrinsic value has no implied vol: it is left out, and f equals f of the same market
    without that option."""
    tag, S0, r, K, T, call, mk, x = iv_markets()[2]
    mk = mk.copy()
    o = 0                                               # 90-strike call, T = 0.25: intrinsic D (F - K) > 0
    mk[o] = 0.98 * max(S0 - K[o] * np.exp(-r * T[o]), 0.0)
    mvol, st = IL.market_vols(S0, r, K, T, call, mk)
    assert st[o] == 1 and np.isnan(mvol[o]) and (np.delete(st, o) == 0).all()
    f, g = IL.iv_loss_grad_batch(x, S0, r, K, T, call, mk)
    keep = np.arange(len(K)) != o
    f2, g2 = IL.iv_loss_grad_batch(x, S0, r, K[keep], T[keep], call[keep], mk[keep])
    np.testing.assert_allclose(f, f2, rtol=1e-14)
    np.testing.assert_allclose(g, g2, rtol=1e-12, atol=1e-14 * np.abs(g).max())
