"""The Greeks on the device: k_price_greeks's (delta, gamma, theta, rho, rho_q) against the dual-number oracle
(tests/greeks_oracle.py), against the device's own prices, determinism over launch compositions, NaN handling,
the checked build and the DoubleHeston drop-in.

Every Greek is defined with the truncation range held at its value for the current inputs (frozen range)."""
import os

import numpy as np
import pytest

import greeks_oracle as G
from conftest import PKG
from oracle import cos_oracle as O

pytestmark = pytest.mark.gpu

TOL = 1e-10              # of each Greek's column scale (largest |entry| of the set's options), as the Jacobian's
CHECKED = os.path.join(PKG, "lib", "libdhj_checked.so")


@pytest.fixture(scope="module")
def ctx():
    import dhj
    c = dhj.Context(0)
    yield c
    c.close()


def _families():
    """(name, params, S0, K, T, call, r, q): the generator grid; calls and puts mixed with a dividend yield; per-set
    spots and strikes; binding strikes (short T, far strikes); a 200 x 20 surface (more than 64 strikes per slice)."""
    rng = np.random.default_rng(21)
    lo, hi = O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1]
    params = lo + (hi - lo) * rng.random((24, 13))
    K5, T5 = np.tile(O.GENERATOR_STRIKES_REL, 3), np.repeat(O.GENERATOR_MATURITIES, 5)
    out = [("grid", params, 100.0, K5, T5, np.ones(15, bool), 0.03, 0.0),
           ("mixed", params, 100.0, K5, T5, np.arange(15) % 2 == 0, 0.03, 0.01)]
    S0 = 80.0 + 40.0 * rng.random(24)
    Kp = S0[:, None] * (0.85 + 0.3 * rng.random((24, 15)))
    out.append(("per_set", params, S0, Kp, T5, np.arange(15) % 3 != 0, 0.02, 0.0))
    Ke, Te = np.linspace(50.0, 150.0, 9), np.array([0.02, 0.1, 1.0])
    out.append(("binding", params[:8], 100.0, np.tile(Ke, 3), np.repeat(Te, 9), np.arange(27) % 3 != 0, 0.03, 0.0))
    Ks, Ts = np.linspace(60.0, 140.0, 200), np.linspace(0.1, 2.0, 20)
    out.append(("surface", params[:3], 100.0, np.tile(Ks, 20), np.repeat(Ts, 200), np.arange(4000) % 2 == 0, 0.03,
                0.0))
    return out


def _err(got, want):
    scale = np.abs(want).max(axis=1, keepdims=True)
    return np.abs(got - want) / scale


@pytest.mark.parametrize("N", [128, 256, 100])
@pytest.mark.parametrize("fam", range(5))
def test_greeks_vs_oracle(ctx, fam, N):
    """Device against the oracle at <= 1e-10 of each Greek's column scale; out_price against dhj_price_list."""
    name, params, S0, K, T, call, r, q = _families()[fam]
    prices, greeks = ctx.price_greeks(params, S0, K, T, call, r, q, N=N)
    want_p, want_g = G.greeks_batch(params, S0, K, T, call, r, q, N=N)
    err = _err(greeks, want_g)
    print(f"{name} N={N}: worst |greek - oracle| / column scale per Greek {err.max(axis=(0, 1))}")
    assert err.max() <= TOL, (name, err.max(axis=(0, 1)))
    # the prices that come with the Greeks against dhj_price_list, whose tuned kernels order the arithmetic
    # differently: <= 1e-13 of the set's largest price (per option, measured up to 1.4e-12 relative on prices near
    # 1e-3 S0 on one B200, ~3e-15 of the set's scale)
    ref = ctx.price_list(params, S0, K, T, call, r, q, N=N)
    assert (np.abs(prices - ref) <= 1e-13 * np.abs(ref).max(axis=1, keepdims=True)).all()
    assert (np.abs(prices - want_p) <= 1e-10 * np.max(S0)).all()


def test_gamma_put_call_and_delta_vs_differences(ctx):
    """gamma_call == gamma_put for the same strike; delta against Richardson differences of price_list in S0 on
    strikes whose widening does not bind (there [a, b] does not move with S0)."""
    name, params, S0, K, T, call, r, q = _families()[0]
    _, gc = ctx.price_greeks(params, S0, K, T, True, r, q)
    _, gp = ctx.price_greeks(params, S0, K, T, False, r, q)
    assert np.array_equal(gc[..., 1], gp[..., 1])
    for c in (True, False):
        _, g = ctx.price_greeks(params, S0, K, T, c, r, q)
        h = 0.5
        d = [(ctx.price_list(params, S0 + m * h, K, T, c, r, q) - ctx.price_list(params, S0 - m * h, K, T, c, r, q))
             / (2 * m * h) for m in (1, 2, 4)]
        r1, r2 = (4 * d[0] - d[1]) / 3, (4 * d[1] - d[2]) / 3
        fd = (16 * r1 - r2) / 15
        free = ~G.binding(params, S0, K, T, r)
        assert free.all()
        err = (np.abs(fd - g[..., 0]) / np.abs(g[..., 0]).max(axis=1, keepdims=True)).max()
        print(f"call={c}: delta vs Richardson differences of price_list {err:.2e}")
        assert err <= 1e-8


def test_greeks_deterministic(ctx):
    """A set's outputs are bit-identical alone, among 10 000 sets and over two calls."""
    name, params, S0, K, T, call, r, q = _families()[1]
    rng = np.random.default_rng(4)
    big = params[rng.integers(0, len(params), 10000)] * (1 + 1e-3 * rng.standard_normal((10000, 13)))
    probe = big[4321].copy()
    p1, g1 = ctx.price_greeks(probe, S0, K, T, call, r, q)
    pb, gb = ctx.price_greeks(big, S0, K, T, call, r, q)
    pb2, gb2 = ctx.price_greeks(big, S0, K, T, call, r, q)
    assert np.array_equal(p1[0], pb[4321]) and np.array_equal(g1[0], gb[4321])
    assert np.array_equal(pb, pb2) and np.array_equal(gb, gb2)


def test_greeks_nan_and_empty(ctx):
    import dhj
    name, params, S0, K, T, call, r, q = _families()[1]
    bad = params[:6].copy()
    bad[1, 2] = np.nan
    bad[3, 12] = np.nan
    bad[4, 4] = np.inf
    prices, greeks = ctx.price_greeks(bad, S0, K, T, call, r, q)
    ref = ctx.price_list(bad, S0, K, T, call, r, q)
    assert np.array_equal(np.isnan(prices), np.isnan(ref)) and np.isnan(ref).any()
    assert np.array_equal(np.isnan(greeks), np.repeat(np.isnan(ref)[..., None], 5, axis=2))
    p0, g0 = ctx.price_greeks(np.empty((0, 13)), S0, K, T, call, r)
    assert p0.shape == (0, 15) and g0.shape == (0, 15, 5)
    pm, gm = ctx.price_greeks(params, S0, [], [], [], r)
    assert pm.shape == (24, 0) and gm.shape == (24, 0, 5)
    lib = dhj.load_library()
    one = np.ascontiguousarray(params[:1])
    Ka, Ta, ca = np.ascontiguousarray(K), np.ascontiguousarray(T), np.ones(15, np.int32)
    out = np.empty(15)
    assert lib.dhj_price_greeks(ctx._h, one, 1, np.array([100.0]), 0, r, 0.0, Ka, 0, Ta, ca, 15, 128, 10.0,
                                out.ctypes.data, None) == -1
    assert lib.dhj_price_greeks(ctx._h, one, 1, np.array([100.0]), 0, r, 0.0, Ka, 0, Ta, ca, 15, 128, 10.0, None,
                                np.empty(75).ctypes.data) == -1


def test_checked_build_greeks():
    """Zero violations and the product build's bits on the binding family, the surface and the multi-chunk slices of
    test_gpu_derivative_edges (449 strikes with binding strikes at the 224 boundary, ragged N, per-set rows, and the
    reversed and one-option compositions)."""
    import dhj
    import test_gpu_derivative_edges as E
    edge = [E._greeks_case(n)[:8] for n in ("bind224-128", "bind224-33", "n449", "per_set")]
    pe, Se, Ke, Te, ce, re, qe, Ne = edge[0]
    edge.append((pe, Se, Ke[::-1], Te[::-1], ce[::-1], re, qe, Ne))
    edge.append((pe, Se, Ke[224:225], Te[224:225], ce[224:225], re, qe, Ne))
    outs = []
    for lib in (None, CHECKED):
        c = dhj.Context(0, library=lib)
        res = [c.price_greeks(*_families()[f][1:]) for f in (3, 4)]
        res += [c.price_greeks(p, s, k, t, cc, rr, qq, N=n) for p, s, k, t, cc, rr, qq, n in edge]
        if lib:
            enabled, counts = c.debug_checks()
            assert enabled and not counts.any(), counts
        outs.append(res)
        c.close()
    for (pa, ga), (pb, gb) in zip(*outs):
        assert np.array_equal(pa, pb) and np.array_equal(ga, gb)


def test_double_heston_greeks(ctx):
    import sys
    p = os.path.join(PKG, "src", "models")
    if p not in sys.path:
        sys.path.insert(0, p)
    from double_heston import DoubleHeston
    params = np.array([0.04, 2.5, 0.04, 0.3, -0.7, 0.04, 0.5, 0.04, 0.2, -0.5, 0.15, -0.04, 0.08])
    for opt in ("C", "put"):
        m = DoubleHeston(100.0, 95.0, 0.5, 0.03, *params, option_type=opt, q=0.01)
        got = m.greeks()
        _, g = ctx.price_greeks(params, 100.0, [95.0], [0.5], [opt == "C"], 0.03, 0.01)
        assert list(got) == ["delta", "gamma", "theta", "rho", "rho_q"]
        assert np.array_equal(np.array(list(got.values())), g[0, 0])
