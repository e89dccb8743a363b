"""Implied volatility on the device: k_implied_vol / k_bs_price through dhj_implied_vol, dhj_implied_vol_dev and
dhj_bs_price, against the mpmath reference (tests/iv_oracle.py).

Domain A is the round-trip contract of tests/test_iv_cpu.py on the device.  Domain B inverts COS prices of the
Double-Heston model: status against a NumPy classification by the no-arbitrage bounds, the price residual of the
returned vol, and call/put consistency up to the COS parity residual."""
import ctypes

import numpy as np
import pytest

import iv_oracle as IV
from oracle import cos_oracle as O

pytestmark = pytest.mark.gpu

EPS = IV.EPS
C_BOUND = 7.0      # as tests/test_iv_cpu.py; on the device: measured max c 3.10, median 0.45 (DESIGN.md §6d)


@pytest.fixture(scope="module")
def ctx():
    import dhj
    c = dhj.Context(0)
    yield c
    c.close()


def _params(n, seed):
    rng = np.random.default_rng(seed)
    lo, hi = O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1]
    return lo + (hi - lo) * rng.random((n, 13))


def _bounds(S0, K, T, r, q, call):
    Sq, KD = S0 * np.exp(-q * T), K * np.exp(-r * T)
    lower = np.where(call, np.maximum(Sq - KD, 0.0), np.maximum(KD - Sq, 0.0))
    return lower, np.where(call, Sq, KD)


def _expected_status(V, S0, K, T, r, q, call):
    """NumPy classification: 1 below the lower bound, 2 at or above the upper bound, else 0.  Prices within 4 ulp of
    a bound may go either way (the device and NumPy round the bounds' exponentials independently): -1."""
    lower, upper = _bounds(S0, K, T, r, q, call)
    st = np.where(V < lower, 1, np.where(V >= upper, 2, 0))
    near = (np.abs(V - lower) <= 4 * EPS * np.maximum(lower, 1e-300)) | (np.abs(V - upper) <= 4 * EPS * upper)
    return np.where(near, -1, st)


def test_domain_a_on_device(ctx):
    d = IV.domain_a(4096, seed=11)
    vol = np.empty(d["V"].size)
    for i in range(vol.size):
        v, st = ctx.implied_vol([d["V"][i]], d["S0"][i], [d["K"][i]], [d["T"][i]], [bool(d["call"][i])], d["r"][i],
                                d["q"][i], return_status=True)
        assert st[0, 0] == 0, i
        vol[i] = v[0, 0]
    c = np.array([IV.c_measure(v, *(d[k][i] for k in ("V", "S0", "K", "T", "r", "q", "call", "sigma")))[0]
                  for i, v in enumerate(vol)])
    print(f"domain A on the device: median c {np.median(c):.3f}, max c {c.max():.3f}")
    assert c.max() <= C_BOUND, c.max()
    assert np.median(c) <= 1.0


def test_bs_price_round_trip(ctx):
    """bs_price -> implied_vol on per-set spots and strikes, calls and puts: |sigma' - sigma| <= 64 eps (sigma +
    V / vega) on every option whose time value is above 64 ulp of its price."""
    rng = np.random.default_rng(2)
    P, M = 64, 24
    S0 = rng.choice([1.0, 100.0, 1e4], P)
    T = np.exp(rng.uniform(np.log(1 / 365), np.log(10.0), M))
    call = np.arange(M) % 2 == 0
    sigma = np.exp(rng.uniform(np.log(0.01), np.log(3.0), (P, M)))
    K = S0[:, None] * np.exp(0.01 * T - rng.uniform(-4, 4, (P, M)) * sigma * np.sqrt(T))
    r, q = 0.04, 0.015
    V = ctx.bs_price(sigma, S0, K, T, call, r, q)
    back, st = ctx.implied_vol(V, S0, K, T, call, r, q, return_status=True)
    lower, _ = _bounds(S0[:, None], K, T, r, q, call)
    sel = (V - lower) > 64 * np.spacing(V)
    assert sel.mean() > 0.9
    assert (st[sel] == 0).all()
    idx = np.flatnonzero(sel)[::7]
    for i in idx:
        p, m = divmod(i, M)
        vega = float(IV.bs_vega(S0[p], K[p, m], T[m], r, q, sigma[p, m]))
        assert abs(back[p, m] - sigma[p, m]) <= 64 * EPS * (sigma[p, m] + V[p, m] / vega), (p, m)


def _domain_b():
    """(name, params, S0, K, T, call, r, q, N) — the generator grid at 4 096 sets; mixed calls and puts with q > 0;
    per-set spots and strikes; the 200 x 20 surface at N = 256."""
    rng = np.random.default_rng(17)
    params = _params(4096, 3)
    K5, T5 = np.tile(O.GENERATOR_STRIKES_REL, 3), np.repeat(O.GENERATOR_MATURITIES, 5)
    S0 = 80.0 + 40.0 * rng.random(256)
    Kp = S0[:, None] * (0.8 + 0.4 * rng.random((256, 15)))
    Ks, Ts = np.linspace(60.0, 140.0, 200), np.linspace(0.1, 2.0, 20)
    return [("grid", params, 100.0, K5, T5, np.ones(15, bool), 0.03, 0.0, 128),
            ("mixed", params[:1024], 100.0, K5, T5, np.arange(15) % 2 == 0, 0.03, 0.02, 128),
            ("per_set", params[:256], S0, Kp, T5, np.arange(15) % 3 != 0, 0.02, 0.01, 128),
            ("surface", params[:8], 100.0, np.tile(Ks, 20), np.repeat(Ts, 200), np.arange(4000) % 2 == 0, 0.03, 0.0,
             256)]


@pytest.mark.parametrize("case", range(4))
def test_domain_b_model_prices(ctx, case):
    name, params, S0, K, T, call, r, q, N = _domain_b()[case]
    V = ctx.price_list(params, S0, K, T, call, r, q, N)
    vol, st = ctx.implied_vol(V, S0, K, T, call, r, q, return_status=True)
    P, M = V.shape
    S0b = np.broadcast_to(np.reshape(S0, (-1, 1)) if np.ndim(S0) else S0, (P, M))
    Kb, Tb, cb = np.broadcast_to(K, (P, M)), np.broadcast_to(T, (P, M)), np.broadcast_to(call, (P, M))
    want = _expected_status(V, S0b, Kb, Tb, r, q, cb)
    assert not (st == 4).any(), name
    sure = want >= 0
    assert (st[sure] == want[sure]).all(), (name, np.argwhere(st[sure] != want[sure])[:5])
    assert np.isin(st[~sure], (0, 1, 2)).all()
    assert np.isnan(vol[st != 0]).all() and np.isfinite(vol[st == 0]).all()
    ok = np.flatnonzero(st == 0)
    rng = np.random.default_rng(case)
    for i in rng.choice(ok, min(ok.size, 2000 if case == 0 else 500), replace=False):
        p, m = divmod(int(i), M)
        a = (S0b[p, m], Kb[p, m], Tb[p, m], r, q)
        got = IV.bs_price(*a, vol[p, m], bool(cb[p, m]))
        vega = IV.bs_vega(*a, vol[p, m]) if vol[p, m] > 0 else 0
        assert abs(float(got) - V[p, m]) <= 64 * EPS * (V[p, m] + vol[p, m] * float(vega)), (name, p, m)


def test_domain_b_call_put_consistency(ctx):
    """Call and put vols at the same (K, T) agree to within the COS parity residual over vega."""
    params = _params(256, 5)
    K5, T5 = np.tile(O.GENERATOR_STRIKES_REL, 3), np.repeat(O.GENERATOR_MATURITIES, 5)
    r, q, S0 = 0.03, 0.02, 100.0
    C = ctx.price_list(params, S0, K5, T5, True, r, q)
    Pp = ctx.price_list(params, S0, K5, T5, False, r, q)
    vc, sc = ctx.implied_vol(C, S0, K5, T5, True, r, q, return_status=True)
    vp, sp = ctx.implied_vol(Pp, S0, K5, T5, False, r, q, return_status=True)
    both = (sc == 0) & (sp == 0)
    assert both.mean() > 0.9
    F, D = S0 * np.exp((r - q) * T5), np.exp(-r * T5)
    s = vc * np.sqrt(T5)
    d1 = (np.log(F / K5) + s * s / 2) / s
    vega = D * F * np.exp(-d1 * d1 / 2) / np.sqrt(2 * np.pi) * np.sqrt(T5)
    resid = np.abs(C - Pp - (S0 * np.exp(-q * T5) - K5 * D)) + 64 * EPS * (C + Pp)
    assert (np.abs(vc - vp)[both] <= 2 * (resid / vega)[both]).all()


def test_dev_equals_host_and_scale_by_spot(ctx):
    """implied_vol_dev on a price_grid_dev surface (scale_by_spot, per-set spots, both on the device) is bit-identical
    to the host variant with explicit per-set strikes strikes * S0 / 100; two calls give identical bits."""
    import torch
    P = 512
    params = _params(P, 8)
    rng = np.random.default_rng(4)
    S0 = 50.0 + 100.0 * rng.random(P)
    strikes, mats = O.GENERATOR_STRIKES_REL, O.GENERATOR_MATURITIES
    nK, nT = strikes.size, mats.size
    dev = torch.device("cuda", 0)
    d_params = torch.from_numpy(params).to(dev)
    d_S0 = torch.from_numpy(S0).to(dev)
    d_price = torch.empty((P, nT, nK), dtype=torch.float64, device=dev)
    ctx.price_grid_dev(d_params.data_ptr(), P, d_S0.data_ptr(), 1, strikes, mats, 0.03, 0.01, 128, 10.0, True, False,
                       d_price.data_ptr())
    Kt, Tt = np.tile(strikes, nT), np.repeat(mats, nK)
    d_vol = torch.empty((P, nT * nK), dtype=torch.float64, device=dev)
    d_st = torch.empty((P, nT * nK), dtype=torch.int32, device=dev)
    ctx.implied_vol_dev(d_price.data_ptr(), P, d_S0.data_ptr(), 1, Kt, Tt, False, 0.03, 0.01, d_vol.data_ptr(),
                        d_st.data_ptr(), scale_by_spot=True)
    torch.cuda.synchronize()
    price = d_price.cpu().numpy().reshape(P, -1)
    host_vol, host_st = ctx.implied_vol(price, S0, Kt[None, :] * S0[:, None] / 100, Tt, False, 0.03, 0.01,
                                        return_status=True)
    assert np.array_equal(d_vol.cpu().numpy(), host_vol, equal_nan=True)
    assert np.array_equal(d_st.cpu().numpy(), host_st)
    assert (host_st == 0).mean() > 0.9
    again, again_st = ctx.implied_vol(price, S0, Kt[None, :] * S0[:, None] / 100, Tt, False, 0.03, 0.01,
                                      return_status=True)
    assert np.array_equal(again, host_vol, equal_nan=True) and np.array_equal(again_st, host_st)
    # without scaling and without a status array, on a scalar spot
    d_vol2 = torch.empty_like(d_vol)
    s0_one = torch.tensor([S0[0]], dtype=torch.float64, device=dev)
    ctx.implied_vol_dev(d_price.data_ptr(), P, s0_one.data_ptr(), 0, Kt, Tt, False, 0.03, 0.01, d_vol2.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(d_vol2.cpu().numpy(), ctx.implied_vol(price, S0[0], Kt, Tt, False, 0.03, 0.01),
                          equal_nan=True)


def test_edge_cases(ctx):
    S0, K, T, r, q = 100.0, 90.0, 0.5, 0.03, 0.01
    lower, upper = _bounds(S0, K, T, r, q, True)
    lower, upper = float(lower), float(upper)
    V = np.array([lower, np.nextafter(lower, 0), upper, np.nan, 5.0, 5.0, 12.0])
    Ks = np.array([K, K, K, K, 0.0, K, -1.0])
    Ts = np.array([T, T, T, T, T, -0.5, T])
    vol = np.empty(V.size)
    st = np.empty(V.size, np.int32)
    for i in range(V.size):    # one maturity per call: T varies
        v, s = ctx.implied_vol([V[i]], S0, [Ks[i]], [Ts[i]], [True], r, q, return_status=True)
        vol[i], st[i] = v[0, 0], s[0, 0]
    assert list(st) == [0, 1, 2, 3, 3, 3, 3]
    assert vol[0] == 0.0 and np.isnan(vol[1:]).all()
    empty = ctx.implied_vol(np.empty((0, 3)), 100.0, [90.0, 100.0, 110.0], [1.0, 1.0, 1.0], True, r)
    assert empty.shape == (0, 3)
    assert ctx.implied_vol(np.empty((4, 0)), 100.0, [], [], True, r).shape == (4, 0)
    assert ctx.bs_price(np.empty((0, 2)), 100.0, [90.0, 100.0], [1.0, 1.0], True, r).shape == (0, 2)


def test_null_pointers_and_strides(ctx):
    import dhj
    lib = ctypes.CDLL(dhj.LIB_PATH)      # raw entry points: no argtypes conversion
    vp, i64, i32, f64 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_double
    buf = np.ones(64)
    ib = np.zeros(64, np.int32)
    p = lambda a: vp(a.ctypes.data)  # noqa: E731

    def iv(price, S0, s0s, strike, ks, mat, call, out, status=None, M=4, P=2):
        return lib.dhj_implied_vol(ctx._h, price, i64(P), S0, i64(s0s), f64(0.03), f64(0.0), strike, i64(ks), mat,
                                   call, i32(M), out, status)
    ok = iv(p(buf), p(buf), 0, p(buf), 0, p(buf), p(ib), p(buf), p(ib))
    assert ok == 0
    for args in ((vp(None), p(buf), 0, p(buf), 0, p(buf), p(ib), p(buf)),
                 (p(buf), vp(None), 0, p(buf), 0, p(buf), p(ib), p(buf)),
                 (p(buf), p(buf), 0, vp(None), 0, p(buf), p(ib), p(buf)),
                 (p(buf), p(buf), 0, p(buf), 0, vp(None), p(ib), p(buf)),
                 (p(buf), p(buf), 0, p(buf), 0, p(buf), vp(None), p(buf)),
                 (p(buf), p(buf), 0, p(buf), 0, p(buf), p(ib), vp(None)),
                 (p(buf), p(buf), 2, p(buf), 0, p(buf), p(ib), p(buf)),
                 (p(buf), p(buf), 0, p(buf), 3, p(buf), p(ib), p(buf))):
        assert iv(*args) == -1
    assert iv(p(buf), p(buf), 0, p(buf), 0, p(buf), p(ib), p(buf), M=-1) == -1
    assert lib.dhj_implied_vol(None, p(buf), i64(1), p(buf), i64(0), f64(0.0), f64(0.0), p(buf), i64(0), p(buf),
                               p(ib), i32(1), p(buf), None) == -1
    assert lib.dhj_bs_price(ctx._h, p(buf), i64(1), p(buf), i64(1), f64(0.0), f64(0.0), p(buf), i64(5), p(buf),
                            p(ib), i32(4), p(buf)) == -1
    assert lib.dhj_implied_vol_dev(ctx._h, vp(None), i64(1), p(buf), i64(0), f64(0.0), f64(0.0), p(buf), i32(0),
                                   p(buf), p(ib), i32(4), p(buf), None, None) == -1
    assert lib.dhj_implied_vol_dev(ctx._h, p(buf), i64(1), p(buf), i64(0), f64(0.0), f64(0.0), vp(None), i32(0),
                                   p(buf), p(ib), i32(4), p(buf), None, None) == -1


def test_double_heston_implied_volatility(ctx):
    import os
    import sys

    import dhj
    from conftest import PKG
    p = os.path.join(PKG, "src", "models")
    if p not in sys.path:
        sys.path.insert(0, p)
    from double_heston import DoubleHeston
    args = (100.0, 95.0, 0.5, 0.03, 0.04, 2.5, 0.04, 0.3, -0.7, 0.04, 0.5, 0.04, 0.2, -0.5, 0.15, -0.04, 0.08)
    for opt, q in (("C", 0.0), ("P", 0.02)):
        m = DoubleHeston(*args, option_type=opt, q=q)
        got = m.implied_volatility()
        c = dhj.default_context()
        price = c.price_list(m._params(), 100.0, [95.0], [0.5], [opt == "C"], 0.03, q)
        want = c.implied_vol(price, 100.0, [95.0], [0.5], [opt == "C"], 0.03, q)[0, 0]
        assert got == want and 0.05 < got < 1.0
        assert isinstance(got, np.float64)
    m = DoubleHeston(*args, q=0.0)
    m.K = -1.0
    assert np.isnan(m.implied_volatility())


def test_launch_count(ctx):
    K5, T5 = np.tile(O.GENERATOR_STRIKES_REL, 3), np.repeat(O.GENERATOR_MATURITIES, 5)
    V = ctx.price_list(_params(100, 1), 100.0, K5, T5, True, 0.03)
    n0 = ctx.launch_count
    ctx.implied_vol(V, 100.0, K5, T5, True, 0.03)
    assert ctx.launch_count == n0 + 1
    ctx.bs_price(np.full_like(V, 0.2), 100.0, K5, T5, True, 0.03)
    assert ctx.launch_count == n0 + 2
