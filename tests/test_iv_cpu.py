"""Implied volatility on the CPU: the mpmath reference (tests/iv_oracle.py) against scipy, and the device arithmetic of
dhj_iv.cuh, compiled by g++ (tests/host_emu/emu_iv.cpp), against the reference: the normalised Black price b in
every evaluation region, the round-trip accuracy contract, every status code and the iteration count."""
import ctypes
import os
import subprocess

import mpmath as mp
import numpy as np
import pytest
from numpy.ctypeslib import ndpointer

import iv_oracle as IV
from conftest import PKG, ROOT

EPS = IV.EPS
C_BOUND = 7.0       # domain A, 4 096 points: measured max c 3.10, median 0.44 (DESIGN.md §6d)

_F = ndpointer(np.float64, flags="C_CONTIGUOUS")
_I = ndpointer(np.int32, flags="C_CONTIGUOUS")


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("emu_iv") / "emu_iv.so")
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I", os.path.join(PKG, "csrc"), "-o", out,
                    os.path.join(ROOT, "tests", "host_emu", "emu_iv.cpp")], check=True)
    lib = ctypes.CDLL(out)
    lib.emu_implied_vol.argtypes = [ctypes.c_int64] + [_F] * 6 + [_I, _F, _I, _I]
    lib.emu_bs_price.argtypes = [ctypes.c_int64] + [_F] * 6 + [_I, _F]
    lib.emu_b.argtypes = [ctypes.c_int64] + [_F] * 6
    lib.emu_erfcx.argtypes = [ctypes.c_double]
    lib.emu_erfcx.restype = ctypes.c_double
    return lib


def _arr(v, n, dtype=np.float64):
    return np.ascontiguousarray(np.broadcast_to(np.asarray(v, dtype=dtype), (n,)))


def implied_vol(lib, V, S0, K, T, r, q, call):
    n = np.broadcast(V, S0, K, T, r, q, call).size
    out, st, it = np.empty(n), np.empty(n, np.int32), np.empty(n, np.int32)
    lib.emu_implied_vol(n, _arr(V, n), _arr(S0, n), _arr(K, n), _arr(T, n), _arr(r, n), _arr(q, n),
                        _arr(call, n, np.int32), out, st, it)
    return out, st, it


@pytest.fixture(scope="module")
def domain_a():
    return IV.domain_a(4096, seed=11)


def test_reference_against_scipy():
    """The mpmath price agrees with a float64 scipy.stats.norm price where the latter is well conditioned
    (out-of-the-money parts above 1e-3 of the spot)."""
    from scipy.stats import norm
    rng = np.random.default_rng(3)
    for _ in range(200):
        S0, T, r, q = 100.0, rng.uniform(0.1, 3), rng.uniform(0, 0.08), rng.uniform(0, 0.03)
        K, sigma, call = rng.uniform(70, 130), rng.uniform(0.1, 0.8), bool(rng.integers(0, 2))
        F, D = S0 * np.exp((r - q) * T), np.exp(-r * T)
        s = sigma * np.sqrt(T)
        d1 = (np.log(F / K) + s * s / 2) / s
        want = D * (F * norm.cdf(d1) - K * norm.cdf(d1 - s)) if call else D * (K * norm.cdf(s - d1) - F * norm.cdf(-d1))
        got = float(IV.bs_price(S0, K, T, r, q, sigma, call))
        assert abs(got - want) <= 1e-12 * S0, (got, want)
        h = 1e-7
        fd = float((IV.bs_price(S0, K, T, r, q, sigma + h, call) - IV.bs_price(S0, K, T, r, q, sigma - h, call)) / (2 * h))
        assert abs(fd - float(IV.bs_vega(S0, K, T, r, q, sigma))) <= 1e-6 * S0
        star = IV.implied_vol(got, S0, K, T, r, q, call, 0.5)
        assert abs(float(star) - sigma) <= 1e-13


def test_emulated_erfcx(emu):
    """The emulation's erfcx (long double, asymptotic series beyond 100) against mpmath on [-26, 1e4]."""
    zs = np.concatenate([np.linspace(-26, 30, 400), np.geomspace(30, 1e4, 100)])
    for z in zs:
        want = mp.exp(mp.mpf(z) ** 2) * mp.erfc(mp.mpf(z))
        assert abs(emu.emu_erfcx(float(z)) - float(want)) <= 4 * EPS * float(want), z


def _b_mp(x, s):
    x, s = mp.mpf(float(x)), mp.mpf(float(s))
    N = lambda z: mp.erfc(-z / mp.sqrt(2)) / 2  # noqa: E731
    return mp.exp(x / 2) * N(x / s + s / 2) - mp.exp(-x / 2) * N(x / s - s / 2)


def test_b_every_region(emu):
    """b(x, s) for x <= 0 against 40-digit mpmath, s log-uniform on [5e-4, 20], h = x/s uniform on [-8, 0]: every
    region of b_norm (series below s = 0.5, erfcx difference, erfc form at h + t >= 5) is within (8 + 2 (h^2 + t^2)) eps,
    the growth being that of e^{-(h^2+t^2)/2} itself (the implied vol's sensitivity grows alike, ~h^2; near the upper
    bound, where t^2 matters, the solver works on the complement, checked to 64 eps).  The plain
    erfcx difference alone loses ~|h|/s eps at small s: above 1000 eps below s = 1e-2 (why the series exists)."""
    rng = np.random.default_rng(5)
    n = 6000
    s = np.exp(rng.uniform(np.log(5e-4), np.log(20.0), n))
    h = -rng.uniform(0.0, 8.0, n)
    x = h * s
    b, series, plain, comp = (np.empty(n) for _ in range(4))
    emu.emu_b(n, x, s, b, series, plain, comp)
    ref = np.array([float(_b_mp(a, c)) for a, c in zip(x, s)])
    err = np.abs(b - ref) / ref / EPS
    bound = 8 + 2 * (h * h + s * s / 4)
    worst = np.argmax(err / bound)
    assert (err <= bound).all(), (err[worst], s[worst], h[worst])
    t = s / 2
    for name, m in (("series", s < 0.5), ("erfcx", (s >= 0.5) & (h + t < 5)), ("erfc", (s >= 0.5) & (h + t >= 5))):
        assert m.sum() > 100, name
    small = s < 1e-2
    assert (np.abs(plain[small] - ref[small]) / ref[small] / EPS).max() > 1000
    up = h + t >= 0
    cref = np.array([float(mp.exp(mp.mpf(float(a)) / 2) - _b_mp(a, c)) for a, c in zip(x[up], s[up])])
    assert (np.abs(comp[up] - cref) / cref / EPS <= 64).all()


def test_domain_a_contract(emu, domain_a):
    """Round trip on domain A: every point has status 0 and c <= C_BOUND (module constant, ~2x the measured max)."""
    d = domain_a
    vol, st, it = implied_vol(emu, d["V"], d["S0"], d["K"], d["T"], d["r"], d["q"], d["call"])
    assert (st == 0).all()
    c = np.array([IV.c_measure(v, *(d[k][i] for k in ("V", "S0", "K", "T", "r", "q", "call", "sigma")))[0]
                  for i, v in enumerate(vol)])
    assert c.max() <= C_BOUND, (c.max(), np.median(c))
    assert np.median(c) <= 1.0


def test_iterations_below_cap(emu, domain_a):
    """The solver's evaluation count on domain A and on a wider stress set (sigma down to 1e-3 and up to 10, T up to
    30 years, |z| up to 12) stays far from the cap of 40."""
    d = domain_a
    _, st, it = implied_vol(emu, d["V"], d["S0"], d["K"], d["T"], d["r"], d["q"], d["call"])
    assert it.max() <= 10, np.bincount(it)
    rng = np.random.default_rng(9)
    n = 20000
    sigma = np.exp(rng.uniform(np.log(1e-3), np.log(10.0), n))
    T = np.exp(rng.uniform(np.log(1 / 365), np.log(30.0), n))
    z = rng.uniform(-12, 12, n)
    call = rng.integers(0, 2, n).astype(np.int32)
    K = 100.0 * np.exp(0.02 * T - z * sigma * np.sqrt(T))
    V = np.empty(n)
    emu.emu_bs_price(n, sigma, _arr(100.0, n), K, T, _arr(0.03, n), _arr(0.01, n), call, V)
    vol, st, it = implied_vol(emu, V, 100.0, K, T, 0.03, 0.01, call)
    # 1 / 2: a float64 price whose time value is below its rounding, or that rounds to the upper bound
    assert set(np.unique(st)) <= {0, 1, 2}
    assert it.max() <= 16, np.bincount(it)


def test_status_codes(emu):
    S0, K, T, r, q = 100.0, 90.0, 0.5, 0.03, 0.01
    Sq, KD = S0 * np.exp(-q * T), K * np.exp(-r * T)
    lb = Sq - KD
    cases = [  # (V, S0, K, T, r, q, call, status, vol)
        (lb, S0, K, T, r, q, 1, 0, 0.0),                               # at the lower bound: sigma = 0
        (0.0, S0, 120.0, T, r, q, 1, 0, 0.0),                          # out of the money at zero
        (np.nextafter(lb, 0), S0, K, T, r, q, 1, 1, np.nan),           # just below intrinsic
        (-1e-300, S0, 120.0, T, r, q, 1, 1, np.nan),
        (Sq, S0, K, T, r, q, 1, 2, np.nan),                            # at the call's upper bound
        (KD * 1.5, S0, K, T, r, q, 0, 2, np.nan),                      # above the put's upper bound
        (np.nan, S0, K, T, r, q, 1, 3, np.nan),
        (np.inf, S0, K, T, r, q, 1, 3, np.nan),
        (5.0, S0, 0.0, T, r, q, 1, 3, np.nan),                         # K <= 0
        (5.0, S0, K, -1.0, r, q, 1, 3, np.nan),                        # T <= 0
        (5.0, 0.0, K, T, r, q, 1, 3, np.nan),                          # S0 <= 0
        (5.0, S0, K, T, np.nan, q, 1, 3, np.nan),
        (5.0, S0, K, T, r, np.inf, 0, 3, np.nan),
    ]
    for V, s0, k, t, rr, qq, call, want_st, want_vol in cases:
        vol, st, _ = implied_vol(emu, V, s0, k, t, rr, qq, call)
        assert st[0] == want_st, (V, s0, k, t, rr, qq, call, st[0])
        if np.isnan(want_vol):
            assert np.isnan(vol[0])
        else:
            assert vol[0] == want_vol
    # the status-4 path: not reachable from a valid price (see test_iterations_below_cap); the code is reported in
    # IV_STATUS and include/dhj.h


def test_bs_price_forward_map(emu):
    """The emulated forward map against the mpmath price: within (8 + 1.5 z^2) eps of V + sigma * vega (rounding of the
    inputs to b moves the price by at most ~eps * sigma * vega), sigma = 0 gives the intrinsic value, bad input NaN."""
    d = IV.domain_a(600, seed=4)
    n = d["V"].size
    got = np.empty(n)
    emu.emu_bs_price(n, d["sigma"], d["S0"], d["K"], d["T"], d["r"], d["q"], d["call"], got)
    for i in range(n):
        a = [d[k][i] for k in ("S0", "K", "T", "r", "q")]
        vega = float(IV.bs_vega(*a, d["sigma"][i]))
        tol = 16 * EPS * (d["V"][i] + d["sigma"][i] * vega)
        assert abs(got[i] - d["V"][i]) <= tol, i
    out = np.empty(3)
    emu.emu_bs_price(3, np.array([0.0, -0.1, np.nan]), _arr(100.0, 3), _arr(90.0, 3), _arr(1.0, 3), _arr(0.0, 3),
                     _arr(0.0, 3), _arr(1, 3, np.int32), out)
    assert out[0] == 10.0 and np.isnan(out[1:]).all()
