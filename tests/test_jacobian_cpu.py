"""The analytic parameter gradient on the CPU: the dual-number oracle (tests/jac_oracle.py) against difference
quotients of the reference prices, and the device arithmetic (dhj_math.cuh's cf_exponent_tangents, walked in
k_price_jac's order by tests/host_emu/emu_grad.cpp) against the oracle."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
from numpy.ctypeslib import ndpointer

import jac_oracle as J
from conftest import PKG, ROOT
from oracle import cos_oracle as O

EMU_DIR = os.path.join(ROOT, "tests", "host_emu")


def _cases():
    """(name, params, S0, K, T, call, r): generator-range sets on the C1 / C5 grid (calls, and calls and puts), and
    the C3 edge strikes (K 50-150, T from 0.02: binding widening)."""
    rng = np.random.default_rng(2)
    lo, hi = O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1]
    params = lo + (hi - lo) * rng.random((12, 13))
    K5, T5 = np.tile(O.GENERATOR_STRIKES_REL, 3), np.repeat(O.GENERATOR_MATURITIES, 5)
    Ke, Te = np.linspace(50.0, 150.0, 6), np.array([0.02, 0.25, 2.0])
    return [("c5_calls", params, 100.0, K5, T5, np.ones(15, bool), 0.03),
            ("c1_mixed", params[:6], 100.0, K5, T5, np.arange(15) % 2 == 1, 0.03),
            ("c3_edge", params[:6], 100.0, np.tile(Ke, 3), np.repeat(Te, 6), np.arange(18) % 3 != 0, 0.03)]


def _richardson(f, params, i, hrel):
    """d f / d params[:, i] by central differences at h, 2h, 4h with two Richardson steps (error O(h^6))."""
    h = hrel * np.abs(params[:, i])[:, None]
    d = []
    for m in (1, 2, 4):
        pp, pm = params.copy(), params.copy()
        pp[:, i] += m * h[:, 0]
        pm[:, i] -= m * h[:, 0]
        d.append((f(pp) - f(pm)) / (2 * m * h))
    r1, r2 = (4 * d[0] - d[1]) / 3, (4 * d[1] - d[2]) / 3
    return (16 * r1 - r2) / 15


@pytest.mark.parametrize("case", range(3))
def test_oracle_jacobian_vs_frozen_differences(case):
    name, params, S0, K, T, call, r = _cases()[case]
    prices, jac = J.price_jacobian_batch(params, S0, K, T, call, r)
    ref, ab = O.price_batch(params, S0, K, T, call, r, return_ab=True)
    assert np.abs(prices - ref).max() <= 1e-11 * S0
    frozen = lambda p: J.price_batch_frozen(p, S0, K, T, call, r, ab)
    assert np.array_equal(frozen(params), J.price_batch_frozen(params, S0, K, T, call, r, ab))
    for i in range(13):
        fd = _richardson(frozen, params, i, 1e-2)
        scale = np.abs(jac[:, :, i]).max(axis=1, keepdims=True)
        err = (np.abs(fd - jac[:, :, i]) / scale).max()
        assert err <= 1e-8, (name, O.PARAM_NAMES[i], err)


def test_oracle_jacobian_vs_unfrozen_differences():
    """The frozen-range Jacobian against differences of the full reference price (whose [a, b] moves with the
    parameters): the difference is below the difference quotients' own rounding noise (measured max 4.7e-6 of the
    column scale on 200 generator sets, 1.5e-6 on these), pinned with margin."""
    name, params, S0, K, T, call, r = _cases()[0]
    _, jac = J.price_jacobian_batch(params, S0, K, T, call, r)
    full = lambda p: O.price_batch(p, S0, K, T, call, r)
    for i in range(13):
        h = 1e-4 * np.abs(params[:, i])[:, None]
        pp, pm = params.copy(), params.copy()
        pp[:, i] += h[:, 0]
        pm[:, i] -= h[:, 0]
        cd = (full(pp) - full(pm)) / (2 * h)
        scale = np.abs(jac[:, :, i]).max(axis=1, keepdims=True)
        assert (np.abs(cd - jac[:, :, i]) / scale).max() <= 2e-5, O.PARAM_NAMES[i]


def _off_kink(x, margin=1e-3):
    """States whose difference quotients are meaningful: not an exact fit (g ~ 0, the quotient is noise) and no
    Feller excess within `margin` of its kink (a central difference there straddles the kink)."""
    p = O.transform_params(x)
    with np.errstate(all="ignore"):
        e = np.stack([p[:, 3] ** 2 - 2 * p[:, 1] * p[:, 2], p[:, 8] ** 2 - 2 * p[:, 6] * p[:, 7]], axis=1)
    return (np.abs(e) > margin).all(axis=1)


def _loss_inputs():
    g = np.load(os.path.join(ROOT, "tests", "golden", "loss_cases.npz"))
    x = g["c1_x"][:8].copy()
    p_lit = np.array([0.04, 2.5, 0.04, 0.3, -0.7, 0.04, 0.5, 0.04, 0.2, -0.5, 0.15, -0.04, 0.08])
    feller = O.inverse_transform_params(p_lit)
    feller[3] = np.log(0.6)                         # sigma1^2 - 2 kappa1 theta1 = 0.16 > 0
    feller[6] = np.log(0.6)                         # (the literature values sit exactly on factor 2's kink)
    bad = x[0].copy()
    bad[1] = np.nan
    x = np.vstack([x, feller, bad])
    return x, float(g["c1_spot"]), float(g["c1_r"]), g["c1_strike"], g["c1_maturity"], g["c1_is_call"], g["c1_market"]


def test_loss_grad_vs_differences():
    x, S0, r, K, T, call, mk = _loss_inputs()
    f, g = J.loss_grad_batch(x, S0, r, K, T, call, mk)
    want = O.loss_batch(x, S0, r, K, T, call, mk)
    assert np.array_equal(f == O.SENTINEL, want == O.SENTINEL) and f[-1] == O.SENTINEL and (g[-1] == 0).all()
    assert O.feller_penalty(O.transform_params(x[-2])) > 0
    ok = f != O.SENTINEL
    assert np.allclose(f[ok], want[ok], rtol=1e-12, atol=1e-24)     # (one row fits exactly: f ~ 1e-28)
    for c in np.flatnonzero(ok & (f > 1e-20) & _off_kink(x)):
        h = 1e-5
        pts = np.repeat(x[c][None, :], 26, axis=0)
        for i in range(13):
            pts[2 * i, i] += h
            pts[2 * i + 1, i] -= h
        fv = O.loss_batch(pts, S0, r, K, T, call, mk)
        cd = (fv[0::2] - fv[1::2]) / (2 * h)
        assert np.abs(cd - g[c]).max() <= 1e-6 * np.abs(g[c]).max(), c


@pytest.fixture(scope="module")
def emu_jac():
    out = os.path.join(EMU_DIR, "_build", "libdhj_emu_grad.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I", os.path.join(PKG, "csrc"),
                    "-x", "c++", os.path.join(EMU_DIR, "emu_grad.cpp"), "-o", out], check=True)
    lib = ctypes.CDLL(out)
    D, I = ndpointer(np.float64, flags="C"), ndpointer(np.int32, flags="C")
    lib.emu_price_jacobian.argtypes = [D, D, D, D, I, ctypes.c_double, ctypes.c_double, ctypes.c_long, ctypes.c_int,
                                       ctypes.c_int, ctypes.c_double, D, D]

    def run(params, S0, K, T, call, r, N=128, q=0.0, L=10.0):
        """S0 a scalar or [P], K [M] or [P, M] (per-set strike rows)."""
        params = np.ascontiguousarray(params, dtype=np.float64).reshape(-1, 13)
        P, M = len(params), len(T)
        prices, jac = np.empty((P, M)), np.empty((P, M, 13))
        S0 = np.ascontiguousarray(np.broadcast_to(np.asarray(S0, dtype=np.float64), (P,)))
        K = np.ascontiguousarray(np.broadcast_to(np.asarray(K, dtype=np.float64), (P, M)))
        lib.emu_price_jacobian(params, S0, K, np.ascontiguousarray(T, dtype=np.float64),
                               np.asarray(call).astype(np.int32), r, q, P, M, N, L, prices, jac)
        return prices, jac
    return run


def _emu_cases():
    """(name, params, S0, K, T, call, r, q, L): _cases() with q = 0 and L = 10; a 129-strike slice at T = 0.05 with
    K 40-160 (many binding strikes), calls and puts; per-set spots 80 / 100 / 130 with per-set strike rows (65
    strikes at T = 0.1, 13 at T = 1), r = 0.02, q = 0.015 and L = 8 or 12."""
    out = [c + (0.0, 10.0) for c in _cases()]
    rng = np.random.default_rng(3)
    lo, hi = O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1]
    params = lo + (hi - lo) * rng.random((3, 13))
    Kw = np.linspace(40.0, 160.0, 129)
    out.append(("wide129", params, 100.0, Kw, np.full(129, 0.05), np.arange(129) % 2 == 0, 0.03, 0.0, 10.0))
    S0 = np.array([80.0, 100.0, 130.0])
    Kp = S0[:, None] * np.linspace(0.6, 1.45, 65)[None, :] * (1 + 0.01 * rng.standard_normal((3, 65)))
    Kp = np.concatenate([Kp, Kp[:, ::5]], axis=1)
    Tp = np.concatenate([np.full(65, 0.1), np.full(13, 1.0)])
    for L in (8.0, 12.0):
        out.append((f"per_set_L{L:g}", params, S0, Kp, Tp, np.arange(78) % 2 == 1, 0.02, 0.015, L))
    return out


@pytest.mark.parametrize("N", [128, 256, 2, 33, 1000])
@pytest.mark.parametrize("case", range(6))
def test_emulated_device_jacobian(emu_jac, case, N):
    """Device arithmetic vs the oracle: <= 1e-10 of the column scale (measured worst 3.0e-11 for N >= 33, c5_calls),
    also at a one-block and ragged N, with binding strikes, per-set rows, q != 0 and L != 10."""
    name, params, S0, K, T, call, r, q, L = _emu_cases()[case]
    prices, jac = emu_jac(params, S0, K, T, call, r, N, q, L)
    want_p, want_j = J.price_jacobian_batch(params, S0, K, T, call, r, q, N=N, L=L, chunk=1)
    scale = np.abs(want_j).max(axis=1, keepdims=True)
    err = (np.abs(jac - want_j) / scale).max()
    print(f"{name} N={N}: worst |jac - oracle| / column scale {err:.2e}")
    # at N = 2 the series has two terms: a column's largest entry falls up to 9x below its N = 128 value while the
    # rounding of a deep in-the-money binding strike's S0-sized terms does not (measured 1.6e-10 on wide129, sigma2
    # column, K = 45.6; every other case <= 7.8e-11)
    assert err <= (3e-10 if N == 2 else 1e-10), name
    assert np.abs(prices - want_p).max() <= 1e-11 * np.max(S0)
