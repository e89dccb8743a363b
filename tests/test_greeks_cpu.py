"""The Greeks on the CPU: the oracle (tests/greeks_oracle.py) against Richardson-extrapolated differences of the
reference prices, the put-call identities, and the device arithmetic (dhj_math.cuh's cf_exponent_time, walked in
k_price_greeks's order by tests/host_emu/emu_greeks.cpp) against the oracle."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
from numpy.ctypeslib import ndpointer

import greeks_oracle as G
import jac_oracle as J
from conftest import PKG, ROOT
from oracle import cos_oracle as O

EMU_DIR = os.path.join(ROOT, "tests", "host_emu")


def _params(n, seed=2):
    rng = np.random.default_rng(seed)
    lo, hi = O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1]
    return lo + (hi - lo) * rng.random((n, 13))


def _cases():
    """(name, params, S0, K, T, call, r, q): the generator grid with calls and puts and a dividend yield, the ragged
    market of loss_cases.npz (K 80-120, T 0.25-1.5, no binding strike), and the C3 edge strikes (binding widening)."""
    g = np.load(os.path.join(ROOT, "tests", "golden", "loss_cases.npz"))
    params = _params(8)
    K5, T5 = np.tile(O.GENERATOR_STRIKES_REL, 3), np.repeat(O.GENERATOR_MATURITIES, 5)
    Ke, Te = np.linspace(50.0, 150.0, 6), np.array([0.02, 0.25, 2.0])
    return [("grid_mixed", params, 100.0, K5, T5, np.arange(15) % 2 == 0, 0.03, 0.01),
            ("ragged", params, float(g["ragged_spot"]), g["ragged_strike"], g["ragged_maturity"],
             g["ragged_is_call"].astype(bool), float(g["ragged_r"]), 0.0),
            ("edge", params[:4], 100.0, np.tile(Ke, 3), np.repeat(Te, 6), np.arange(18) % 3 != 0, 0.03, 0.0)]


def _richardson(f, x0, h):
    """d f / dx at x0 by central differences at h, 2h, 4h with two Richardson steps (error O(h^6))."""
    d = [(f(x0 + m * h) - f(x0 - m * h)) / (2 * m * h) for m in (1, 2, 4)]
    r1, r2 = (4 * d[0] - d[1]) / 3, (4 * d[1] - d[2]) / 3
    return (16 * r1 - r2) / 15


def _col_err(got, want):
    return (np.abs(got - want) / np.abs(want).max(axis=1, keepdims=True)).max()


@pytest.mark.parametrize("case", range(2))
def test_oracle_delta_gamma_vs_full_differences(case):
    """Delta and gamma against differences in S0 of the FULL reference price on strikes whose widening does not bind:
    [a, b] does not move with S0 there, so the frozen-range derivative is the derivative of the price itself.
    Delta <= 1e-8 of its column scale (measured 6e-9).  Gamma is a second difference: measured 1e-6 of its scale on
    these inputs (Richardson over h = 1, 2), pinned at 1e-5."""
    name, params, S0, K, T, call, r, q = _cases()[case]
    assert not G.binding(params, S0, K, T, r).any()
    prices, greeks = G.greeks_batch(params, S0, K, T, call, r, q)
    full = lambda s: O.price_batch(params, s, K, T, call, r, q)
    assert np.abs(prices - full(S0)).max() <= 1e-11 * S0
    assert _col_err(_richardson(full, S0, 0.01 * S0), greeks[..., 0]) <= 1e-8, name
    d2 = [(full(S0 + h) - 2 * full(S0) + full(S0 - h)) / h ** 2 for h in (0.01 * S0, 0.02 * S0)]
    assert _col_err((4 * d2[0] - d2[1]) / 3, greeks[..., 1]) <= 1e-5, name


@pytest.mark.parametrize("case", range(3))
def test_oracle_time_rate_vs_frozen_differences(case):
    """Theta, rho and rho_q against differences of the frozen-range price in T, r and q: <= 1e-8 of scale."""
    name, params, S0, K, T, call, r, q = _cases()[case]
    _, greeks = G.greeks_batch(params, S0, K, T, call, r, q)
    _, ab = O.price_batch(params, S0, K, T, call, r, q, return_ab=True)
    frozen = lambda TT=T, rr=r, qq=q: J.price_batch_frozen(params, S0, K, TT, call, rr, ab, q=qq)
    M = len(T)
    dT = np.stack([_richardson(lambda t: frozen(TT=np.where(np.arange(M) == j, t, T))[:, j], T[j], 1e-3 * T[j])
                   for j in range(M)], axis=1)
    assert _col_err(-dT, greeks[..., 2]) <= 1e-8, name
    assert _col_err(_richardson(lambda x: frozen(rr=x), r, 1e-3), greeks[..., 3]) <= 1e-8, name
    assert _col_err(_richardson(lambda x: frozen(qq=x), q, 1e-3), greeks[..., 4]) <= 1e-8, name
    prices = frozen()
    assert np.abs(greeks[..., 4] + greeks[..., 3] + T * prices).max() <= 1e-12 * S0 * T.max()


def test_oracle_time_rate_vs_full_differences():
    """Theta and rho against central differences of the full reference price, whose [a, b] moves with T and r, on the
    ragged market: the difference (frozen-range term plus difference error) was measured at 2.3e-6 of the column scale
    at h = 1e-3; pinned at the Jacobian tests' 2e-5."""
    name, params, S0, K, T, call, r, q = _cases()[1]
    _, greeks = G.greeks_batch(params, S0, K, T, call, r, q)
    full = lambda TT=T, rr=r: O.price_batch(params, S0, K, TT, call, rr, q)
    h, M = 1e-3, len(T)
    dT = np.stack([(full(TT=np.where(np.arange(M) == j, T[j] + h, T))[:, j]
                    - full(TT=np.where(np.arange(M) == j, T[j] - h, T))[:, j]) / (2 * h) for j in range(M)], axis=1)
    assert _col_err(-dT, greeks[..., 2]) <= 2e-5
    assert _col_err((full(rr=r + h) - full(rr=r - h)) / (2 * h), greeks[..., 3]) <= 2e-5


@pytest.mark.parametrize("case", range(3))
def test_oracle_put_call_identities(case):
    """gamma_call == gamma_put; delta and rho of call minus put against the derivatives of the parity
    C - P = S0 e^{-qT} - K e^{-rT}.  The truncated series has its own parity residual: measured at most 1.9e-10 S0 on
    the first two cases (N = 128, L = 10) and pinned at 1e-9 S0; the Greek identities inherit it (delta 1.9e-10, rho
    2.1e-9 of its scale), pinned at 1e-9 and 1e-8.  The edge case's binding strikes and T = 0.02 are not held to it."""
    name, params, S0, K, T, call, r, q = _cases()[case]
    q = 0.01
    Vc, gc = G.greeks_batch(params, S0, K, T, True, r, q)
    Vp, gp = G.greeks_batch(params, S0, K, T, False, r, q)
    assert np.array_equal(gc[..., 1], gp[..., 1])
    if name == "edge":
        return
    resid = Vc - Vp - (S0 * np.exp(-q * T) - K * np.exp(-r * T))
    assert np.abs(resid).max() <= 1e-9 * S0
    assert np.abs(gc[..., 0] - gp[..., 0] - np.exp(-q * T)).max() <= 1e-9
    assert np.abs(gc[..., 3] - gp[..., 3] - K * T * np.exp(-r * T)).max() <= 1e-8 * np.abs(gc[..., 3]).max()


@pytest.fixture(scope="module")
def emu_greeks():
    out = os.path.join(EMU_DIR, "_build", "libdhj_emu_greeks.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I", os.path.join(PKG, "csrc"),
                    "-x", "c++", os.path.join(EMU_DIR, "emu_greeks.cpp"), "-o", out], check=True)
    lib = ctypes.CDLL(out)
    D, I = ndpointer(np.float64, flags="C"), ndpointer(np.int32, flags="C")
    lib.emu_price_greeks.argtypes = [D, D, D, D, I, ctypes.c_double, ctypes.c_double, ctypes.c_long, ctypes.c_int,
                                     ctypes.c_int, ctypes.c_double, D, D]

    def run(params, S0, K, T, call, r, q, N=128):
        params = np.ascontiguousarray(params, dtype=np.float64).reshape(-1, 13)
        P, M = len(params), len(T)
        prices, greeks = np.empty((P, M)), np.empty((P, M, 5))
        lib.emu_price_greeks(params, np.full(P, float(S0)), np.ascontiguousarray(np.tile(K, (P, 1)), dtype=np.float64),
                             np.ascontiguousarray(T, dtype=np.float64), np.asarray(call).astype(np.int32), r, q, P, M,
                             N, 10.0, prices, greeks)
        return prices, greeks
    return run


@pytest.mark.parametrize("N", [128, 256, 100])
@pytest.mark.parametrize("case", range(3))
def test_emulated_device_greeks(emu_greeks, case, N):
    """Device arithmetic against the oracle: <= 1e-10 of each Greek's column scale, the Jacobian emulation's bound."""
    name, params, S0, K, T, call, r, q = _cases()[case]
    prices, greeks = emu_greeks(params, S0, K, T, call, r, q, N)
    want_p, want_g = G.greeks_batch(params, S0, K, T, call, r, q, N=N)
    scale = np.abs(want_g).max(axis=1, keepdims=True)
    err = (np.abs(greeks - want_g) / scale).max(axis=(0, 1))
    assert err.max() <= 1e-10, (name, dict(zip(G.GREEKS, err)))
    assert np.abs(prices - want_p).max() <= 1e-11 * S0
