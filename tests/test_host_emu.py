"""Checks the kernel ARITHMETIC (option-pricing-ffn-lbfgs_b200/csrc/dhj_math.cuh) on the CPU: the header is
compiled with g++ into a test-only emulation (tests/host_emu/emu.cpp) that walks k in the kernel's lane
order, and compared with the reference's golden values.  This keeps algebra mistakes out of GPU time; it is
not a product path (nothing under the package loads it) and it differs from the device only in libm."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
from numpy.ctypeslib import ndpointer

from conftest import PKG, ROOT, rel_err

EMU_DIR = os.path.join(ROOT, "tests", "host_emu")
WALKS = ("r01", "batch", "dense")


@pytest.fixture(scope="module")
def emu():
    out = os.path.join(EMU_DIR, "_build", "libdhj_emu.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I", os.path.join(PKG, "csrc"),
                    "-x", "c++", os.path.join(EMU_DIR, "emu.cpp"), "-o", out], check=True)
    lib = ctypes.CDLL(out)
    D, I = ndpointer(np.float64, flags="C"), ndpointer(np.int32, flags="C")
    lib.emu_price_list.argtypes = [D, D, ctypes.c_int, D, ctypes.c_int, D, I, ctypes.c_double, ctypes.c_double,
                                   ctypes.c_long, ctypes.c_int, ctypes.c_int, ctypes.c_double, D, D]
    lib.emu_loss.argtypes = [D, ctypes.c_long, ctypes.c_double, ctypes.c_double, D, D, I, D, ctypes.c_int,
                             ctypes.c_int, D]

    def price_list(params, S0, strike, mat, call, r, q=0.0, N=128, L=10.0):
        params = np.ascontiguousarray(params, dtype=np.float64).reshape(-1, 13)
        P = len(params)
        S0 = np.ascontiguousarray(np.broadcast_to(np.asarray(S0, dtype=np.float64), (P,)))
        mat = np.ascontiguousarray(mat, dtype=np.float64)
        M = len(mat)
        strike = np.ascontiguousarray(np.broadcast_to(np.asarray(strike, dtype=np.float64), (P, M)))
        call = np.ascontiguousarray(np.broadcast_to(np.asarray(call), (M,)).astype(np.int32))
        out, ab = np.empty((P, M)), np.empty((P, M, 2))
        lib.emu_price_list(params, S0, 1, strike, M, mat, call, r, q, P, M, N, L, out, ab)
        return out, ab

    U8 = ndpointer(np.uint8, flags="C")
    lib.emu_price_walk.argtypes = [ctypes.c_int, D, D, D, D, I, ctypes.c_double, ctypes.c_double, ctypes.c_long,
                                   ctypes.c_int, ctypes.c_int, ctypes.c_double, D, U8]

    def price_walk(walk, params, S0, strike, mat, call, r, q=0.0, N=128, L=10.0):
        """(prices[P, M], binding[P, M]) in the order of walk "r01", "batch" or "dense"."""
        params = np.ascontiguousarray(params, dtype=np.float64).reshape(-1, 13)
        P, M = len(params), len(mat)
        S0 = np.ascontiguousarray(np.broadcast_to(np.asarray(S0, dtype=np.float64), (P,)))
        strike = np.ascontiguousarray(np.broadcast_to(np.asarray(strike, dtype=np.float64), (P, M)))
        call = np.ascontiguousarray(np.broadcast_to(np.asarray(call), (M,)).astype(np.int32))
        out, bind = np.empty((P, M)), np.empty((P, M), dtype=np.uint8)
        lib.emu_price_walk(WALKS.index(walk), params, S0, strike, np.ascontiguousarray(mat, dtype=np.float64), call,
                           r, q, P, M, N, L, out, bind)
        return out, bind.astype(bool)

    def loss(x, S0, r, strike, mat, call, market, N=128):
        x = np.ascontiguousarray(x, dtype=np.float64).reshape(-1, 13)
        out = np.empty(len(x))
        lib.emu_loss(x, len(x), S0, r, np.ascontiguousarray(strike, dtype=np.float64),
                     np.ascontiguousarray(mat, dtype=np.float64),
                     np.ascontiguousarray(np.asarray(call).astype(np.int32)),
                     np.ascontiguousarray(market, dtype=np.float64), len(mat), N, out)
        return out

    price_list.walk = price_walk
    return price_list, loss


def test_emu_grid15(emu, golden):
    price_list, _ = emu
    g = golden("prices_grid15.npz")
    K = np.tile(g["k_rel"][None, :] * g["spots"][:, None] / 100.0, (1, 3))
    T = np.repeat(g["maturities"], 5)
    got, ab = price_list(g["params"], g["spots"], K, T, np.ones(15), float(g["r"]))
    err = rel_err(got.reshape(150, 3, 5), g["prices"])
    assert err.max() <= 1e-12 and np.median(err) <= 5e-14
    assert np.abs(ab.reshape(150, 3, 5, 2) - g["ab"]).max() <= 4e-15


@pytest.mark.parametrize("tag", ["main", "edge"])
def test_emu_dense(emu, golden, tag):
    price_list, _ = emu
    g = golden("dense_surface.npz")
    Ks, Ts = g[f"{tag}_strikes"], g[f"{tag}_maturities"]
    K = np.tile(Ks, len(Ts)); T = np.repeat(Ts, len(Ks))
    got, _ = price_list(g["params"], 100.0, K, T, np.ones(K.size), float(g["r"]), N=256)
    want = g[f"{tag}_prices"].reshape(4, -1)
    assert (np.abs(got - want) / 100.0).max() <= 2e-13


def test_emu_edge_cases(emu, golden):
    price_list, _ = emu
    g = golden("edge_cases.npz")
    for i in range(len(g["prices"])):
        S0, K, T, r, q, call, N = g["meta"][i]
        got = price_list(g["params"][i], S0, [K], [T], [int(call)], r, q, int(N))[0][0, 0]
        want = g["prices"][i]
        if np.isnan(want):
            assert np.isnan(got)
        elif g["params"][i][3] <= 1e-3:
            assert abs(got - want) <= 1e-3 * want           # sigma -> 0: the reference itself cancels (DESIGN §4)
        else:
            scale = max(S0, K) * max(1.0, np.exp(g["ab"][i][1]))
            assert abs(got - want) <= 1e-10 * abs(want) or abs(got - want) <= 4e-14 * scale, i


def test_emu_loss(emu, golden):
    _, loss = emu
    g = golden("loss_cases.npz")
    for tag in ("c1", "ragged"):
        got = loss(g[f"{tag}_x"], float(g[f"{tag}_spot"]), float(g[f"{tag}_r"]), g[f"{tag}_strike"],
                   g[f"{tag}_maturity"], g[f"{tag}_is_call"], g[f"{tag}_market"])
        want = g[f"{tag}_loss"]
        assert np.array_equal(got == 1e10, want == 1e10)
        assert (np.abs(got - want) <= 1e-9 * np.maximum(1.0, np.abs(want))).all()


# ---- the current kernels' orders (k_price_batch, k_price_dense) on families b and c of test_gpu_price_edges ----------
@pytest.mark.parametrize("walk", ["batch", "dense"])
@pytest.mark.parametrize("N", [2, 33, 256, 257, 1000, 2048])
def test_emu_walks_binding_positions(emu, walk, N):
    """Binding strikes at every position of 8-strike slices (their own pass, (a, b) and jump recurrences) through
    both kernels' orders, against the C oracle at the GPU test's bounds; the emulation finds the same binding
    strikes as the oracle."""
    from test_gpu_price_edges import _batch_binding_list, _check
    params, K, T, call, mask = _batch_binding_list()
    got, bind = emu[0].walk(walk, params, 100.0, K, T, call, 0.03, 0.01, N)
    assert (bind == mask).all()
    _check(f"emulated {walk} walk, binding positions N={N}", got, params, 100.0, K, T, call, 0.03, 0.01, N)


@pytest.mark.parametrize("walk", ["batch", "dense"])
@pytest.mark.parametrize("N", [255, 256, 257, 512, 1000, 2048])
def test_emu_walks_recurrence_family(emu, walk, N):
    """Low-diffusion, jump-dominated sets whose blocks beyond k = 256 carry weight: the jump term's rotation and
    Gaussian ratio and the segment starts' rotation between the exact blocks, against the C oracle."""
    from test_gpu_price_edges import REC_STRIKES, _check, _rec_case
    params, K, T, call, mask = _rec_case(REC_STRIKES[walk])
    got, bind = emu[0].walk(walk, params, 100.0, K, T, call, 0.03, 0.0, N)
    assert (bind == mask).all()
    _check(f"emulated {walk} walk, recurrence family N={N}", got, params, 100.0, K, T, call, 0.03, 0.0, N)


def test_emu_walks_agree_with_r01_order(emu):
    """The three orders price the C2 grid alike to 1e-12 relative (the arithmetic is the same up to summation order
    and the recurrences)."""
    from test_gpu_derivative_edges import _params
    params = _params(20, 27)
    K, T = np.tile(np.linspace(90.0, 110.0, 5), 3), np.repeat([0.25, 0.5, 1.0], 5)
    ref, _ = emu[0].walk("r01", params, 100.0, K, T, np.arange(15) % 2 == 0, 0.03)
    for walk in ("batch", "dense"):
        got, _ = emu[0].walk(walk, params, 100.0, K, T, np.arange(15) % 2 == 0, 0.03)
        assert rel_err(got, ref).max() <= 1e-12, walk
