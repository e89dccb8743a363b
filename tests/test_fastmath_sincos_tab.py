"""Accuracy of fm::sincos_tab / fm::cos_tab (dhj_fastmath.cuh), the table-driven sincos of the pricing engine's
characteristic function and payoff cosine, compiled for the host, against mpmath at 40 digits.  The arguments are
those the engine produces: the payoff angle xi - u a with |u a| <= N pi |a| / (b - a) and |xi| of the same order,
the E_j angle -Im(d_j) T and the contraction's segment starts k theta, up to a few thousand for N <= 1024."""
import ctypes
import os
import subprocess

import mpmath as mp
import numpy as np
import pytest
from numpy.ctypeslib import ndpointer

from conftest import PKG, ROOT

mp.mp.dps = 40


@pytest.fixture(scope="module")
def lib():
    d = os.path.join(ROOT, "tests", "host_emu")
    out = os.path.join(d, "_build", "libsincos_tab_emu.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-mfma", "-fPIC", "-shared", "-I", os.path.join(PKG, "csrc"),
                    "-x", "c++", os.path.join(d, "sincos_tab_emu.cpp"), "-o", out], check=True)
    lib = ctypes.CDLL(out)
    D = ndpointer(np.float64, flags="C")
    lib.fm_sincos_tab.argtypes = [D, ctypes.c_int, D, D]
    lib.fm_cos_tab.argtypes = [D, ctypes.c_int, D]
    return lib


def ulp_err(got, exact):
    """|got - exact| in ulps of exact (exact: list of mpf)."""
    out = np.empty(len(got))
    for i, (g, e) in enumerate(zip(got, exact)):
        out[i] = float(abs(mp.mpf(float(g)) - e) / mp.mpf(float(np.spacing(abs(float(e))))))
    return out


def _eval(lib, x):
    x = np.ascontiguousarray(x, dtype=np.float64)
    s, c, c2 = np.empty_like(x), np.empty_like(x), np.empty_like(x)
    lib.fm_sincos_tab(x, x.size, s, c)
    lib.fm_cos_tab(x, x.size, c2)
    return s, c, c2


def test_sincos_tab_accuracy(lib):
    rng = np.random.default_rng(11)
    x = np.concatenate([rng.uniform(-4000, 4000, 4000), rng.uniform(-300, 300, 3000), rng.uniform(-0.05, 0.05, 1000),
                        rng.uniform(-1e5, 1e5, 500),
                        np.arange(-256, 257) * (np.pi / 256),                    # table nodes
                        (np.arange(-256, 256) + 0.5) * (np.pi / 256),            # interval ends |r| = pi/512
                        [0.0, -0.0, 1e-300, np.pi / 2, np.pi, 100 * np.pi]])
    s, c, c2 = _eval(lib, x)
    ms = [mp.mpf(float(v)) for v in x]
    es, ec = ulp_err(s, [mp.sin(v) for v in ms]), ulp_err(c, [mp.cos(v) for v in ms])
    # <= 1.5 ulp; up to 2 where the result lies a binade below its table entry (|result| < 2^-7: the entry's
    # rounding is then worth a whole ulp of the result); near zeros of sin / cos bound the error in absolute terms
    for e, v in ((es, s), (ec, c)):
        a = np.abs(v)
        assert e[a >= 2.0 ** -7].max() <= 1.5, e[a >= 2.0 ** -7].max()
        assert e[a > 1e-3].max() <= 2.0, e[a > 1e-3].max()
    assert np.abs(s - np.sin(x)).max() <= 3e-16 and np.abs(c - np.cos(x)).max() <= 3e-16
    assert np.array_equal(c, c2)                                  # cos_tab is sincos_tab's cosine, bit for bit
    assert s[-6] == 0.0 and c[-6] == 1.0


def test_sincos_tab_special(lib):
    s, c, c2 = _eval(lib, np.array([np.nan, np.inf, -np.inf]))
    assert np.isnan(s).all() and np.isnan(c).all() and np.isnan(c2).all()
