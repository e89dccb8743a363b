"""Monte Carlo path scheme on the CPU: the device's stream, Box-Muller, Poisson inversion, path step and payoffs
(csrc/dhj_mc.cuh, compiled by g++ into tests/host_emu/emu_mc.cpp) against the NumPy restatement (tests/mc_oracle.py)
and scipy."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
from numpy.ctypeslib import ndpointer

import mc_oracle as MO
from conftest import PKG, ROOT

_F = ndpointer(np.float64, flags="C_CONTIGUOUS")
_I = ndpointer(np.int32, flags="C_CONTIGUOUS")
_U64 = ndpointer(np.uint64, flags="C_CONTIGUOUS")
_U32 = ndpointer(np.uint32, flags="C_CONTIGUOUS")
_i64, _i32, _f64, _u64 = ctypes.c_int64, ctypes.c_int32, ctypes.c_double, ctypes.c_uint64

# a typical set (inside the generator's box), a set that violates the Feller condition (2 kappa theta = 0.12 < sigma^2
# = 0.25: most paths truncate the variance) with frequent jumps, and a set without jumps.  Far deeper in the violation
# (sigma^2 / (2 kappa theta) ~ 70) the Euler map near v = 0 amplifies ulp-level differences of the normals from step
# to step and no two implementations agree to 1e-12 (DESIGN.md §6f); these sets stay clear of that.
SETS = np.array([
    [0.04, 2.0, 0.04, 0.3, -0.6, 0.03, 0.8, 0.05, 0.2, -0.4, 0.15, -0.05, 0.08],
    [0.02, 2.0, 0.03, 0.5, -0.8, 0.04, 1.0, 0.04, 0.25, -0.5, 1.0, -0.1, 0.15],
    [0.05, 3.0, 0.05, 0.4, -0.7, 0.02, 1.0, 0.03, 0.15, -0.3, 0.0, -0.05, 0.08],
])


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("emu_mc") / "emu_mc.so")
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I", os.path.join(PKG, "csrc"), "-o", out,
                    os.path.join(ROOT, "tests", "host_emu", "emu_mc.cpp")], check=True)
    lib = ctypes.CDLL(out)
    lib.emu_mc_words.argtypes = [_u64, _i64, _U64, _U32, _U64, _U64]
    lib.emu_box_muller.argtypes = [_i64, _U64, _U64, _F, _F]
    lib.emu_poisson_inverse.argtypes = [_i64, _F, _f64, _I]
    lib.emu_mc_paths.argtypes = [_F, _f64, _f64, _f64, _f64, _i32, _i32, _u64, _i64, _U64, _F]
    lib.emu_mc_payoff.argtypes = [_i64, _F, _i32, _i32, _i32, _f64, _f64, _F]
    return lib


def emu_paths(lib, p, S0, r, q, T, n_steps, n_obs, seed, paths):
    paths = np.ascontiguousarray(paths, dtype=np.uint64)
    out = np.empty((paths.size, 4))
    lib.emu_mc_paths(np.ascontiguousarray(p, dtype=np.float64), S0, r, q, T, n_steps, n_obs, seed, paths.size, paths,
                     out)
    return out


def test_stream_words_bit_identical(emu):
    """Philox words of the DHJ2 stream, including seeds and path indices at and above 2^32, and the counter word's
    high steps."""
    rng = np.random.default_rng(5)
    paths = np.concatenate([np.arange(8, dtype=np.uint64),
                            np.array([2**32 - 1, 2**32, 2**32 + 1, 2**63 + 12345, 2**64 - 1], dtype=np.uint64),
                            rng.integers(0, 2**63, 32, dtype=np.uint64)])
    for seed in (0, 1, 2**32 - 1, 2**32, 2**32 + 7, 0xDEADBEEFCAFEF00D, 2**64 - 1):
        for ctr in (0, 1, 2, 3, 4 * 251 + 3, 4 * (2**28 - 1) + 3):
            c = np.full(paths.size, ctr, dtype=np.uint32)
            w0, w1 = np.empty(paths.size, np.uint64), np.empty(paths.size, np.uint64)
            emu.emu_mc_words(seed, paths.size, paths, c, w0, w1)
            r0, r1 = MO.mc_words(seed, paths, ctr)
            assert np.array_equal(w0, r0) and np.array_equal(w1, r1), (seed, ctr)


def test_stream_tag_differs_from_generator():
    """The DHJ2 stream never shares a counter with the generator's DHJ1 stream: same (index, slot), other words."""
    from oracle.cos_oracle import counter_words
    idx = np.arange(16, dtype=np.uint64)
    a0, _ = counter_words(3, idx, 0)
    b0, _ = MO.mc_words(3, idx, 0)
    assert not np.any(a0 == b0)


def test_box_muller_matches_numpy(emu):
    """The library's Box-Muller (own log / sqrt / sincos) against NumPy's on the same words: <= 4 ulp of the radius."""
    rng = np.random.default_rng(9)
    w0 = rng.integers(0, 2**64, 4096, dtype=np.uint64)
    w1 = rng.integers(0, 2**64, 4096, dtype=np.uint64)
    w0[:3] = [0, 2**64 - 1, 2**11]
    z0, z1 = np.empty(w0.size), np.empty(w0.size)
    emu.emu_box_muller(w0.size, w0, w1, z0, z1)
    r0, r1 = MO.box_muller(w0, w1)
    R = np.hypot(r0, r1)                   # 0 for u1 = 1 (w0 = 2^64 - 1): both give exact zeros there
    assert np.all(np.abs(z0 - r0) <= 4 * 2.0 ** -52 * R)
    assert np.all(np.abs(z1 - r1) <= 4 * 2.0 ** -52 * R)


@pytest.mark.parametrize("lam_dt", [1e-4, 0.01, 0.5, 3.0])
def test_poisson_inversion_matches_scipy(emu, lam_dt):
    """N = smallest n with U < F(n) equals scipy's poisson.ppf away from the CDF's jumps (U within 1e-12 of a value of
    the CDF is left out), on a grid of U that includes the far tail."""
    from scipy.stats import poisson
    U = np.concatenate([np.linspace(0.0, 1.0, 20001)[1:-1], 1.0 - np.geomspace(1e-3, 1e-11, 200)])
    cdf = poisson.cdf(np.arange(0, 80), lam_dt)
    keep = np.min(np.abs(U[:, None] - cdf[None, :]), axis=1) > 1e-12
    U = np.ascontiguousarray(U[keep])
    got = np.empty(U.size, np.int32)
    emu.emu_poisson_inverse(U.size, U, lam_dt, got)
    want = poisson.ppf(U, lam_dt)
    assert np.array_equal(got, want.astype(np.int32))
    assert np.array_equal(got, MO.poisson_inverse(U, np.exp(-lam_dt), lam_dt))


def test_poisson_inversion_cap(emu):
    """The inversion stops at 64 jumps (documented cap), and a NaN intensity gives none."""
    got = np.empty(2, np.int32)
    emu.emu_poisson_inverse(2, np.array([0.999999, 0.5]), 200.0, got)
    assert got.tolist() == [64, 64]
    emu.emu_poisson_inverse(2, np.array([0.3, 0.9]), np.nan, got)
    assert got.tolist() == [0, 0]


@pytest.mark.parametrize("n_steps,n_obs", [(1, 1), (7, 7), (7, 1), (252, 252), (252, 12)])
def test_path_statistics_match_oracle(emu, n_steps, n_obs):
    """S_T, the sum, max and min at the observation dates of 64 paths x 3 sets agree to 1e-12 relative, with the
    same number of jumps on every step; the truncating set really truncates and the jump set really jumps."""
    paths = np.concatenate([np.arange(60, dtype=np.uint64), np.array([2**32, 2**32 + 1, 2**40 + 3, 2**63], np.uint64)])
    seed = 2**32 + 11
    S0, r, q, T = 100.0, 0.03, 0.01, 1.0
    d = MO.draws(seed, paths, n_steps)
    for p in SETS:
        got = emu_paths(emu, p, S0, r, q, T, n_steps, n_obs, seed, paths)
        st = MO.path_stats(p, S0, r, q, T, n_steps, n_obs, paths=paths, d=d)
        want = np.stack([st["ST"], st["sum"], st["max"], st["min"]], axis=1)
        assert np.all(np.isfinite(got))
        assert np.max(np.abs(got - want) / np.abs(want)) <= 1e-12, p
    if n_steps == 252:
        st = MO.path_stats(SETS[1], S0, r, q, T, n_steps, n_obs, paths=paths, d=d)
        assert st["N"].max() >= 1 and (st["truncated"] > 0).sum() >= 16
        st = MO.path_stats(SETS[2], S0, r, q, T, n_steps, n_obs, paths=paths, d=d)
        assert st["N"].max() == 0


def test_payoffs_match_oracle(emu):
    """Every kind, call and put, on the same path statistics: identical bits (the payoff has no transcendental)."""
    paths = np.arange(64, dtype=np.uint64)
    stats = emu_paths(emu, SETS[0], 100.0, 0.03, 0.0, 0.5, 26, 13, 4, paths)
    st = {"ST": stats[:, 0], "sum": stats[:, 1], "max": stats[:, 2], "min": stats[:, 3]}
    for kind in range(6):
        for call in (0, 1):
            for K, B in ((0.0, 110.0), (100.0, 105.0), (95.0, 92.0), (100.0, 1e300)):
                got = np.empty(64)
                emu.emu_mc_payoff(64, stats, 13, kind, call, K, B, got)
                want = MO.payoff(st, 13, kind, call, K, B)
                assert np.array_equal(got, want), (kind, call, K, B)


def test_scheme_is_a_martingale_in_expectation():
    """The scheme's discounted forward is an exact martingale: over 4 096 paths of the oracle, the mean of
    e^{-(r-q)T} S_T / S0 is within 4 standard errors of 1 on a coarse and a fine grid."""
    for n_steps in (4, 64):
        st = MO.path_stats(SETS[1], 100.0, 0.05, 0.02, 2.0, n_steps, n_steps, n_paths=4096)
        y = np.exp(-(0.05 - 0.02) * 2.0) * st["ST"] / 100.0
        assert abs(y.mean() - 1.0) <= 4 * y.std(ddof=1) / np.sqrt(y.size)
