"""Pins oracle/cos_oracle.py to fixtures produced by the unmodified reference (tests/golden/make_golden.py).

The oracle is NumPy on the same libm as the reference, written in the reference's operation order, so
the scalar restatement is expected to be bit-identical and the vectorised one within a few ulp.
"""
import numpy as np
import pytest

from conftest import rel_err
from oracle import cos_oracle as O

SCALAR_TOL = 1e-15      # scalar restatement: same operations in the same order
# vectorised restatement: NumPy's array loops for complex multiply are SIMD/FMA-dispatched while the
# scalar path is not, so a few prices move by some ulp of sum|summands| (measured here: max 3.4e-13
# relative, median 1e-15, 28 % bit-identical on 2 250 prices; SURVEY §8c measured 1.0e-13)
VEC_TOL = 1e-12


def test_survey_literals_are_tripwires(golden):
    """SURVEY.md §8c known-answer literals, recomputed by the reference into known_answers.npz."""
    g = golden("known_answers.npz")
    lit = np.array([[12.747652821906351, 9.173273829175123, 6.24553807185953, 4.007886084802539, 2.420075396920669],
                    [15.270182516467568, 11.972625306950297, 9.14571864274245, 6.803206414460713, 4.928582339601269],
                    [19.314600566413443, 16.2638895064355, 13.545233402249403, 11.1599576440257, 9.099103247472208]])
    assert np.array_equal(g["prices"], lit)
    assert np.array_equal(g["ab"], np.array([(-1.4132777861296757, 1.4432777861296755),
                                              (-1.9993873329093776, 2.0593873329093775),
                                              (-2.8282625135277004, 2.9482625135277005)]))
    assert float(g["demo_call"]) == 13.872851144174323
    assert float(g["demo_put"]) == 8.995793594010637


def test_scalar_oracle_known_answers(golden):
    g = golden("known_answers.npz")
    for i, T in enumerate(g["maturities"]):
        for j, K in enumerate(g["strikes"]):
            got = O.price_scalar(g["params"], 100.0, float(K), float(T), 0.05)
            assert rel_err(got, g["prices"][i, j]) <= SCALAR_TOL
        a, b = O.truncation_range_scalar(g["params"], 100.0, 100.0, float(T), 0.05)
        assert (a, b) == tuple(g["ab"][i])
    assert rel_err(O.price_scalar(g["demo_params"], 100, 100, 1.0, 0.05, True), g["demo_call"]) <= SCALAR_TOL
    assert rel_err(O.price_scalar(g["demo_params"], 100, 100, 1.0, 0.05, False), g["demo_put"]) <= SCALAR_TOL


def test_scalar_oracle_grid_sample(golden):
    g = golden("prices_grid15.npz")
    worst = 0.0
    for p in range(0, 150, 15):
        for i, T in enumerate(g["maturities"]):
            for j, kr in enumerate(g["k_rel"]):
                K = kr * g["spots"][p] / 100.0
                got = O.price_scalar(g["params"][p], g["spots"][p], K, float(T), float(g["r"]))
                worst = max(worst, float(rel_err(got, g["prices"][p, i, j])))
    assert worst <= SCALAR_TOL, worst


def test_vector_oracle_grid15(golden):
    g = golden("prices_grid15.npz")
    strikes = g["k_rel"][None, :] * g["spots"][:, None] / 100.0                  # [P,5]
    K = np.tile(strikes, (1, 3))                                                 # maturity-major
    T = np.repeat(g["maturities"], 5)
    got, ab = O.price_batch(g["params"], g["spots"], K, T, np.ones(15), float(g["r"]), return_ab=True)
    err = rel_err(got.reshape(150, 3, 5), g["prices"])
    assert err.max() <= VEC_TOL, err.max()
    assert np.abs(ab.reshape(150, 3, 5, 2) - g["ab"]).max() <= 1e-14


@pytest.mark.parametrize("tag", ["main", "edge"])
def test_vector_oracle_dense_surface(golden, tag):
    g = golden("dense_surface.npz")
    Ks, Ts = g[f"{tag}_strikes"], g[f"{tag}_maturities"]
    K = np.tile(Ks, len(Ts)); T = np.repeat(Ts, len(Ks))
    got, ab = O.price_batch(g["params"], 100.0, K, T, np.ones(K.size), float(g["r"]), N=256, return_ab=True)
    want = g[f"{tag}_prices"].reshape(4, -1)
    # deep OTM short-dated prices are rounding noise (SURVEY H4): judge abs error against S0
    assert (np.abs(got - want) / 100.0).max() <= 2e-13
    big = np.abs(want) > 0.5        # the C3 main grid has prices >= 0.6 (SURVEY §8d)
    assert rel_err(got[big], want[big]).max() <= 1e-11
    assert np.abs(ab.reshape(want.shape + (2,)) - g[f"{tag}_ab"].reshape(want.shape + (2,))).max() <= 1e-14


def test_oracle_edge_cases(golden):
    g = golden("edge_cases.npz")
    n = g["prices"].shape[0]
    assert n >= 70
    for i in range(n):
        S0, K, T, r, q, call, N = g["meta"][i]
        want = g["prices"][i]
        got_s = O.price_scalar(g["params"][i], S0, K, T, r, bool(call), q, int(N))
        got_v = O.price_batch(g["params"][i], S0, [K], [T], [call], r, q, int(N))[0, 0]
        if np.isnan(want):
            assert np.isnan(got_s) and np.isnan(got_v)
            continue
        assert rel_err(got_s, want) <= 1e-13 or abs(got_s - want) <= 1e-13 * S0, (i, got_s, want)
        assert abs(got_v - want) <= 5e-13 * max(S0, K), (i, got_v, want)
        a, b = O.truncation_range_scalar(g["params"][i], S0, K, T, r)
        assert np.allclose([a, b], g["ab"][i], rtol=1e-15, atol=0, equal_nan=True)


def test_oracle_cf(golden):
    g = golden("cf_values.npz")
    P, nT, nU = g["cf"].shape
    for p in range(P):
        for i, tau in enumerate(g["taus"]):
            vec = O.cf_vec(g["us"][None, :], np.array([[tau]]), g["params"][p][None, :], float(g["r"]), float(g["q"]))[0]
            for j, u in enumerate(g["us"]):
                s = O.cf_scalar(u, tau, g["params"][p], float(g["r"]), float(g["q"]))
                want = g["cf"][p, i, j]
                assert abs(s - want) <= 1e-15 * abs(want)
                assert abs(vec[j] - want) <= 1e-13 * abs(want)
    assert np.all(g["cf"][:, :, 0] == 1.0)          # phi(0) = 1 exactly (SURVEY A.4)


def test_oracle_cf_complex(golden):
    """characteristic_function at complex phi: the vectorised oracle against the reference's values."""
    g = golden("cf_complex.npz")
    for p in range(g["params"].shape[0]):
        for i, tau in enumerate(g["taus"]):
            vec = O.cf_vec(g["us"], float(tau), g["params"][p], float(g["r"]), float(g["q"]))
            assert np.abs(vec - g["cf"][p, i]).max() <= 2e-13 * np.maximum(1.0, np.abs(g["cf"][p, i])).max()


@pytest.mark.parametrize("tag", ["c1", "ragged"])
def test_oracle_loss_and_fd(golden, tag):
    g = golden("loss_cases.npz")
    m = (float(g[f"{tag}_spot"]), float(g[f"{tag}_r"]), g[f"{tag}_strike"], g[f"{tag}_maturity"],
         g[f"{tag}_is_call"], g[f"{tag}_market"])
    got = O.loss_batch(g[f"{tag}_x"], *m)
    want = g[f"{tag}_loss"]
    assert np.array_equal(got == O.SENTINEL, want == 1e10)
    assert (want == 1e10).sum() >= 2                      # NaN / inf parameter cases hit the sentinel
    assert (want > 100).sum() >= 3                        # Feller penalty active
    assert np.abs(got - want).max() <= 1e-9               # north-star bound
    # far tighter in practice (the loss at the true parameters is ~1e-28, i.e. pure rounding noise)
    assert np.all(np.abs(got - want) <= 1e-13 + 1e-11 * np.abs(want))
    # scalar path on a few
    for i in (0, 5, 27, 30):
        assert rel_err(O.loss_scalar(g[f"{tag}_x"][i], *m), want[i]) <= 1e-13
    # finite-difference stencil and gradient rule
    for c in range(g[f"{tag}_fd_f"].shape[0]):
        pts, dx = O.fd_stencil(g[f"{tag}_x"][c])
        f = O.loss_batch(pts, *m)
        assert np.abs(f - g[f"{tag}_fd_f"][c]).max() <= 1e-12
        f0, grad = O.loss_fd(g[f"{tag}_x"][c], *m)
        # forward differences with h=1e-8 turn ~1e-15 loss rounding noise into ~1e-7 gradient
        # noise (SURVEY H1): that noise floor, not an algorithmic difference, is the bound here
        noise = (1e-13 * abs(f0) + 1e-15) / O.FD_STEP
        assert np.abs(grad - g[f"{tag}_fd_g"][c]).max() <= noise


def test_oracle_initial_guess(golden):
    g = golden("initial_guess.npz")
    np.random.seed(0)
    m = (float(g["spot"]), g["strike"], g["maturity"], g["market"])
    assert np.array_equal(O.initial_guess(0, *m), g["g0"])
    assert np.array_equal(O.initial_guess(1, *m), g["g1"])
    assert np.array_equal(O.initial_guess(2, *m), g["g2"])
    assert np.array_equal(O.initial_guess(1, *m), g["g1_second_draw"])
    # SURVEY §8c: f(x0) literals for the C1 market
    assert float(g["f_g0"]) == 9.7610424427883e-05
    assert float(g["f_g1"]) == 11.100198535727506


def test_oracle_generator_draws(golden):
    g = golden("generator_seed42.npz")
    np.random.seed(42)
    params, spots, noise = O.generator_draws(20)
    assert np.array_equal(params, g["params"])
    assert np.array_equal(spots, g["spots"])
    K = O.GENERATOR_STRIKES_REL[None, :] * spots[:, None] / 100.0
    K = np.tile(K, (1, 3)); T = np.repeat(O.GENERATOR_MATURITIES, 5)
    assert np.array_equal(K, g["strikes"]) and np.array_equal(np.tile(T, (20, 1)), g["maturities"])
    model = O.price_batch(params, spots, K, T, np.ones(15), O.GENERATOR_RATE)
    assert rel_err(model, g["model_prices"]).max() <= VEC_TOL
    market = g["model_prices"] + noise * g["model_prices"]         # synthetic_generator.py:141-142
    assert np.array_equal(market, g["market_prices"])
    # SURVEY §8c literal
    assert g["model_prices"][0, 0] == 12.426829764997922


# ---- the C restatement (oracle/cos_oracle.c) -------------------------------------------------------------------
def test_c_oracle_grid15_bit_identical(golden):
    g = golden("prices_grid15.npz")
    K = np.tile(g["k_rel"][None, :] * g["spots"][:, None] / 100.0, (1, 3))
    T = np.repeat(g["maturities"], 5)
    got, ab = O.c_price_batch(g["params"], g["spots"], K, T, np.ones(15), float(g["r"]), return_ab=True)
    err = rel_err(got.reshape(150, 3, 5), g["prices"])
    print("C oracle vs reference: max rel err %.3e, bit-identical %.1f %%" % (err.max(), 100 * (err == 0).mean()))
    # not bit-identical: NumPy evaluates real exp / sin / cos / log with its own SIMD kernels, this file with glibc;
    # the differences are single ulps amplified by the conditioning of the COS sum (SURVEY H4)
    assert err.max() <= 2e-13 and np.median(err) <= 2e-15
    assert (err == 0).mean() >= 0.3
    assert np.abs(ab.reshape(150, 3, 5, 2) - g["ab"]).max() <= 2e-15


def test_c_oracle_edge_cases_and_dense(golden):
    g = golden("edge_cases.npz")
    for i in range(g["prices"].shape[0]):
        S0, K, T, r, q, call, N = g["meta"][i]
        got = O.c_price_batch(g["params"][i], S0, [K], [T], [call], r, q, int(N))[0, 0]
        want = g["prices"][i]
        if np.isnan(want):
            assert np.isnan(got)
        else:
            scale = max(S0, K) * max(1.0, np.exp(g["ab"][i][1]))          # magnitude of the summands (SURVEY H4)
            assert abs(got - want) <= 1e-12 * abs(want) or abs(got - want) <= 4e-14 * scale, (i, got, want)
    d = golden("dense_surface.npz")
    for tag in ("main", "edge"):
        Ks, Ts = d[f"{tag}_strikes"], d[f"{tag}_maturities"]
        got = O.c_price_batch(d["params"], 100.0, np.tile(Ks, len(Ts)), np.repeat(Ts, len(Ks)), np.ones(Ks.size * Ts.size),
                              float(d["r"]), N=256)
        assert np.abs(got - d[f"{tag}_prices"].reshape(4, -1)).max() <= 1e-12


def test_c_oracle_loss(golden):
    g = golden("loss_cases.npz")
    for tag in ("c1", "ragged"):
        got = O.c_loss_batch(g[f"{tag}_x"], float(g[f"{tag}_spot"]), float(g[f"{tag}_r"]), g[f"{tag}_strike"],
                             g[f"{tag}_maturity"], g[f"{tag}_is_call"], g[f"{tag}_market"])
        want = g[f"{tag}_loss"]
        assert np.array_equal(got == 1e10, want == 1e10)
        assert np.all(np.abs(got - want) <= 1e-15 + 1e-13 * np.abs(want))


def test_oracle_passes_the_reference_suites_own_checks():
    """The only checks the reference's tests/test_suite.py holds for this path (sections 3.1-3.4, :194-262): ATM 1Y call
    in (2, 15); prices decreasing in strike (>= 3 of 4 differences) and increasing in maturity; finite in 4 scenarios.
    Applied to the oracle (the GPU path gets the same checks in tests/test_gpu_dropin.py)."""
    p = np.array([0.04, 2.0, 0.04, 0.3, -0.5, 0.04, 1.5, 0.04, 0.2, -0.3, 0.1, 0.0, 0.1])
    atm = O.price_scalar(p, 100.0, 100.0, 1.0, 0.05)
    assert 2.0 < atm < 15.0 and abs(atm - 13.545233402249403) < 1e-12          # SURVEY §4: the suite prints 13.5452
    by_strike = [O.price_scalar(p, 100.0, K, 1.0, 0.05) for K in (90, 95, 100, 105, 110)]
    assert np.sum(np.diff(by_strike) < 0) >= 3
    by_maturity = [O.price_scalar(p, 100.0, 100.0, T, 0.05) for T in (0.25, 0.5, 1.0)]
    assert np.all(np.diff(by_maturity) > 0)
    for S, K, T in ((100, 100, 0.25), (100, 100, 2.0), (100, 80, 1.0), (100, 120, 1.0)):
        assert np.isfinite(O.price_scalar(p, S, K, T, 0.05))
    # put-call parity of the demo (double_heston.py:292-299, tolerance 0.01)
    d = np.array([0.04, 2.0, 0.04, 0.3, -0.5, 0.04, 1.5, 0.04, 0.2, -0.3, 0.5, -0.05, 0.10])
    c, q = O.price_scalar(d, 100, 100, 1.0, 0.05, True), O.price_scalar(d, 100, 100, 1.0, 0.05, False)
    assert abs((c - q) - (100 - 100 * np.exp(-0.05))) < 0.01


def test_c_oracle_noisy_trajectories(golden):
    """Every loss the reference optimiser evaluated on the four noisy markets (tests/golden/calib_noisy.npz, 7 056
    evaluations incl. sentinel and Feller-active points) from the C restatement; a sub-sample from the scalar port."""
    g = golden("calib_noisy.npz")
    total = 0
    for m in range(int(g["n_markets"])):
        args = (float(g[f"m{m}_spot"]), float(g["r"]), g[f"m{m}_strike"], g[f"m{m}_maturity"], np.ones(15), g[f"m{m}_market"])
        for s in (0, 2):
            xs, fs = g[f"m{m}_s{s}_xs"], g[f"m{m}_s{s}_fs"]
            got = O.c_loss_batch(xs, *args)
            assert np.array_equal(got == 1e10, fs == 1e10)
            assert np.all(np.abs(got - fs) <= 2e-13 * np.maximum(1.0, np.abs(fs)))      # glibc vs npymath, summation order
            for i in (0, fs.size // 2, fs.size - 1):
                assert abs(O.loss_scalar(xs[i], *args) - fs[i]) <= 1e-15 * max(1.0, abs(fs[i]))
            total += fs.size
    assert total == 7056


def test_counter_stream_known_answers():
    """Philox4x32-10 against the Random123 known-answer vectors (kat_vectors: zero, all-ones and pi-digit inputs),
    and the structure of the counter stream built on it (the product's definition: csrc/dhj_generate.cuh)."""
    def kat(ctr, key):
        return [int(v) for v in O.philox4x32_10(np.array([ctr], dtype=np.uint32), np.array([key], dtype=np.uint32))[0]]
    assert kat([0, 0, 0, 0], [0, 0]) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert kat([0xffffffff] * 4, [0xffffffff] * 2) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert kat([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]
    p, s, nz = O.counter_draws(7, 0, 1200, 500)
    lo, hi = O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1]
    assert (p >= lo).all() and (p <= hi).all()
    assert s[0] == 100.0 and s[500] == 100.0 and s[1000] == 100.0 and s[499] != 100.0     # histories restart
    # AR(1) inside a history (synthetic_generator.py:105-109), raw draws at its head
    raw, _, _ = O.counter_draws(7, 0, 1200, 1)                          # path_len 1: the raw i.i.d. draws
    assert np.array_equal(p[500], raw[500]) and np.array_equal(p[501], 0.9 * p[500] + (1 - 0.9) * raw[501])
    # any sub-range reproduces the same values: a function of (seed, index) only
    p2, s2, n2 = O.counter_draws(7, 700, 100, 500)
    assert np.array_equal(p2, p[700:800]) and np.array_equal(s2, s[700:800]) and np.array_equal(n2, nz[700:800])
    big = O.counter_draws(3, 0, 20000, 1)[2]
    assert abs(big.std() - 0.02) < 3e-4 and abs(big.mean()) < 3e-4


def test_counter_generate_grid():
    """counter_generate on any nT x nK grid: the default is the generator's 3 x 5 grid, bit for bit; an option's noise
    slot depends on its column only, so the first 15 noise columns of a 32-option grid are the 15-option noise."""
    g = O.counter_generate(9, 480, 40, 500)
    e = O.counter_generate(9, 480, 40, 500, strikes_rel=O.GENERATOR_STRIKES_REL, maturities=O.GENERATOR_MATURITIES,
                           L=10)
    for key in g:
        assert np.array_equal(g[key], e[key]), key
    assert g["model"].shape == (40, 15) and g["noise"].shape == (40, 15)
    w = O.counter_generate(9, 480, 40, 500, strikes_rel=np.linspace(80.0, 120.0, 32), maturities=[0.5])
    assert w["model"].shape == (40, 32) and w["noise"].shape == (40, 32)
    assert np.array_equal(w["noise"][:, :15], g["noise"]) and np.array_equal(w["params"], g["params"])
    assert np.array_equal(w["market"], w["model"] + w["noise"] * w["model"])
    assert np.array_equal(w["loss"], np.mean(((w["model"] - w["market"]) / w["market"]) ** 2, axis=1))


def test_counter_stream_exact_invariants():
    """persistence = 0 gives the raw draws, persistence = 1 repeats each path's head row, noise_sd = 0 gives
    market == model and a zero loss; all bit for bit."""
    raw = O.counter_draws(5, 0, 300, 1)[0]
    assert np.array_equal(O.counter_draws(5, 0, 300, 100, persistence=0.0)[0], raw)
    p1 = O.counter_draws(5, 30, 270, 100, persistence=1.0)[0]                 # paths start at 100 and 200
    heads = np.repeat(raw[[0, 100, 200]], 100, axis=0)[30:]
    assert np.array_equal(p1, heads)
    g = O.counter_generate(5, 30, 20, 100, noise_sd=0.0)
    assert np.array_equal(g["market"], g["model"]) and (g["loss"] == 0.0).all()


def test_counter_stream_64bit_words():
    """The key's high word (seed >> 32) and the counter's high word (index >> 32) reach the draws; a path that
    straddles index 2^32 continues its recurrences across it."""
    p7, s7, n7 = O.counter_draws(7, 0, 64, 1)
    for seed in (2 ** 32 + 7, 2 ** 63 + 7):                                   # same low word as seed 7
        p, s, nz = O.counter_draws(seed, 0, 64, 1)
        assert (p != p7).all(axis=1).all() and (nz != n7).all()
    w_lo = O.counter_words(7, np.array([5], dtype=np.uint64), 0)
    w_hi = O.counter_words(7, np.array([2 ** 32 + 5], dtype=np.uint64), 0)
    assert w_lo[0][0] != w_hi[0][0] and w_lo[1][0] != w_hi[1][0]
    c = 2 ** 32
    assert c % 500 not in (0, 1)                                              # index 2^32 is inside a path
    first = c - 700
    p, s, nz = O.counter_draws(7, first, 1400, 500)
    raw = O.counter_draws(7, first, 1400, 1)[0]
    z0, _ = O.counter_normal_pair(7, np.arange(first, first + 1400, dtype=np.uint64), 7)
    ret = 0.0003 + 0.01 * z0
    t = np.arange(first, first + 1400) % 500
    for k in range(1, 1400):
        if t[k] == 0:
            assert np.array_equal(p[k], raw[k]) and s[k] == 100.0
        else:
            assert np.array_equal(p[k], 0.9 * p[k - 1] + (1 - 0.9) * raw[k]), k
            assert s[k] == s[k - 1] * (1.0 + ret[k]), k
    straddle = np.flatnonzero((np.arange(first, first + 1400) // 500) == c // 500)
    assert straddle[0] + first < c < straddle[-1] + first                   # the path around 2^32 is all there
