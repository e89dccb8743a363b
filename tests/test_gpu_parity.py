"""GPU parity tests proper: every call goes through the C-ABI of libdhj.so (ctypes) and is compared with
the golden fixtures produced by the unmodified reference, and with the NumPy oracle on seeded samples.

Tolerances (north-star): 1e-10 relative price error, 1e-9 absolute loss error per evaluation.
Where a price is itself rounding noise of a badly conditioned sum (deep OTM short-dated, T = 30y: SURVEY
H4) the error is judged against the conditioning scale max(S0, K) * e^b instead, as the reference's own
NumPy-vectorised restatement has to be (tests/test_oracle_golden.py).
"""
import numpy as np
import pytest

from conftest import rel_err
from oracle import cos_oracle as O

pytestmark = pytest.mark.gpu

PRICE_RTOL = 1e-10
LOSS_ATOL = 1e-9


@pytest.fixture(scope="module")
def ctx():
    import dhj
    c = dhj.Context(0)
    yield c
    c.close()


def test_known_answers(ctx, golden):
    g = golden("known_answers.npz")
    got = ctx.price_grid(g["params"], 100.0, g["strikes"], g["maturities"], 0.05)[0]
    assert rel_err(got, g["prices"]).max() <= PRICE_RTOL
    demo = ctx.price_list(g["demo_params"], 100.0, [100.0, 100.0], [1.0, 1.0], [1, 0], 0.05)[0]
    assert rel_err(demo, [g["demo_call"], g["demo_put"]]).max() <= PRICE_RTOL
    # put-call parity, the one check the reference's demo performs (double_heston.py:292-299)
    assert abs((demo[0] - demo[1]) - (100 - 100 * np.exp(-0.05))) < 0.01


def test_grid15_golden(ctx, golden):
    g = golden("prices_grid15.npz")
    got = ctx.price_grid(g["params"], g["spots"], g["k_rel"], g["maturities"], float(g["r"]), scale_by_spot=True)
    err = rel_err(got, g["prices"])
    print("grid15: max rel err %.3e median %.3e" % (err.max(), np.median(err)))
    assert err.max() <= PRICE_RTOL
    # same through the list entry point with per-set strikes, in a scrambled option order
    K = np.tile(g["k_rel"][None, :] * g["spots"][:, None] / 100.0, (1, 3))
    T = np.repeat(g["maturities"], 5)
    perm = np.random.default_rng(1).permutation(15)
    got2 = ctx.price_list(g["params"], g["spots"], K[:, perm], T[perm], np.ones(15), float(g["r"]))
    assert rel_err(got2, g["prices"].reshape(150, 15)[:, perm]).max() <= PRICE_RTOL


def test_truncation_range_golden(ctx, golden):
    g = golden("prices_grid15.npz")
    K = (g["k_rel"] * 100.0 / 100.0)
    sel = np.where(g["spots"] == 100.0)[0]
    ab = ctx.truncation_range(g["params"][sel], 100.0, np.tile(K, 3), np.repeat(g["maturities"], 5), float(g["r"]))
    want = g["ab"][sel].reshape(len(sel), 15, 2)
    assert np.abs(ab - want).max() <= 1e-13


@pytest.mark.parametrize("tag", ["main", "edge"])
def test_dense_surface_golden(ctx, golden, tag):
    g = golden("dense_surface.npz")
    Ks, Ts = g[f"{tag}_strikes"], g[f"{tag}_maturities"]
    got = ctx.price_grid(g["params"], 100.0, Ks, Ts, float(g["r"]), N=256)
    want = g[f"{tag}_prices"]
    abs_err = np.abs(got - want) / 100.0
    print(tag, "abs/S0 max %.3e" % abs_err.max())
    assert abs_err.max() <= 2e-13
    big = want > 0.5
    assert rel_err(got[big], want[big]).max() <= PRICE_RTOL
    if tag == "edge":
        # the widening must actually bind somewhere in this fixture, else the slow path is untested
        ab = g["edge_ab"]
        assert (np.abs(ab[:, :, 0, 0] - ab[:, :, -1, 0]) > 0).any() or (np.abs(ab[:, :, 0, 1] - ab[:, :, -1, 1]) > 0).any()


def test_edge_cases_golden(ctx, golden):
    g = golden("edge_cases.npz")
    worst = 0.0
    for i in range(g["prices"].shape[0]):
        S0, K, T, r, q, call, N = g["meta"][i]
        want = g["prices"][i]
        got = ctx.price_list(g["params"][i], S0, [K], [T], [call], r, q, int(N))[0, 0]
        if np.isnan(want):
            assert np.isnan(got), (i, got)
            continue
        sigma1 = g["params"][i][3]
        if sigma1 <= 1e-3:
            # vol-of-vol -> 0: the reference's beta-d cancels catastrophically (its own value moves by
            # 3e-4 between sigma=1e-6 and 1e-3); only a loose agreement is meaningful (DESIGN.md §4)
            assert abs(got - want) <= 1e-3 * want
            continue
        a, b = g["ab"][i]
        scale = max(S0, K) * max(1.0, np.exp(b))            # magnitude of the summands (SURVEY H4)
        err = abs(got - want)
        assert err <= PRICE_RTOL * abs(want) or err <= 4e-14 * scale, (i, got, want, err / scale)
        worst = max(worst, err / scale)
    print("edge cases: worst abs err / conditioning scale = %.3e" % worst)


def test_cf_golden(ctx, golden):
    g = golden("cf_values.npz")
    for p in range(g["cf"].shape[0]):
        for i, tau in enumerate(g["taus"]):
            got = ctx.cf(g["params"][p], float(g["r"]), float(g["q"]), float(tau), g["us"])
            want = g["cf"][p, i]
            # the exponent X of phi = exp(X) carries ~1e-15*|X| absolute error, |X| up to ~150 here
            assert (np.abs(got - want) <= 2e-13 * np.abs(want) + 1e-300).all(), (p, i)


def test_cf_complex_golden(ctx, golden):
    """characteristic_function at COMPLEX phi (dhj_cf_complex) against the reference's own values."""
    g = golden("cf_complex.npz")
    worst = 0.0
    for p in range(g["params"].shape[0]):
        for i, tau in enumerate(g["taus"]):
            got = ctx.cf(g["params"][p], float(g["r"]), float(g["q"]), float(tau), g["us"])
            want = g["cf"][p, i]
            worst = max(worst, (np.abs(got - want) / np.maximum(np.abs(want), 1e-300)).max())
    print("complex-phi CF: max rel err %.3e" % worst)
    assert worst <= 1e-12
    # real frequencies through the complex entry point agree with the real one
    u = np.linspace(0.5, 60.0, 9)
    a = ctx.cf(g["params"][0], 0.03, 0.0, 0.5, u)
    b = ctx.cf(g["params"][0], 0.03, 0.0, 0.5, u.astype(np.complex128))
    assert np.abs(a - b).max() <= 2e-13 * np.abs(a).max()


def test_chi_psi(ctx):
    # double_heston.py:141-158 against the scalar oracle
    a, b, x = -2.8282625135277004, 2.9482625135277005, np.log(95.0 / 100.0)
    ks = np.array([0, 1, 2, 17, 64, 127, 255])
    chi, psi = ctx.chi_psi(ks, x, b, a, b)
    for j, k in enumerate(ks):
        c_ref, p_ref = O._chi_psi_scalar(int(k), x, b, a, b)
        assert abs(chi[j] - c_ref) <= 1e-13 * max(1.0, abs(c_ref))
        assert abs(psi[j] - p_ref) <= 1e-13 * max(1.0, abs(p_ref))


def test_random_sample_vs_oracle(ctx):
    """2 000 seeded parameter sets x the 15-option grid against the vectorised oracle (C2 sub-sample)."""
    rng = np.random.default_rng(20260101)
    P = 2000
    params = rng.uniform(O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1], size=(P, 13))
    got = ctx.price_grid(params, 100.0, O.GENERATOR_STRIKES_REL, O.GENERATOR_MATURITIES, 0.03)
    K = np.tile(O.GENERATOR_STRIKES_REL, 3); T = np.repeat(O.GENERATOR_MATURITIES, 5)
    want = O.price_batch(params, 100.0, K, T, np.ones(15), 0.03).reshape(P, 3, 5)
    err = rel_err(got, want)
    print("C2 sub-sample: max rel err %.3e median %.3e" % (err.max(), np.median(err)))
    assert err.max() <= PRICE_RTOL


@pytest.mark.parametrize("N", [1, 2, 31, 32, 33, 100, 129, 300, 512, 1000, 2048])
def test_ragged_n(ctx, N):
    rng = np.random.default_rng(N)
    params = rng.uniform(O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1], size=(7, 13))
    K = np.array([80.0, 100.0, 125.0]); T = np.array([0.5, 0.5, 1.5]); c = np.array([1, 0, 1])
    got = ctx.price_list(params, 100.0, K, T, c, 0.02, 0.01, N)
    want = O.price_batch(params, 100.0, K, T, c, 0.02, 0.01, N)
    assert (np.abs(got - want) <= 1e-10 * np.abs(want) + 1e-11).all()


def test_empty_and_errors(ctx):
    import dhj
    assert ctx.price_list(np.zeros((0, 13)), 100.0, [100.0], [1.0], [1], 0.05).shape == (0, 1)
    assert ctx.price_list(np.ones((2, 13)), 100.0, [], [], [], 0.05).shape == (2, 0)
    with pytest.raises(dhj.NativeError):
        ctx.price_list(np.ones((1, 13)), 100.0, [100.0], [1.0], [1], 0.05, N=0)
    # NaN parameters give NaN prices, not an error (the reference returns NaN silently)
    p = np.full((1, 13), np.nan)
    assert np.isnan(ctx.price_list(p, 100.0, [100.0], [1.0], [1], 0.05)).all()


def test_loss_paths_agree_bitwise(ctx, golden):
    """Small batches run the fused loss kernel, large ones expand -> pricing kernel -> reduce (dhj_abi.cu run_loss):
    the same states must give the same bits either way, for losses and FD gradients."""
    g = golden("loss_cases.npz")
    mk = ctx.market(float(g["c1_spot"]), float(g["c1_r"]), g["c1_strike"], g["c1_maturity"], g["c1_is_call"],
                    g["c1_market"])
    rng = np.random.default_rng(5)
    x = g["c1_x"][0] + 0.05 * rng.standard_normal((3000, 13))
    x[7, 3] = 4.0                                                  # Feller penalty active
    x[11, 0] = np.nan                                              # sentinel
    f_big, g_big = mk.loss_fd(x, 1e-8)                             # 42 000 evaluations: split path
    f_small, g_small = mk.loss_fd(x[:64], 1e-8)                    # 896 evaluations: fused kernel
    assert np.array_equal(f_big[:64], f_small, equal_nan=True) and np.array_equal(g_big[:64], g_small, equal_nan=True)
    l_big = mk.loss_batch(np.tile(x, (7, 1)))                      # 21 000 evaluations: split path
    l_small = mk.loss_batch(x[:500])
    assert np.array_equal(l_big[:500], l_small, equal_nan=True) and np.array_equal(l_small[:64], f_small, equal_nan=True)
    assert f_small[11] == 1e10 and f_small[7] > 1.0
    mk.close()


@pytest.mark.parametrize("tag", ["c1", "ragged"])
def test_loss_golden(ctx, golden, tag):
    g = golden("loss_cases.npz")
    mk = ctx.market(float(g[f"{tag}_spot"]), float(g[f"{tag}_r"]), g[f"{tag}_strike"], g[f"{tag}_maturity"],
                    g[f"{tag}_is_call"], g[f"{tag}_market"])
    got = mk.loss_batch(g[f"{tag}_x"])
    want = g[f"{tag}_loss"]
    assert np.array_equal(got == 1e10, want == 1e10)
    err = np.abs(got - want)
    print(tag, "loss: max abs err %.3e (rel to loss %.3e)" % (err.max(), (err / np.abs(want)).max()))
    assert (err <= LOSS_ATOL * np.maximum(1.0, np.abs(want))).all()
    # one-launch FD: f, the 14 stencil losses and scipy's gradient rule
    n_fd = g[f"{tag}_fd_f"].shape[0]
    f, grad, f_all = mk.loss_fd(g[f"{tag}_x"][:n_fd], 1e-8, want_all=True)
    assert np.abs(f_all - g[f"{tag}_fd_f"]).max() <= LOSS_ATOL
    assert np.array_equal(f, f_all[:, 0])
    for c in range(n_fd):
        x = g[f"{tag}_x"][c]
        dx = (x + 1e-8) - x
        assert np.array_equal(grad[c], (f_all[c, 1:] - f_all[c, 0]) / dx)          # the rule itself, exactly
        noise = (1e-13 * abs(f[c]) + 1e-15) / 1e-8                                  # SURVEY H1 noise floor
        assert np.abs(grad[c] - g[f"{tag}_fd_g"][c]).max() <= 10 * noise
    # model prices at x (calibrate's re-pricing)
    pr = mk.prices(g[f"{tag}_x"][:3])
    want_pr = O.price_batch(O.transform_params(g[f"{tag}_x"][:3]), float(g[f"{tag}_spot"]), g[f"{tag}_strike"],
                            g[f"{tag}_maturity"], g[f"{tag}_is_call"], float(g[f"{tag}_r"]))
    assert rel_err(pr, want_pr).max() <= PRICE_RTOL
    mk.close()


def test_trajectory_replay(ctx, golden):
    """Every x the REFERENCE optimiser visited (3 starts, 3 206 evaluations): GPU loss within 1e-9 abs."""
    g = golden("calib_trajectory.npz")
    mk = ctx.market(float(g["spot"]), float(g["r"]), g["strike"], g["maturity"], g["is_call"], g["market"])
    worst = 0.0
    for s in range(3):
        xs, fs = g[f"s{s}_xs"], g[f"s{s}_fs"]
        got = mk.loss_batch(xs)
        assert np.array_equal(got == 1e10, fs == 1e10)
        err = np.abs(got - fs) / np.maximum(1.0, np.abs(fs))
        worst = max(worst, err.max())
    print("trajectory replay: worst abs loss error %.3e over 3206 reference evaluations" % worst)
    assert worst <= LOSS_ATOL
    mk.close()


def test_many_markets(ctx):
    """Per-calibration markets (C5 shape): market_index routes each x to its own spot/strikes/prices."""
    rng = np.random.default_rng(5)
    n = 6
    params = rng.uniform(O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1], size=(n, 13))
    spots = rng.uniform(90, 110, size=n)
    K = np.tile(O.GENERATOR_STRIKES_REL[None, :] * spots[:, None] / 100.0, (1, 3))
    T = np.repeat(O.GENERATOR_MATURITIES, 5)
    market = O.price_batch(params, spots, K, T, np.ones(15), 0.03) * (1 + 0.02 * rng.standard_normal((n, 15)))
    mk = ctx.market(spots, 0.03, K, T, np.ones(15), market)
    x = O.inverse_transform_params(params) + 0.05 * rng.standard_normal((n, 13))
    idx = np.array([3, 0, 5, 1, 4, 2])
    got = mk.loss_batch(x, idx)
    for i in range(n):
        j = idx[i]
        want = O.loss_batch(x[i], spots[j], 0.03, K[j], T, np.ones(15), market[j])[0]
        assert abs(got[i] - want) <= LOSS_ATOL
    f, grad = mk.loss_fd(x, 1e-8, idx)
    assert np.abs(f - got).max() == 0.0
    mk.close()


def test_loss_general_path(ctx):
    """A market with 12 strikes on one maturity (> 8 per slice) takes the expand / dense-price / reduce path."""
    rng = np.random.default_rng(9)
    params = rng.uniform(O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1], size=13)
    K = np.concatenate([np.linspace(85, 115, 12), [95.0, 100.0, 105.0]])
    T = np.concatenate([np.full(12, 0.5), np.full(3, 1.0)])
    call = np.concatenate([np.ones(12), [0, 1, 0]])
    market = O.price_batch(params, 100.0, K, T, call, 0.02)[0] * (1 + 0.01 * rng.standard_normal(15))
    mk = ctx.market(100.0, 0.02, K, T, call, market)
    x = O.inverse_transform_params(params)[None, :] + 0.1 * rng.standard_normal((5, 13))
    got = mk.loss_batch(x)
    want = O.loss_batch(x, 100.0, 0.02, K, T, call, market)
    assert np.abs(got - want).max() <= LOSS_ATOL
    f, grad, f_all = mk.loss_fd(x, 1e-8, want_all=True)
    assert np.array_equal(f, got)
    for c in range(5):
        dx = (x[c] + 1e-8) - x[c]
        assert np.array_equal(grad[c], (f_all[c, 1:] - f_all[c, 0]) / dx)
        pts, _ = O.fd_stencil(x[c])
        assert np.abs(f_all[c] - O.loss_batch(pts, 100.0, 0.02, K, T, call, market)).max() <= LOSS_ATOL
    assert rel_err(mk.prices(x), O.price_batch(O.transform_params(x), 100.0, K, T, call, 0.02)).max() <= PRICE_RTOL
    mk.close()


def test_many_strikes_and_slices(ctx):
    """300 strikes on one slice (chunks of 224 and 76 strikes) and 40 maturities (more slices than a block batch)."""
    rng = np.random.default_rng(10)
    params = rng.uniform(O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1], size=(3, 13))
    K = np.linspace(70, 130, 300); T = np.full(300, 0.75)
    call = (np.arange(300) % 3 != 0).astype(int)
    got = ctx.price_list(params, 100.0, K, T, call, 0.03)
    want = O.price_batch(params, 100.0, K, T, call, 0.03)
    assert (np.abs(got - want) <= 1e-10 * np.abs(want) + 1e-12).all()
    T2 = np.linspace(0.1, 2.0, 40); K2 = np.full(40, 100.0)
    got2 = ctx.price_list(params, 100.0, K2, T2, np.ones(40), 0.03)
    assert rel_err(got2, O.price_batch(params, 100.0, K2, T2, np.ones(40), 0.03)).max() <= PRICE_RTOL


def test_full_size_c2_properties(ctx):
    """BASELINE config C2 at FULL size (1 048 576 parameter sets x 15 options, N = 128) through size-independent
    properties: run-to-run determinism, agreement of the grid and list entry points, put-call parity on every
    price, monotonicity in strike and maturity, and the oracle on a scattered sub-sample."""
    rng = np.random.default_rng(20260101)
    P = 1 << 20
    params = rng.uniform(O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1], size=(P, 13))
    Ks, Ts, r = O.GENERATOR_STRIKES_REL, O.GENERATOR_MATURITIES, 0.03
    calls = ctx.price_grid(params, 100.0, Ks, Ts, r)
    again = ctx.price_grid(params, 100.0, Ks, Ts, r)
    assert np.array_equal(calls, again)                                   # deterministic, launch to launch
    assert np.isfinite(calls).all() and (calls > 0).all()
    puts = ctx.price_grid(params, 100.0, Ks, Ts, r, is_call=False)
    parity = calls - puts - (100.0 - Ks[None, None, :] * np.exp(-r * Ts)[None, :, None])
    print("C2 full size: max |put-call parity residual| = %.3e over %d prices" % (np.abs(parity).max(), calls.size))
    assert np.abs(parity).max() < 1e-4                                    # COS truncation level of the reference (2e-10..1e-5)
    assert (np.diff(calls, axis=2) < 0).all()                             # decreasing in strike
    assert (np.diff(calls, axis=1) > 0).all()                             # increasing in maturity
    sel = rng.choice(P, size=1500, replace=False)
    K = np.tile(Ks, 3); T = np.repeat(Ts, 5)
    want = O.price_batch(params[sel], 100.0, K, T, np.ones(15), r).reshape(-1, 3, 5)
    assert rel_err(calls[sel], want).max() <= PRICE_RTOL
    lst = ctx.price_list(params[sel], 100.0, K, T, np.ones(15), r).reshape(-1, 3, 5)
    assert np.array_equal(lst, calls[sel])                                # list and grid entry points agree bit for bit


def test_host_path_chunking_and_memory_kinds(ctx):
    """The host-buffer entry points stream chunks of <= 131 072 sets through three slots: results must not depend
    on chunk boundaries, on per-set strikes / spots being present, or on the caller's memory being pinned."""
    import torch
    rng = np.random.default_rng(12)
    P = 300_001              # pageable: three uniform chunks, the last one ragged; pinned: ramped schedule
                             # 16 384, 32 768, 131 072, 70 625, 32 768, 16 384 (dhj_abi.cu run_price_host)
    params = rng.uniform(O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1], size=(P, 13))
    spots = rng.uniform(80, 120, size=P)
    Ks, Ts = O.GENERATOR_STRIKES_REL, O.GENERATOR_MATURITIES
    pageable = ctx.price_grid(params, spots, Ks, Ts, 0.03, scale_by_spot=True)
    pin_p = torch.from_numpy(params).pin_memory(); pin_s = torch.from_numpy(spots).pin_memory()
    pin_o = torch.empty((P, 3, 5), dtype=torch.float64).pin_memory()
    pinned = ctx.price_grid(pin_p.numpy(), pin_s.numpy(), Ks, Ts, 0.03, scale_by_spot=True, out=pin_o.numpy())
    assert np.array_equal(pageable, pinned)
    # per-set strike rows through the list entry point give the same bits as the scaled grid
    K = np.tile(Ks[None, :] * spots[:, None] / 100.0, (1, 3)); T = np.repeat(Ts, 5)
    lst = ctx.price_list(params, spots, K, T, np.ones(15), 0.03)
    assert np.array_equal(lst.reshape(P, 3, 5), pageable)
    # rows around the chunk boundaries against single-set calls
    for p in (0, 16383, 16384, 49151, 49152, 131071, 131072, 180223, 180224, 262143, 262144, P - 16385, P - 1):
        one = ctx.price_grid(params[p], spots[p], Ks, Ts, 0.03, scale_by_spot=True)[0]
        assert np.array_equal(one, pageable[p]), p
    sel = rng.choice(P, size=300, replace=False)
    want = O.price_batch(params[sel], spots[sel], K[sel], T, np.ones(15), 0.03).reshape(-1, 3, 5)
    assert rel_err(pageable[sel], want).max() <= PRICE_RTOL


def test_nan_and_inf_parameters_give_nan_everywhere(ctx):
    """Every single parameter set to NaN / +inf / -inf in turn: the reference returns NaN (or, rarely, inf) silently;
    nothing may come back as a plausible finite price, because the loss turns non-finite prices into the sentinel."""
    base = np.array([0.04, 2.0, 0.04, 0.3, -0.5, 0.04, 1.5, 0.04, 0.2, -0.3, 0.1, -0.02, 0.1])
    rows = []
    for j in range(13):
        for bad in (np.nan, np.inf, -np.inf):
            p = base.copy(); p[j] = bad; rows.append(p)
    rows = np.array(rows)
    K = np.tile([90.0, 100.0, 110.0], 2); T = np.repeat([0.5, 1.0], 3)
    got = ctx.price_list(rows, 100.0, K, T, [1, 1, 0, 0, 1, 1], 0.03)
    with np.errstate(all="ignore"):
        want = O.price_batch(rows, 100.0, K, T, [1, 1, 0, 0, 1, 1], 0.03)
    # where the reference is non-finite so are we; a finite reference value (e.g. lambda = -inf is not one) must match
    assert (~np.isfinite(got[~np.isfinite(want)])).all()
    fin = np.isfinite(want)
    assert np.isfinite(got[fin]).all() and rel_err(got[fin], want[fin]).max() <= 1e-9 if fin.any() else True
    mk = ctx.market(100.0, 0.03, K, T, [1, 1, 0, 0, 1, 1], np.full(6, 5.0))
    x = np.tile(O.inverse_transform_params(base), (6, 1))
    x[0, 1] = np.nan; x[1, 3] = np.inf; x[2, 0] = -np.inf; x[3, 11] = np.nan; x[4, 4] = np.nan
    loss = mk.loss_batch(x)
    with np.errstate(all="ignore"):
        ref = O.loss_batch(x, 100.0, 0.03, K, T, [1, 1, 0, 0, 1, 1], np.full(6, 5.0))
    # (x = -inf for v1_0 means v1_0 = exp(-inf) = 0: a finite loss in the reference too)
    assert np.array_equal(loss == 1e10, ref == 1e10) and (loss == 1e10).sum() == 4
    assert np.abs(loss - ref).max() <= LOSS_ATOL
    mk.close()


def test_large_sample_vs_c_oracle(ctx):
    """20 000 parameter sets x 15 options (300 000 prices) against the C restatement of the reference
    (oracle/cos_oracle.c, pinned to the golden fixtures in tests/test_oracle_golden.py), puts and per-set spots included."""
    rng = np.random.default_rng(31)
    P = 20000
    params = rng.uniform(O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1], size=(P, 13))
    spots = rng.uniform(70, 140, size=P)
    K = np.tile(O.GENERATOR_STRIKES_REL[None, :] * spots[:, None] / 100.0, (1, 3)); T = np.repeat(O.GENERATOR_MATURITIES, 5)
    call = (np.arange(15) % 2 == 0)
    got = ctx.price_list(params, spots, K, T, call, 0.03, 0.01)
    want = O.c_price_batch(params, spots, K, T, call, 0.03, 0.01)
    err = rel_err(got, want)
    print("300k prices vs C oracle: max rel err %.3e, median %.3e, 99.9 %% below %.3e"
          % (err.max(), np.median(err), np.quantile(err, 0.999)))
    assert err.max() <= PRICE_RTOL


def test_loss_many_slices(ctx):
    """A market with 40 distinct maturities (more slices than one block batch holds): the loss goes through the
    expand / price / reduce path and still matches the oracle."""
    rng = np.random.default_rng(13)
    params = rng.uniform(O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1], size=13)
    T = np.linspace(0.1, 2.0, 40); K = 100.0 + 10.0 * np.sin(np.arange(40)); call = (np.arange(40) % 2).astype(int)
    market = O.price_batch(params, 100.0, K, T, call, 0.02)[0] * (1 + 0.01 * rng.standard_normal(40))
    mk = ctx.market(100.0, 0.02, K, T, call, market)
    x = O.inverse_transform_params(params)[None, :] + 0.05 * rng.standard_normal((4, 13))
    f, g = mk.loss_fd(x)
    want = O.loss_batch(x, 100.0, 0.02, K, T, call, market)
    assert np.abs(f - want).max() <= LOSS_ATOL
    assert np.array_equal(mk.loss_batch(x), f)
    mk.close()
