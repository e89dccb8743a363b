"""Monte Carlo pricing of path-dependent options on the B200 (dhj_mc_price, csrc/dhj_mc.cuh): replication of the NumPy
restatement path for path, the scheme's exact martingale, agreement with the COS price, the estimator's identities,
bit-determinism and independence of the call's composition and of how the host cuts it, argument checks, the checked
build and the DoubleHeston front."""
import ctypes
import os
import sys

import numpy as np
import pytest

import mc_oracle as MO
from conftest import PKG
from oracle import cos_oracle as O

pytestmark = pytest.mark.gpu

CHECKED = os.path.join(PKG, "lib", "libdhj_checked.so")
KINDS = MO.KINDS
# Sets that truncate the variance (the second violates the Feller condition on both factors) but stay clear of the
# regime where the Euler map near v = 0 amplifies ulp-level differences (DESIGN.md §6f)
SETS = np.array([
    [0.04, 2.0, 0.04, 0.3, -0.6, 0.03, 0.8, 0.05, 0.2, -0.4, 0.15, -0.05, 0.08],
    [0.02, 2.0, 0.03, 0.5, -0.8, 0.04, 1.0, 0.04, 0.25, -0.5, 1.0, -0.1, 0.15],
    [0.05, 3.0, 0.05, 0.4, -0.7, 0.02, 1.0, 0.03, 0.15, -0.3, 0.0, -0.05, 0.08],
])
# steps per year of the European-vs-COS test: of 64 / 128 / 256 / 512, the only grid whose measured difference from COS
# stayed below one standard error of 2^22 paths on every option at T = 1 (DESIGN.md §6f)
STEPS_PER_YEAR = 512


@pytest.fixture(scope="module")
def ctx():
    import dhj
    c = dhj.Context(0)
    yield c
    c.close()


def _book():
    """Every kind x call / put at K = 100, plus K = 0 calls (forwards) of the European and the Asian."""
    kind, call, K, B = [], [], [], []
    for k in KINDS:
        for c in (1, 0):
            kind.append(k); call.append(c); K.append(100.0)
            B.append({"up-and-out": 118.0, "up-and-in": 118.0, "down-and-out": 86.0, "down-and-in": 86.0}.get(k, np.nan))
    for k in ("european", "asian"):
        kind.append(k); call.append(1); K.append(0.0); B.append(np.nan)
    return kind, call, K, B


def test_replicates_oracle(ctx):
    """256 paths, 3 sets with their own spots: every kind x call / put equals the NumPy restatement's discounted mean to
    1e-12 relative (and its standard error to 1e-10); no path's monitored extreme lies within 1e-9 of its barrier."""
    kind, call, K, B = _book()
    S0 = np.array([100.0, 97.0, 104.0])
    r, q, T, n_steps, n_obs, seed = 0.03, 0.01, 1.0, 64, 16, 2**32 + 5
    got, err = ctx.mc_price(SETS, S0, T, kind, call, K, r, q, barrier=B, n_paths=256, n_steps=n_steps, n_obs=n_obs,
                            seed=seed)
    want, werr, stats = MO.mc_price(SETS, S0, r, q, T, n_steps, n_obs, kind, call, K, B, seed, 256)
    for st in stats:
        for b in (118.0, 86.0):
            assert np.min(np.abs(np.concatenate([st["max"], st["min"]]) - b)) > 1e-9 * b
        assert (st["max"] >= 118.0).any() and (st["max"] < 118.0).any()
        assert (st["min"] <= 86.0).any() and (st["min"] > 86.0).any()
    assert np.count_nonzero(want) >= want.size - 3
    assert np.all(np.abs(got - want) <= 1e-12 * np.abs(want))
    assert np.all(np.abs(err - werr) <= 1e-10 * np.abs(werr))


@pytest.mark.parametrize("T", [0.25, 1.0, 5.0])
def test_forward_is_unbiased(ctx, T):
    """A call with K = 0 prices the forward S0 e^{-qT} within 4 standard errors on a coarse and a fine grid, up to the
    generator's top jump intensity: the scheme is an exact martingale, with no discretisation bias to allow for."""
    rng = np.random.default_rng(int(T * 100))
    params = rng.uniform(O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1], size=(4, 13))
    params[:, 10] = [0.0, 0.05, 0.15, 0.25]
    S0, r, q = 100.0, 0.03, 0.02
    for steps in (max(1, int(4 * T)), int(252 * T)):
        price, err = ctx.mc_price(params, S0, T, "european", 1, 0.0, r, q, n_paths=1 << 20, n_steps=steps, seed=11)
        fwd = S0 * np.exp(-q * T)
        assert np.all(np.abs(price[:, 0] - fwd) <= 4 * err[:, 0]), (steps, price[:, 0] - fwd, err[:, 0])


@pytest.mark.parametrize("T", [0.25, 1.0])
def test_european_matches_cos(ctx, T):
    """European calls and puts on the generator's parameter box agree with the COS price (price_list, N = 512) within
    4 standard errors at 2^22 paths on STEPS_PER_YEAR steps per year."""
    rng = np.random.default_rng(2024 + int(T * 4))
    params = rng.uniform(O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1], size=(6, 13))
    K = np.array([90.0, 100.0, 110.0] * 2)
    call = np.array([1, 1, 1, 0, 0, 0])
    S0, r, q = 100.0, O.GENERATOR_RATE, 0.0
    steps = max(1, int(round(STEPS_PER_YEAR * T)))
    price, err = ctx.mc_price(params, S0, T, "european", call, K, r, q, n_paths=1 << 22, n_steps=steps, seed=3)
    cos = ctx.price_list(params, S0, K, np.full(6, T), call, r, q, N=512)
    assert np.all(np.abs(price - cos) <= 4 * err), np.max(np.abs(price - cos) / err)


def test_estimator_identities(ctx):
    """In + out = European (up and down), put-call parity of the estimator for the European and the Asian, all to
    1e-12 S0 on one call; an Asian with one observation and an up-and-out with B = 1e300 give the European's bits."""
    kind = ["european", "european", "asian", "asian", "up-and-out", "up-and-in", "down-and-out", "down-and-in",
            "european", "asian", "up-and-out", "up-and-out"]
    call = [1, 0, 1, 0, 1, 1, 1, 1, 1, 1, 1, 0]
    K = [95.0, 95.0, 95.0, 95.0, 95.0, 95.0, 95.0, 95.0, 0.0, 0.0, 95.0, 95.0]
    B = [np.nan] * 4 + [112.0, 112.0, 90.0, 90.0, np.nan, np.nan, 1e300, 1e300]
    S0, r, q, T = 100.0, 0.04, 0.01, 0.75
    price, _ = ctx.mc_price(SETS, S0, T, kind, call, K, r, q, barrier=B, n_paths=100_003, n_steps=48, n_obs=12, seed=9)
    disc, tol = np.exp(-r * T), 1e-12 * S0
    assert np.all(np.abs(price[:, 4] + price[:, 5] - price[:, 0]) <= tol)
    assert np.all(np.abs(price[:, 6] + price[:, 7] - price[:, 0]) <= tol)
    assert np.all(np.abs((price[:, 0] - price[:, 1]) - (price[:, 8] - disc * 95.0)) <= tol)
    assert np.all(np.abs((price[:, 2] - price[:, 3]) - (price[:, 9] - disc * 95.0)) <= tol)
    assert np.array_equal(price[:, 10], price[:, 0]) and np.array_equal(price[:, 11], price[:, 1])
    p1, e1 = ctx.mc_price(SETS, S0, T, ["asian", "european"], 1, 95.0, r, q, n_paths=100_003, n_steps=48, n_obs=1,
                          seed=9)
    assert np.array_equal(p1[:, 0], p1[:, 1]) and np.array_equal(e1[:, 0], e1[:, 1])


def test_determinism_and_independence(ctx):
    """Same bits from two calls; a set priced alone equals the set inside a batch; an option's output does not depend on
    the other options or their order; equal sets give equal outputs; n_paths not a multiple of the chunk."""
    kind, call, K, B = _book()
    params = np.concatenate([SETS, SETS[1:2]])
    args = dict(n_paths=256 * 37 + 101, n_steps=30, n_obs=10, seed=77)
    a = ctx.mc_price(params, 100.0, 0.5, kind, call, K, 0.02, barrier=B, **args)
    b = ctx.mc_price(params, 100.0, 0.5, kind, call, K, 0.02, barrier=B, **args)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
    assert np.array_equal(a[0][1], a[0][3]) and np.array_equal(a[1][1], a[1][3])
    for p in range(4):
        alone = ctx.mc_price(params[p], 100.0, 0.5, kind, call, K, 0.02, barrier=B, **args)
        assert np.array_equal(alone[0][0], a[0][p]) and np.array_equal(alone[1][0], a[1][p])
    perm = np.random.default_rng(1).permutation(len(kind))
    c = ctx.mc_price(params, 100.0, 0.5, [kind[i] for i in perm], np.array(call)[perm], np.array(K)[perm], 0.02,
                     barrier=np.array(B)[perm], **args)
    assert np.array_equal(c[0], a[0][:, perm]) and np.array_equal(c[1], a[1][:, perm])
    one = ctx.mc_price(params, 100.0, 0.5, kind[5], call[5], K[5], 0.02, barrier=B[5], **args)
    assert np.array_equal(one[0][:, 0], a[0][:, 5])


def test_host_split_does_not_change_bits(ctx):
    """The host cuts a call into launches of bounded scratch (groups of sets, or runs of one set's chunks); the carried
    (n, mean, M2) makes every cut give the same bits.  Forced small cuts at a small size, and the natural cut of a call
    whose chunk partials exceed the default scratch (2^24 + 5 paths x 64 options)."""
    kind, call, K, B = _book()
    args = dict(n_paths=256 * 200 + 37, n_steps=8, n_obs=4, seed=5)
    ref = ctx.mc_price(SETS, 100.0, 1.0, kind, call, K, 0.03, barrier=B, **args)
    try:
        for cap in ("1", "3000", "20000", "60000"):
            os.environ["DHJ_MC_SCRATCH_ENTRIES"] = cap
            got = ctx.mc_price(SETS, 100.0, 1.0, kind, call, K, 0.03, barrier=B, **args)
            assert np.array_equal(got[0], ref[0]) and np.array_equal(got[1], ref[1]), cap
        M = 64
        kinds = [KINDS[i % 6] for i in range(M)]
        Ks = np.linspace(80.0, 120.0, M)
        Bs = np.where(np.arange(M) % 6 >= 2, np.where(np.arange(M) % 6 < 4, 125.0, 80.0), np.nan)
        big = dict(n_paths=(1 << 24) + 5, n_steps=2, n_obs=2, seed=1)
        os.environ["DHJ_MC_SCRATCH_ENTRIES"] = str(1 << 23)
        whole = ctx.mc_price(SETS[0], 100.0, 0.1, kinds, 1, Ks, 0.03, barrier=Bs, **big)
        del os.environ["DHJ_MC_SCRATCH_ENTRIES"]
        n0 = ctx.launch_count
        split = ctx.mc_price(SETS[0], 100.0, 0.1, kinds, 1, Ks, 0.03, barrier=Bs, **big)
        assert ctx.launch_count - n0 == 4          # two runs of chunks, a path launch and a finalize each
        assert np.array_equal(whole[0], split[0]) and np.array_equal(whole[1], split[1])
    finally:
        os.environ.pop("DHJ_MC_SCRATCH_ENTRIES", None)


def _raw(ctx, params=SETS, P=None, S0=(100.0,), s0_stride=0, T=1.0, n_steps=4, n_obs=2, M=1, kind=(0,), call=(1,),
         strike=(100.0,), barrier=None, n_paths=64):
    import dhj
    params = np.ascontiguousarray(params, dtype=np.float64).reshape(-1, 13)
    P = params.shape[0] if P is None else P
    kind = np.ascontiguousarray(kind, dtype=np.int32)
    call = np.ascontiguousarray(call, dtype=np.int32)
    strike = np.ascontiguousarray(strike, dtype=np.float64)
    bar = None if barrier is None else np.ascontiguousarray(barrier, dtype=np.float64)
    out = np.empty(max(1, P) * max(1, M) * 2)
    return ctx._lib.dhj_mc_price(ctx._h, params, P, np.ascontiguousarray(S0, dtype=np.float64), s0_stride, 0.03, 0.0,
                                 T, n_steps, n_obs, M, kind, call, strike,
                                 None if bar is None else bar.ctypes.data, 0, n_paths, out, None)


def test_argument_errors(ctx):
    """Every DHJ_ERR_ARG case of the header; n_paths = 1 gives stderr NaN; NaN parameters give NaN, not an error."""
    import dhj
    assert _raw(ctx) == 0
    bad = [dict(P=0), dict(M=0), dict(n_steps=0), dict(n_obs=0), dict(n_paths=0), dict(n_steps=6, n_obs=4),
           dict(n_steps=(1 << 28) + 4, n_obs=4), dict(T=0.0), dict(T=-1.0), dict(T=np.inf), dict(T=np.nan),
           dict(kind=(6,)), dict(kind=(-1,)), dict(strike=(-1.0,)), dict(strike=(np.nan,)), dict(strike=(np.inf,)),
           dict(kind=(2,)), dict(kind=(4,), barrier=(0.0,)), dict(kind=(3,), barrier=(-5.0,)),
           dict(kind=(5,), barrier=(np.nan,)), dict(kind=(2,), barrier=(np.inf,)), dict(s0_stride=2),
           dict(M=65, kind=(0,) * 65, call=(1,) * 65, strike=(100.0,) * 65)]
    for b in bad:
        assert _raw(ctx, **b) == -1, b
    assert _raw(ctx, M=64, kind=(0,) * 64, call=(1,) * 64, strike=(100.0,) * 64) == 0
    with pytest.raises(dhj.NativeError, match=r"\(-1\)"):
        ctx.mc_price(SETS, 100.0, 1.0, "up-and-out", 1, 100.0, 0.03)           # barrier option without a barrier
    with pytest.raises(ValueError):
        ctx.mc_price(SETS, 100.0, 1.0, "lookback", 1, 100.0, 0.03)
    price, err = ctx.mc_price(SETS, 100.0, 1.0, "european", 1, 100.0, 0.03, n_paths=1, n_steps=4)
    assert np.all(np.isfinite(price)) and np.all(np.isnan(err))
    for i in range(13):
        p = SETS[:1].copy()
        p[0, i] = np.nan
        price, err = ctx.mc_price(p, 100.0, 1.0, KINDS, 1, 100.0, 0.03, barrier=[np.nan, np.nan, 120, 120, 80, 80],
                                  n_paths=512, n_steps=4)
        assert np.all(np.isnan(price)) and np.all(np.isnan(err)), i


def test_checked_build_mc():
    """The checked build reports no violation and gives the product build's bits (ragged last chunk, split host loop,
    64 options)."""
    import dhj
    kind, call, K, B = _book()
    kinds = [KINDS[i % 6] for i in range(64)]
    Bs = np.where(np.arange(64) % 6 >= 2, np.where(np.arange(64) % 6 < 4, 125.0, 80.0), np.nan)
    outs = []
    for lib in (None, CHECKED):
        c = dhj.Context(0, library=lib)
        res = [c.mc_price(SETS, 100.0, 1.0, kind, call, K, 0.03, barrier=B, n_paths=256 * 9 + 7, n_steps=12, n_obs=3,
                          seed=2)]
        res.append(c.mc_price(SETS[:2], 100.0, 0.5, kinds, 0, np.linspace(80, 120, 64), 0.03, barrier=Bs,
                              n_paths=3000, n_steps=6, seed=4))
        try:
            os.environ["DHJ_MC_SCRATCH_ENTRIES"] = "700"
            res.append(c.mc_price(SETS, 100.0, 1.0, kind, call, K, 0.03, barrier=B, n_paths=256 * 9 + 7, n_steps=12,
                                  n_obs=3, seed=2))
        finally:
            os.environ.pop("DHJ_MC_SCRATCH_ENTRIES", None)
        if lib:
            enabled, counts = c.debug_checks()
            assert enabled and not counts.any(), counts
        outs.append(res)
        c.close()
    for (pa, ea), (pb, eb) in zip(*outs):
        assert np.array_equal(pa, pb) and np.array_equal(ea, eb)
    assert np.array_equal(outs[0][0][0], outs[0][2][0])


def test_double_heston_monte_carlo(ctx):
    """DoubleHeston(...).monte_carlo equals Context.mc_price for the same arguments (default grid ceil(252 T))."""
    sys.path.insert(0, PKG)
    from src.models.double_heston import DoubleHeston
    import dhj
    p = SETS[0]
    for opt, kind, B in (("C", "european", None), ("P", "down-and-in", 90.0), ("call", "asian", None),
                         ("C", "up-and-out", 115.0)):
        m = DoubleHeston(100.0, 98.0, 0.3, 0.03, *p, option_type=opt, q=0.01)
        got = m.monte_carlo(kind, barrier=B, n_paths=5000, n_obs=None, seed=8)
        want = dhj.default_context().mc_price(p, 100.0, 0.3, kind, opt.upper()[0] == "C", 98.0, 0.03, 0.01,
                                              barrier=None if B is None else [B], n_paths=5000, n_steps=76, seed=8)
        assert got[0] == want[0][0, 0] and got[1] == want[1][0, 0]
    m = DoubleHeston(100.0, 98.0, 0.3, 0.03, *p, option_type="C")
    got = m.monte_carlo("asian", n_paths=5000, n_steps=60, n_obs=12, seed=8)
    want = ctx.mc_price(p, 100.0, 0.3, "asian", 1, 98.0, 0.03, n_paths=5000, n_steps=60, n_obs=12, seed=8)
    assert got == (want[0][0, 0], want[1][0, 0])
