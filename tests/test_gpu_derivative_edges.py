"""The derivative kernels at the edges of their shared item loop (chan_items / chan_pass in csrc/dhj_jac.cuh) and of
the host code that feeds them, against the dual-number oracles (tests/jac_oracle.py, tests/greeks_oracle.py,
tests/iv_loss_oracle.py):

* strikes in more than one chunk (kJacChunk = 64 for the Jacobian, kGreeksChunk = 224 for the Greeks), binding
  strikes (their own pass and (a, b)) on both sides of a chunk boundary and in a slice where every strike binds, a
  ragged last block of 32 cosine terms, 40 maturities, per-set spots and strike rows, q != 0 and L != 10;
* bitwise independence of an option's outputs from the other strikes of its slice;
* Market.loss_grad over many markets (the row_index of k_price_jac and of the reductions), with either objective,
  and run_loss_grad cut into more than one launch;
* the synchronous staged chunks of price_jacobian / price_greeks with per-set S0 and strike rows.

Every derivative is defined with the truncation range held at its value for the current inputs (frozen range)."""
import numpy as np
import pytest

import greeks_oracle as G
import iv_loss_oracle as IL
import jac_oracle as J
from oracle import cos_oracle as O
from test_gpu_greeks import TOL as GREEKS_TOL
from test_gpu_iv_calibration import F_TOL as IV_F_TOL, G_TOL as IV_G_TOL
from test_gpu_jacobian import JAC_TOL

pytestmark = pytest.mark.gpu

STAGE_BYTES = 32 << 20                       # kStageChunkBytes (dhj_abi.cu)
P_LIT = np.array([0.04, 2.5, 0.04, 0.3, -0.7, 0.04, 0.5, 0.04, 0.2, -0.5, 0.15, -0.04, 0.08])
EPS = np.finfo(float).eps


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


def _bind_slice(n, positions):
    """(K, call) of one slice of n strikes at S0 = 100: deep in-the-money strikes at `positions` (K = 30 calls and
    K = 300 puts in turn: at T <= 0.05 their +-0.1 widening binds for every generator-range set), near-the-money
    strikes (85-115, calls and puts) elsewhere."""
    K = np.linspace(85.0, 115.0, n)
    call = np.arange(n) % 2 == 0
    far = np.asarray(positions)
    K[far[0::2]], call[far[0::2]] = 30.0, True
    K[far[1::2]], call[far[1::2]] = 300.0, False
    return K, call


def _assert_binding(params, S0, K, T, r, L, want):
    """The strikes that bind are exactly `want` ([M] or [P, M]) for every set: the fixture sits on its edge."""
    got = G.binding(params, S0, K, T, r, L)
    assert np.array_equal(got, np.broadcast_to(want, got.shape)), [np.flatnonzero(g).tolist() for g in got]


# ---- the price Jacobian at the chunk and binding edges ------------------------------------------------------------
BIND_JAC = (0, 63, 64, 65, 128)


def _jac_case(name):
    """(params, S0, K, T, call, r, q, N, L, binding mask or None)"""
    if name.startswith("n"):                                  # one slice of n strikes, T = 0.5: no binding
        n = int(name[1:])
        K = np.linspace(70.0, 130.0, n)
        return _params(3, n), 100.0, K, np.full(n, 0.5), np.arange(n) % 2 == 0, 0.03, 0.0, 128, 10.0, np.zeros(n, bool)
    if name.startswith("bind_edges"):                         # 129 strikes, binding at 0, 63, 64, 65, 128
        N = int(name.split("-")[1])
        K, call = _bind_slice(129, BIND_JAC)
        mask = np.isin(np.arange(129), BIND_JAC)
        return _params(3, 1), 100.0, K, np.full(129, 0.05), call, 0.03, 0.0, N, 10.0, mask
    if name == "all_bind":                                    # 70 strikes, every one binds (two chunks)
        K = np.concatenate([np.linspace(20.0, 45.0, 35), np.linspace(250.0, 400.0, 35)])
        return _params(3, 2), 100.0, K, np.full(70, 0.02), K < 100.0, 0.03, 0.0, 128, 10.0, np.ones(70, bool)
    if name == "slices40":                                    # 40 maturities of 5 strikes, T 0.05-2
        K, T = np.tile(O.GENERATOR_STRIKES_REL, 40), np.repeat(np.linspace(0.05, 2.0, 40), 5)
        return _params(3, 3), 100.0, K, T, np.arange(200) % 3 != 0, 0.03, 0.0, 128, 10.0, None
    if name.startswith("per_set"):                            # per-set spots and strike rows, q != 0, L != 10
        N, L = {"per_set_L8": (128, 8.0), "per_set_L12": (256, 12.0)}[name]
        S0 = np.array([80.0, 100.0, 130.0])
        rel = np.linspace(0.6, 1.45, 65)
        Kp = S0[:, None] * rel[None, :] * (1 + 0.01 * np.random.default_rng(4).standard_normal((3, 65)))
        K = np.concatenate([Kp, Kp[:, ::5]], axis=1)         # 65 strikes at T = 0.1, 13 at T = 1
        T = np.concatenate([np.full(65, 0.1), np.full(13, 1.0)])
        call = np.arange(78) % 2 == 1
        return _params(3, 5), S0, K, T, call, 0.02, 0.015, N, L, None
    raise KeyError(name)


JAC_CASES = ["n63", "n64", "n65", "n128", "n129", "n200", "bind_edges-2", "bind_edges-33", "bind_edges-100",
             "bind_edges-128", "bind_edges-1000", "all_bind", "slices40", "per_set_L8", "per_set_L12"]


@pytest.mark.parametrize("name", JAC_CASES)
def test_price_jacobian_edges_vs_oracle(ctx, name):
    params, S0, K, T, call, r, q, N, L, mask = _jac_case(name)
    if mask is not None:
        _assert_binding(params, S0, K, T, r, L, mask)
    prices, jac = ctx.price_jacobian(params, S0, K, T, call, r, q, N=N, L=L)
    want_p, want_j = J.price_jacobian_batch(params, S0, K, T, call, r, q, N=N, L=L, chunk=1)
    scale = np.abs(want_j).max(axis=1, keepdims=True)
    if name == "all_bind":
        # every strike is deep in the money: the price is intrinsic value to ~1e-10, so some columns are ~1e-10
        # while the terms they are summed from are S0-sized.  The host emulation of the device arithmetic is off the
        # oracle by 5.6e-14 S0 there (7e-4 of the smallest column), so the column scale is floored at 1e-2 S0
        # (an absolute bound of 1e-12 S0); the prices, which a wrong pass would move, keep their 1e-10 S0 pin
        scale = np.maximum(scale, 1e-2 * np.max(S0))
    err = np.abs(jac - want_j) / scale
    print(f"{name}: worst |jac - oracle| / column scale {err.max():.2e}")
    assert err.max() <= JAC_TOL, err.max(axis=(0, 1))
    S0r = np.broadcast_to(np.asarray(S0, dtype=float).reshape(-1, 1), prices.shape)
    assert (np.abs(prices - want_p) <= 1e-10 * S0r).all(), np.abs(prices - want_p).max()
    # the prices that come with the Jacobian are the pricing kernel's to 1e-12 where the price is not tiny
    ref = ctx.price_list(params, S0, K, T, call, r, q, N=N, L=L)
    big = ref >= 1e-3 * S0r
    rel = np.abs(prices / ref - 1)[big]
    print(f"{name}: worst |price - price_list| / price_list {rel.max():.2e} over {big.sum()} prices")
    assert (rel <= 1e-12).all(), rel.max()


def test_price_jacobian_slice_composition_bitwise(ctx):
    """Each option's price and Jacobian row are bit-identical inside the 129-strike slice, alone as a one-option list
    and inside the slice with the strike order reversed."""
    params, S0, K, T, call, r, q, N, L, mask = _jac_case("bind_edges-128")
    p, j = ctx.price_jacobian(params, S0, K, T, call, r, q, N=N, L=L)
    pr, jr = ctx.price_jacobian(params, S0, K[::-1], T[::-1], call[::-1], r, q, N=N, L=L)
    assert np.array_equal(p, pr[:, ::-1]) and np.array_equal(j, jr[:, ::-1])
    for o in range(len(K)):
        p1, j1 = ctx.price_jacobian(params, S0, K[o:o + 1], T[o:o + 1], call[o:o + 1], r, q, N=N, L=L)
        assert np.array_equal(p[:, o:o + 1], p1) and np.array_equal(j[:, o:o + 1], j1), o


# ---- the Greeks at the 224 edge ---------------------------------------------------------------------------------
BIND_GREEKS = (0, 223, 224, 448)


def _greeks_case(name):
    """(params, S0, K, T, call, r, q, N, binding mask or None)"""
    if name.startswith("n"):
        n = int(name[1:])
        K = np.linspace(60.0, 140.0, n)
        return _params(3, n), 100.0, K, np.full(n, 0.5), np.arange(n) % 2 == 0, 0.03, 0.01, 128, np.zeros(n, bool)
    if name.startswith("bind224"):                            # 449 strikes, binding at 0, 223, 224, 448
        N = int(name.split("-")[1])
        K, call = _bind_slice(449, BIND_GREEKS)
        mask = np.isin(np.arange(449), BIND_GREEKS)
        return _params(3, 6), 100.0, K, np.full(449, 0.05), call, 0.03, 0.0, N, mask
    if name == "per_set":                                     # per-set spots and strike rows, 225 strikes at T = 0.05
        S0 = np.array([80.0, 100.0, 130.0])
        rel = np.linspace(0.75, 1.3, 225)
        K = S0[:, None] * rel[None, :]
        K[:, [0, 224]] = S0[:, None] * np.array([0.3, 3.0])    # binding at both ends of the two chunks
        call = rel < 1.0
        mask = np.zeros(225, bool)
        mask[[0, 224]] = True
        return _params(3, 7), S0, K, np.full(225, 0.05), call, 0.02, 0.01, 128, mask
    raise KeyError(name)


GREEKS_CASES = ["n223", "n224", "n225", "n449", "bind224-33", "bind224-128", "bind224-1000", "per_set"]


@pytest.mark.parametrize("name", GREEKS_CASES)
def test_price_greeks_edges_vs_oracle(ctx, name):
    params, S0, K, T, call, r, q, N, mask = _greeks_case(name)
    _assert_binding(params, S0, K, T, r, 10.0, mask)
    prices, greeks = ctx.price_greeks(params, S0, K, T, call, r, q, N=N)
    want_p, want_g = G.greeks_batch(params, S0, K, T, call, r, q, N=N, chunk=1)
    err = np.abs(greeks - want_g) / np.abs(want_g).max(axis=1, keepdims=True)
    print(f"{name}: worst |greek - oracle| / column scale per Greek {err.max(axis=(0, 1))}")
    assert err.max() <= GREEKS_TOL, err.max(axis=(0, 1))
    S0r = np.broadcast_to(np.asarray(S0, dtype=float).reshape(-1, 1), prices.shape)
    assert (np.abs(prices - want_p) <= 1e-10 * S0r).all(), np.abs(prices - want_p).max()


def test_price_greeks_slice_composition_bitwise(ctx):
    """Each option's price and Greeks are bit-identical inside the 449-strike slice, alone as a one-option list and
    inside the slice with the strike order reversed."""
    params, S0, K, T, call, r, q, N, mask = _greeks_case("bind224-128")
    p, g = ctx.price_greeks(params, S0, K, T, call, r, q, N=N)
    pr, gr = ctx.price_greeks(params, S0, K[::-1], T[::-1], call[::-1], r, q, N=N)
    assert np.array_equal(p, pr[:, ::-1]) and np.array_equal(g, gr[:, ::-1])
    for o in range(len(K)):
        p1, g1 = ctx.price_greeks(params, S0, K[o:o + 1], T[o:o + 1], call[o:o + 1], r, q, N=N)
        assert np.array_equal(p[:, o:o + 1], p1) and np.array_equal(g[:, o:o + 1], g1), o


# ---- the analytic loss over many markets ------------------------------------------------------------------------
def _multi_market(ctx, n_mk, per_market):
    """n_mk markets of 15 options (per-market spots 80-130 and strike rows, calls and puts, 2 % noisy model prices);
    per_market perturbed states per market, a Feller-active state (market 1) and a NaN state (market 0), in shuffled
    order.  Returns (S0, r, K, T, call, market, x, market_index)."""
    rng = np.random.default_rng(30 + n_mk)
    S0 = rng.uniform(80.0, 130.0, n_mk)
    T = np.repeat(O.GENERATOR_MATURITIES, 5)
    rel = np.tile(O.GENERATOR_STRIKES_REL, 3) / 100.0
    K = S0[:, None] * rel[None, :] * (1 + 0.01 * rng.standard_normal((n_mk, 15)))
    call = np.arange(15) % 3 != 0
    p_true = P_LIT * (1 + 0.2 * rng.uniform(-1, 1, (n_mk, 13)))
    r = 0.03
    market = ctx.price_list(p_true, S0, K, T, call, r) * (1 + 0.02 * rng.standard_normal((n_mk, 15)))
    assert (market > 0).all()
    x_true = O.inverse_transform_params(p_true)
    idx = np.repeat(np.arange(n_mk), per_market)
    x = x_true[idx] + 0.1 * rng.standard_normal((len(idx), 13))
    feller = x_true[1].copy()
    feller[3] = np.log(0.6)                          # sigma1^2 > 2 kappa1 theta1: the Feller term is active
    nan = x_true[0].copy()
    nan[2] = np.nan
    x = np.vstack([x, feller, nan])
    idx = np.concatenate([idx, [1, 0]])
    perm = rng.permutation(len(idx))
    return S0, r, K, T, call, market, x[perm], idx[perm].astype(np.int32)


def _check_against_oracle(tag, f, g, want_f, want_g, f_tol, g_tol, f_ref=None):
    """Sentinel pattern equal; f within f_tol relative (of f_ref if given, else of the oracle's f), g within g_tol of
    the oracle's |g|inf.  Returns the worst errors."""
    sent = f == O.SENTINEL
    assert np.array_equal(sent, want_f == O.SENTINEL) and (g[sent] == 0).all()
    ok = ~sent
    ferr = np.abs(f[ok] / (want_f[ok] if f_ref is None else f_ref[ok]) - 1).max()
    gerr = (np.abs(g[ok] - want_g[ok]).max(axis=1) / np.abs(want_g[ok]).max(axis=1)).max()
    print(f"{tag}: worst |f - ref| / ref {ferr:.2e}, |g - oracle| / |g|inf {gerr:.2e}")
    assert ferr <= f_tol and gerr <= g_tol, (ferr, gerr)
    return ferr, gerr


def test_loss_grad_many_markets(ctx):
    """Market.loss_grad(x, market_index) over 16 markets: against the oracle market by market, f against loss_batch,
    and each state bit-identical to the same state on a one-market Market built from its own row."""
    S0, r, K, T, call, market, x, idx = _multi_market(ctx, 16, 3)
    mk = ctx.market(S0, r, K, T, call, market)
    f, g = mk.loss_grad(x, idx)
    fl = mk.loss_batch(x, idx)
    assert (f == O.SENTINEL).sum() == 1 and np.isnan(x[f == O.SENTINEL]).any()
    assert (O.feller_penalty(O.transform_params(x[x[:, 3] == np.log(0.6)])) > 0).all()
    want_f, want_g = np.empty_like(f), np.empty_like(g)
    for m in range(16):
        sel = idx == m
        want_f[sel], want_g[sel] = J.loss_grad_batch(x[sel], S0[m], r, K[m], T, call, market[m])
    # f is the device loss (loss_batch), to 1e-12 relative; both are the oracle's to 1e-9
    _check_against_oracle("16 markets, f vs loss_batch", f, g, want_f, want_g, 1e-12, 1e-9, f_ref=fl)
    _check_against_oracle("16 markets, f vs oracle", f, g, want_f, want_g, 1e-9, 1e-9)
    for m in range(16):
        sel = idx == m
        one = ctx.market(S0[m], r, K[m], T, call, market[m])
        f1, g1 = one.loss_grad(x[sel])
        assert np.array_equal(f1, f[sel]) and np.array_equal(g1, g[sel]), m
        one.close()
    mk.close()


def _iv_check(ctx, S0, r, K, T, call, market, x, idx, tag):
    """The IV objective of a multi-market Market against the oracle market by market, and each state bit-identical to
    the same state on a one-market Market of its own row.  Returns the Market (objective "iv")."""
    n_mk = len(S0)
    mk = ctx.market(S0, r, K, T, call, market)
    mvol, st = mk.set_objective("iv")
    f, g = mk.loss_grad(x, idx)
    want_f, want_g = np.empty_like(f), np.zeros_like(g)
    for m in range(n_mk):
        want_mvol, want_st = IL.market_vols(S0[m], r, K[m], T, call, market[m])
        assert np.array_equal(st[m], want_st)
        ok = want_st == 0
        assert np.isnan(mvol[m, ~ok]).all()
        assert np.abs(mvol[m, ok] - want_mvol[ok]).max() <= 1e-12 * want_mvol[ok].max()
        sel = idx == m
        want_f[sel], want_g[sel] = IL.iv_loss_grad_batch(x[sel], S0[m], r, K[m], T, call, market[m], mvol=want_mvol)
    _check_against_oracle(tag, f, g, want_f, want_g, IV_F_TOL, IV_G_TOL)
    assert np.array_equal(f, mk.loss_batch(x, idx))
    for m in range(n_mk):
        sel = idx == m
        one = ctx.market(S0[m], r, K[m], T, call, market[m])
        one.set_objective("iv")
        f1, g1 = one.loss_grad(x[sel])
        assert np.array_equal(f1, f[sel]) and np.array_equal(g1, g[sel]), m
        one.close()
    return mk


def test_iv_loss_grad_many_markets(ctx):
    """The IV objective over 8 markets x 3 states (and a NaN state): loss_grad against the oracle, one-market
    bit-identity, and implied_vols(x, market_index) against the oracle's vols of the same model prices."""
    S0, r, K, T, call, market, x, idx = _multi_market(ctx, 8, 3)
    mk = _iv_check(ctx, S0, r, K, T, call, market, x, idx, "8 markets, IV objective")
    vol, st = mk.implied_vols(x, idx)
    prices = mk.prices(x, idx)
    worst = 0.0
    for b in range(len(x)):
        m = idx[b]
        sig, veg, want_st = IL.implied_vols(prices[b], S0[m], K[m], T, r, call)
        assert np.array_equal(st[b], want_st), b
        for o in np.flatnonzero(want_st == 0):
            bound = 64 * EPS * (sig[o] + prices[b, o] / veg[o])
            worst = max(worst, abs(vol[b, o] - sig[o]) / bound)
            assert abs(vol[b, o] - sig[o]) <= bound, (b, o, vol[b, o], sig[o])
    print(f"implied_vols over 8 markets: worst |vol - oracle| / (64 eps (vol + V / vega)) {worst:.2e}")
    mk.close()


# ---- the loss gradient through the Jacobian's chunks --------------------------------------------------------------
def _chunked_market():
    """One market: 90 strikes at T = 0.02 in descending order (the Jacobian's second chunk holds the 7 lowest, whose
    widening binds: out-of-the-money puts of 2e-6 to 2e-5), 10 strikes at T = 0.25; 1 % noisy model prices.  The set
    is the narrowest-range one of 400 generator draws, so that binding strikes keep an implied vol."""
    p = np.array([0.02613558, 2.87969453, 0.05233965, 0.42570295, -0.77831005, 0.02036183, 0.52444276, 0.039139,
                  0.14679072, -0.58975979, 0.18240007, -0.06447898, 0.04699621])
    K = np.concatenate([np.linspace(120.0, 78.0, 90), np.linspace(90.0, 110.0, 10)])
    T = np.concatenate([np.full(90, 0.02), np.full(10, 0.25)])
    call = K >= 100.0
    mask = np.zeros(100, bool)
    mask[83:90] = True
    return p, 100.0, 0.03, K, T, call, mask


# The binding strikes of this market are out-of-the-money puts of 1.6e-9 to 2e-5, whose prices carry ~2.7e-13 of
# absolute rounding: the price objective weights them by 1 / market^2 and the IV objective by 1 / vega, so f and g
# are conditioned far worse than on the other markets.  The host emulation of the device arithmetic (emu_grad.cpp,
# the kernel's order with the host's libm) is off the oracle by 1.6e-6 (f) and 1.6e-7 (g) on the price objective and
# by 5.9e-6 (f) and 5.7e-6 (g) on the IV objective; the bounds below are those with 5-10x headroom.  A wrong pass or
# row moves f and g by O(1).
CHUNKED_PRICE_TOL = (1e-5, 1e-6)             # (f vs oracle, g vs oracle)
CHUNKED_IV_TOL = (5e-5, 5e-5)


@pytest.mark.parametrize("objective", ["price", "iv"])
def test_loss_grad_through_jacobian_chunks(ctx, objective):
    p, S0, r, K, T, call, mask = _chunked_market()
    _assert_binding(p, S0, K, T, r, 10.0, mask)
    market = O.price_batch(p, S0, K, T, call, r)[0] * (1 + 0.01 * np.random.default_rng(12).standard_normal(100))
    assert (market > 0).all()
    x = O.inverse_transform_params(p)[None, :] + 0.05 * np.random.default_rng(13).standard_normal((3, 13))
    mk = ctx.market(S0, r, K, T, call, market)
    if objective == "price":
        f, g = mk.loss_grad(x)
        want_f, want_g = J.loss_grad_batch(x, S0, r, K, T, call, market)
        _check_against_oracle("100-option market, price objective, f vs loss_batch", f, g, want_f, want_g, 1e-12,
                              CHUNKED_PRICE_TOL[1], f_ref=mk.loss_batch(x))
        _check_against_oracle("100-option market, price objective, f vs oracle", f, g, want_f, want_g,
                              *CHUNKED_PRICE_TOL)
    else:
        mvol, st = mk.set_objective("iv")
        assert (st[0, mask] == 0).all(), st[0, mask]    # the binding strikes are in the objective
        f, g = mk.loss_grad(x)
        want_f, want_g = IL.iv_loss_grad_batch(x, S0, r, K, T, call, market)
        assert (f != O.SENTINEL).all()
        _check_against_oracle("100-option market, IV objective", f, g, want_f, want_g, *CHUNKED_IV_TOL)
    mk.close()


# ---- run_loss_grad in more than one launch ------------------------------------------------------------------------
def test_loss_grad_multi_launch(ctx):
    """The 200 x 20 surface as one market with 2 500 states: run_loss_grad cuts them into launches of
    2^27 // (14 M) states; states on both sides of the cut are bit-identical alone and match the oracle."""
    Ks, Ts = np.linspace(80.0, 120.0, 200), np.linspace(0.25, 2.0, 20)
    K, T = np.tile(Ks, 20), np.repeat(Ts, 200)
    call = K >= 90.0
    M, B = len(K), 2500
    chunk = (1 << 27) // (14 * M)
    n_chunks = -(-B // chunk)
    assert n_chunks == 2
    r = 0.03
    market = ctx.price_list(P_LIT, 100.0, K, T, call, r)[0] * (1 + 0.01 * np.random.default_rng(14).standard_normal(M))
    assert (market > 0).all()
    rng = np.random.default_rng(15)
    x = O.inverse_transform_params(P_LIT)[None, :] + 0.1 * rng.standard_normal((B, 13))
    mk = ctx.market(100.0, r, K, T, call, market)
    n0 = ctx.launch_count
    f, g = mk.loss_grad(x)
    assert ctx.launch_count - n0 == 1 + 3 * n_chunks
    assert (f != O.SENTINEL).all()
    edge = [0, chunk - 1, chunk, B - 1]
    for c in edge:
        f1, g1 = mk.loss_grad(x[c:c + 1])
        assert f1[0] == f[c] and np.array_equal(g1[0], g[c]), c
    fe, ge = mk.loss_grad(x[edge])
    assert np.array_equal(fe, f[edge]) and np.array_equal(ge, g[edge])
    for c in (chunk - 1, chunk):
        want_f, want_g = J.loss_grad_batch(x[c:c + 1], 100.0, r, K, T, call, market)
        _check_against_oracle(f"surface state {c}", f[c:c + 1], g[c:c + 1], want_f, want_g, 1e-9, 1e-9)
    mk.close()


# ---- the synchronous staged chunks with per-set rows ------------------------------------------------------------
def _per_set_rows(P, M, seed):
    rng = np.random.default_rng(seed)
    S0 = rng.uniform(80.0, 130.0, P)
    K = S0[:, None] * np.tile(np.linspace(0.8, 1.2, M // 10), 10)[None, :] * (1 + 0.01 * rng.standard_normal((P, M)))
    T = np.repeat(np.linspace(0.1, 2.0, 10), M // 10)
    return _params(P, seed), S0, K, T, np.arange(M) % 3 != 0


@pytest.mark.parametrize("what", ["jacobian", "greeks"])
def test_staged_chunks_per_set_rows(ctx, what):
    """price_jacobian / price_greeks with per-set S0 and strike rows are cut into three chunks of at most 32 MiB of
    staged rows (params, S0 and the strike row in; prices and derivatives out): the rows equal those of a per-chunk
    call bit for bit, and the rows next to each cut match the oracle."""
    M = 200
    width = 13 if what == "jacobian" else 5
    per_row = 8 * (13 + 1 + M + M + width * M)
    chunk = STAGE_BYTES // per_row
    P = 2 * chunk + 100
    assert -(-P // chunk) == 3
    params, S0, K, T, call = _per_set_rows(P, M, 40)
    run = ctx.price_jacobian if what == "jacobian" else ctx.price_greeks
    n0 = ctx.launch_count
    prices, der = run(params, S0, K, T, call, 0.03, 0.01)
    assert ctx.launch_count - n0 == 3
    for lo in range(0, P, chunk):
        pc, dc = run(params[lo:lo + chunk], S0[lo:lo + chunk], K[lo:lo + chunk], T, call, 0.03, 0.01)
        assert np.array_equal(prices[lo:lo + chunk], pc) and np.array_equal(der[lo:lo + chunk], dc), lo
    rows = np.array([chunk - 1, chunk, 2 * chunk - 1, 2 * chunk])
    if what == "jacobian":
        want_p, want_d = J.price_jacobian_batch(params[rows], S0[rows], K[rows], T, call, 0.03, 0.01)
        tol = JAC_TOL
    else:
        want_p, want_d = G.greeks_batch(params[rows], S0[rows], K[rows], T, call, 0.03, 0.01)
        tol = GREEKS_TOL
    err = np.abs(der[rows] - want_d) / np.abs(want_d).max(axis=1, keepdims=True)
    print(f"{what}, rows at the cuts: worst |d - oracle| / column scale {err.max():.2e}")
    assert err.max() <= tol
    assert (np.abs(prices[rows] - want_p) <= 1e-10 * S0[rows, None]).all()
