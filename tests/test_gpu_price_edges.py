"""The pricing kernels (k_price_batch, k_price_dense) and the fused loss kernel (k_loss_batch) at their structural
edges, against the C oracle (oracle/cos_oracle.c):

* k_price_dense: slices on both sides of the pair / single split of a 32-lane round and of one and two chunks of
  kDenseChunk = 224 strikes; binding strikes (their own pass, (a, b) and jump recurrences) at lane and chunk
  boundaries; a slice where every strike binds; per-set spots and strike rows with q != 0 and L != 10; scale_by_spot;
* k_price_batch: binding strikes at every slice position j = 0..7 (the extra pass reads its rotation steps through
  the pointer shift by jb), several in one slice; launches on both sides of the <true> / <false> choice;
* both kernels where the block-to-block recurrences of the jump term (rotation and Gaussian ratio, exact every kReseed
  = 8 blocks) and of the segment starts carry weight: low-diffusion, jump-dominated sets up to N = 2048;
* bit-identity of an option's price however its slice is composed, where the design says so;
* k_loss_batch at its dispatch edges (run_loss in dhj_abi.cu): 8 vs 9 strikes per slice, 32 vs 33 slices, N != 128,
  per-market rows, several units per block, and the FD counters across growing and shrinking batches.

Every fixture asserts the edge it sits on (which strikes bind, which kernel and which loss path the dispatch rule
picks), so that it cannot drift off it."""
import numpy as np
import pytest

from oracle import cos_oracle as O
from test_gpu_derivative_edges import _assert_binding, _bind_slice, _params
from test_gpu_parity import LOSS_ATOL, PRICE_RTOL

pytestmark = pytest.mark.gpu

BATCH_MAX = 8                 # kBatchMaxStrikes (dhj_batch.cuh): larger slices go to k_price_dense
DENSE_CHUNK = 224             # kDenseChunk (dhj_dense.cuh)
PRICE_ITEMS = 32              # kPriceItems: a fused-loss unit holds at most this many slices
SPLIT_UNITS = 8192            # run_loss: from this many loss evaluations on, the split path
FD_POINTS = 14
COND = 1e-13                  # bound on |price - oracle| / (max(S0, K) max(1, e^b)) where the price is not
                              # relative-accurate (deep out of the money: SURVEY H4, as in test_c3_full_shape_edge)


@pytest.fixture(scope="module")
def ctx():
    import dhj
    c = dhj.Context(0)
    yield c
    c.close()


# ---- dispatch rules, restated -------------------------------------------------------------------------------------
def _max_slice(T):
    return np.unique(np.asarray(T), return_counts=True)[1].max()


def _kernel(T):
    """The pricing kernel launch_price picks for an option list with maturities T."""
    return "batch" if _max_slice(T) <= BATCH_MAX else "dense"


def _loss_path(T, n_units):
    """The path run_loss takes for a price-objective market with maturities T and n_units loss evaluations."""
    fused = _max_slice(T) <= BATCH_MAX and len(np.unique(T)) <= PRICE_ITEMS and n_units < SPLIT_UNITS
    return "fused" if fused else "split"


def _pick_units_per_batch(n_units, items_per_unit, resident_blocks):
    """pick_units_per_batch (dhj_abi.cu)."""
    best, best_cost = 1, None
    for upb in range(max(1, PRICE_ITEMS // items_per_unit), 0, -1):
        blocks = -(-n_units // upb)
        cost = -(-blocks // resident_blocks) * (9 + 10 * (-(-upb * items_per_unit // 4)))
        if best_cost is None or cost < best_cost:
            best, best_cost = upb, cost
    return best


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- the oracle comparison ----------------------------------------------------------------------------------------
def _check(tag, got, params, S0, K, T, call, r, q=0.0, N=128, L=10.0):
    """got against the C oracle: 1e-10 relative, or COND of the conditioning scale.  Returns the oracle's prices."""
    want, ab = O.c_price_batch(params, S0, K, T, call, r, q, N=N, L=L, return_ab=True)
    S0r = np.broadcast_to(np.asarray(S0, dtype=float).reshape(-1, 1), want.shape)
    scale = np.maximum(S0r, np.broadcast_to(K, want.shape)) * np.maximum(1.0, np.exp(ab[..., 1]))
    err = np.abs(got - want)
    ok = (err <= PRICE_RTOL * np.abs(want)) | (err <= COND * scale)
    big = np.abs(want) >= 1e-3 * S0r
    print(f"{tag}: worst |p - oracle| / scale {(err / scale).max():.2e} (bound {COND:.0e}), "
          f"worst relative over prices >= 1e-3 S0 {(err[big] / np.abs(want[big])).max():.2e} (bound {PRICE_RTOL:.0e})")
    assert ok.all(), (np.argwhere(~ok)[:5].tolist(), (err / scale).max())
    return want


# ---- a. k_price_dense at its chunk and lane edges -----------------------------------------------------------------
BIND_DENSE = (0, 31, 32, 63, 64, DENSE_CHUNK - 1, DENSE_CHUNK, 2 * DENSE_CHUNK)   # lane rounds and chunks


def _dense_case(name):
    """(params, S0, K, T, call, r, q, N, L, binding mask)"""
    if name.startswith("n"):                                  # one slice of n strikes, T = 0.5: no binding
        n = int(name[1:])
        K = np.linspace(70.0, 130.0, n)
        return _params(3, 100 + n), 100.0, K, np.full(n, 0.5), np.arange(n) % 2 == 0, 0.03, 0.0, 128, 10.0, \
            np.zeros(n, bool)
    if name.startswith("bind449"):                            # 449 strikes binding at lane and chunk edges
        K, call = _bind_slice(449, BIND_DENSE)
        return _params(3, 8), 100.0, K, np.full(449, 0.05), call, 0.03, 0.0, int(name.split("-")[1]), 10.0, \
            np.isin(np.arange(449), BIND_DENSE)
    if name == "all_bind":                                    # 70 strikes, every one binds
        K = np.concatenate([np.linspace(20.0, 45.0, 35), np.linspace(250.0, 400.0, 35)])
        return _params(3, 9), 100.0, K, np.full(70, 0.02), K < 100.0, 0.03, 0.0, 128, 10.0, np.ones(70, bool)
    if name.startswith("per_set"):                            # per-set spots and strike rows, q != 0, L != 10
        N, L = {"per_set_L8": (128, 8.0), "per_set_L12": (256, 12.0)}[name]
        S0 = np.array([80.0, 100.0, 130.0])
        rel = np.linspace(0.75, 1.3, 65)
        Kp = S0[:, None] * rel[None, :] * (1 + 0.01 * np.random.default_rng(10).standard_normal((3, 65)))
        Kp[:, [0, 64]] = S0[:, None] * np.array([0.3, 3.0])    # binding at both ends of the first slice
        K = np.concatenate([Kp, Kp[:, 1:64:4]], axis=1)         # 65 strikes at T = 0.05, 16 at T = 1
        T = np.concatenate([np.full(65, 0.05), np.full(16, 1.0)])
        mask = np.zeros(81, bool)
        mask[[0, 64]] = True
        return _params(3, 11), S0, K, T, np.arange(81) % 2 == 1, 0.02, 0.015, N, L, mask
    raise KeyError(name)


DENSE_CASES = ["n9", "n31", "n32", "n33", "n63", "n64", "n65", "n223", "n224", "n225", "n448", "n449",
               "bind449-2", "bind449-33", "bind449-128", "bind449-257", "bind449-1000", "all_bind",
               "per_set_L8", "per_set_L12"]


@pytest.mark.parametrize("name", DENSE_CASES)
def test_dense_edges_vs_oracle(ctx, name):
    params, S0, K, T, call, r, q, N, L, mask = _dense_case(name)
    assert _kernel(T) == "dense"
    _assert_binding(params, S0, K, T, r, L, mask)
    got = ctx.price_list(params, S0, K, T, call, r, q, N=N, L=L)
    _check(f"dense {name}", got, params, S0, K, T, call, r, q, N, L)


def test_dense_grid_scale_by_spot(ctx):
    """price_grid(scale_by_spot=True) with 12 strikes per maturity: the dense kernel scales each set's strikes by
    its own spot."""
    rng = np.random.default_rng(12)
    params, spots = _params(6, 12), rng.uniform(80.0, 125.0, 6)
    Ks, Ts = np.linspace(80.0, 120.0, 12), np.array([0.1, 0.5, 1.5])
    assert _kernel(np.repeat(Ts, 12)) == "dense"
    got = ctx.price_grid(params, spots, Ks, Ts, 0.03, 0.01, scale_by_spot=True)
    K = np.tile(Ks[None, :] * spots[:, None] / 100.0, (1, 3))
    _check("dense grid, scale_by_spot", got.reshape(6, -1), params, spots, K, np.repeat(Ts, 12), True, 0.03, 0.01)


# ---- b. k_price_batch binding strikes at every slice position ------------------------------------------------------
BIND_PATTERNS = [(j,) for j in range(8)] + [(1, 6), tuple(range(8))]


def _batch_binding_list():
    """One option list of 17 slices: 8-strike slices with binding strikes at each j = 0..7, at {1, 6} and all 8, and
    slices of 1..7 strikes whose last strike binds; maturities 0.05 - 0.001 i (the widening of K = 30 / 300 binds
    for every generator-range set).  Returns (params, K, T, call, mask)."""
    Ks, calls, Ts, masks = [], [], [], []
    shapes = [(8, p) for p in BIND_PATTERNS] + [(n, (n - 1,)) for n in range(1, 8)]
    for i, (n, pos) in enumerate(shapes):
        K, call = _bind_slice(n, pos)
        Ks.append(K); calls.append(call); Ts.append(np.full(n, 0.05 - 0.001 * i))
        masks.append(np.isin(np.arange(n), pos))
    return _params(3, 13), np.concatenate(Ks), np.concatenate(Ts), np.concatenate(calls), np.concatenate(masks)


@pytest.mark.parametrize("N", [2, 33, 256, 257, 1000, 2048])
def test_batch_binding_positions_vs_oracle(ctx, N):
    params, K, T, call, mask = _batch_binding_list()
    assert _kernel(T) == "batch" and _max_slice(T) == 8
    _assert_binding(params, 100.0, K, T, 0.03, 10.0, mask)
    got = ctx.price_list(params, 100.0, K, T, call, 0.03, 0.01, N=N)
    _check(f"batch binding positions N={N}", got, params, 100.0, K, T, call, 0.03, 0.01, N)


def test_batch_launch_sizes(ctx):
    """k_price_batch<true> (full 32-item batches) for a launch of more than 64 x resident blocks x 32 items, <false>
    (pick_units_per_batch) below: 40 one-strike slices, 2^20 sets; staged in chunks of 131 072 sets (run_price_host),
    5.2 M items per launch, more than any resident count (at most 16 blocks of 128 threads per SM) can put on the
    <false> side.  Rows from the big launch equal the same rows priced alone and in a 1 000-set launch bit for bit,
    and a sample matches the oracle."""
    P, M = 1 << 20, 40
    T = np.linspace(0.02, 2.0, M)
    K = 100.0 * np.exp(0.3 * np.sin(np.arange(M)))
    call = np.arange(M) % 3 != 0
    chunk = 131072
    assert M * chunk > 64 * _sm_count() * 16 * PRICE_ITEMS            # <true> whatever the occupancy
    assert 1000 * M <= 64 * _sm_count() * 1 * PRICE_ITEMS               # <false> whatever the occupancy
    params = _params(P, 14)
    big = ctx.price_list(params, 100.0, K, T, call, 0.03)
    rows = np.array([0, 1, chunk - 1, chunk, 5 * chunk + 17, P - 1])
    for p in rows:
        assert np.array_equal(ctx.price_list(params[p], 100.0, K, T, call, 0.03)[0], big[p]), p
    mid = ctx.price_list(params[chunk - 500:chunk + 500], 100.0, K, T, call, 0.03)
    assert np.array_equal(mid, big[chunk - 500:chunk + 500])
    sample = np.concatenate([rows, np.random.default_rng(14).choice(P, 58, replace=False)])
    _check("batch <true> launch sample", big[sample], params[sample], 100.0, K, T, call, 0.03)


# ---- c. the recurrence family: late blocks that carry weight ------------------------------------------------------
def _rec_params():
    """Low-diffusion (v0 = theta = 3e-4 in both factors), jump-dominated sets: lambda in {1, 3}, mu in {-0.3, 0.25},
    sigma_j in {0.005, 0.02}."""
    rows = []
    for lam in (1.0, 3.0):
        for mu in (-0.3, 0.25):
            for sj in (0.005, 0.02):
                rows.append([3e-4, 2.0, 3e-4, 0.05, -0.5, 3e-4, 1.0, 3e-4, 0.04, -0.3, lam, mu, sj])
    return np.array(rows)


def _rec_case(n):
    """(params, K[P, M], T, call, binding mask): n strikes 70-140 at T = 0.5 and 2 per set, plus two binding
    strikes per maturity placed 0.05 inside each end of the set's own range (a put at b0 - 0.05, a call at
    a0 + 0.05: both in the money, with their own (a, b) 0.05 wider than the regular pass's)."""
    params = _rec_params()
    Ts = (0.5, 2.0)
    K, T, call, mask = [], [], [], []
    for t in Ts:
        a0, b0 = O.truncation_range_vec(params[:, None, :], 100.0, np.full((1, 1), 100.0), np.full((1, 1), t),
                                        0.03)
        K.append(np.concatenate([np.broadcast_to(np.linspace(70.0, 140.0, n), (len(params), n)),
                                 100.0 * np.exp(b0 - 0.05), 100.0 * np.exp(a0 + 0.05)], axis=1))
        T.append(np.full(n + 2, t))
        call.append(np.concatenate([np.arange(n) % 2 == 0, [False, True]]))
        mask.append(np.concatenate([np.zeros(n, bool), [True, True]]))
    return params, np.concatenate(K, axis=1), np.concatenate(T), np.concatenate(call), np.concatenate(mask)


REC_STRIKES = {"batch": 5, "dense": 40}


def _rec_late_weight(n):
    """Per (set, maturity): max over the regular strikes of |p(2048) - p(256)| / S0 (C oracle)."""
    params, K, T, call, mask = _rec_case(n)
    d = np.abs(O.c_price_batch(params, 100.0, K, T, call, 0.03, N=2048)
               - O.c_price_batch(params, 100.0, K, T, call, 0.03, N=256)) / 100.0
    d[:, mask] = 0.0
    return np.stack([d[:, T == t].max(axis=1) for t in np.unique(T)], axis=1)


@pytest.mark.parametrize("kernel", ["batch", "dense"])
@pytest.mark.parametrize("N", [255, 256, 257, 512, 1000, 2048])
def test_recurrence_family_vs_oracle(ctx, kernel, N):
    params, K, T, call, mask = _rec_case(REC_STRIKES[kernel])
    assert _kernel(T) == kernel
    _assert_binding(params, 100.0, K, T, 0.03, 10.0, mask)
    # the blocks beyond k = 256 carry weight in every item (slice of one set): 5e-7 S0 at least (lambda = 1,
    # mu = 0.25 is the weakest), 5 000 times the price tolerance; up to 7e-5 S0
    late = _rec_late_weight(REC_STRIKES[kernel])
    assert (late > 5e-7).all() and late.max() > 1e-5, late
    got = ctx.price_list(params, 100.0, K, T, call, 0.03, N=N)
    _check(f"recurrence family, {kernel} kernel, N={N} (late weight {late.min():.1e}..{late.max():.1e} S0)", got,
           params, 100.0, K, T, call, 0.03, 0.0, N)


# ---- d. bit-identity where the design claims the same bits ----------------------------------------------------------
def _alone(ctx, params, S0, K, T, call, r, q, N, kernel):
    """Each option priced as a one-option slice: through the batch kernel alone, or through the dense kernel next to
    a 9-strike slice at another maturity."""
    out = np.empty((len(params), len(K)))
    for o in range(len(K)):
        if kernel == "batch":
            Ko, To, co = K[o:o + 1], T[o:o + 1], call[o:o + 1]
        else:
            Ko = np.concatenate([[K[o]], np.linspace(90.0, 110.0, 9)])
            To = np.concatenate([[T[o]], np.full(9, T[o] + 1.0)])
            co = np.concatenate([[call[o]], np.ones(9, bool)])
        assert _kernel(To) == kernel
        out[:, o] = ctx.price_list(params, S0, Ko, To, co, r, q, N=N)[:, 0]
    return out


@pytest.mark.parametrize("N", [128, 1000])
def test_dense_slice_composition_bitwise(ctx, N):
    """Each option of the 449-strike binding slice: the same bits inside the slice, inside the reversed slice and
    alone (segment_sums2 equals segment_sums per strike; a price does not depend on its chunk or lane)."""
    params, S0, K, T, call, r, q, N, L, mask = _dense_case(f"bind449-{N}")
    p = ctx.price_list(params, S0, K, T, call, r, q, N=N)
    pr = ctx.price_list(params, S0, K[::-1], T[::-1], call[::-1], r, q, N=N)
    assert np.array_equal(p, pr[:, ::-1])
    assert np.array_equal(p, _alone(ctx, params, S0, K, T, call, r, q, N, "dense"))


@pytest.mark.parametrize("N", [128, 1000])
def test_batch_slice_composition_bitwise(ctx, N):
    """Each option of the binding 8-strike slices: the same bits inside its slice, inside the reversed slice and
    alone; and the batch kernel's price of an option alone agrees with the dense kernel's to 1e-12 relative where it
    is >= 1e-3 S0 (different summation orders)."""
    params, K, T, call, mask = _batch_binding_list()
    sel = slice(0, 80)                                        # the ten 8-strike slices
    K, T, call = K[sel], T[sel], call[sel]
    p = ctx.price_list(params, 100.0, K, T, call, 0.03, N=N)
    pr = ctx.price_list(params, 100.0, K[::-1], T[::-1], call[::-1], 0.03, N=N)
    assert np.array_equal(p, pr[:, ::-1])
    assert np.array_equal(p, _alone(ctx, params, 100.0, K, T, call, 0.03, 0.0, N, "batch"))
    dense = _alone(ctx, params, 100.0, K, T, call, 0.03, 0.0, N, "dense")
    big = p >= 1e-3 * 100.0
    rel = np.abs(dense[big] / p[big] - 1)
    print(f"batch vs dense kernel N={N}: worst relative difference {rel.max():.2e} over {big.sum()} prices")
    assert (rel <= 1e-12).all()


# ---- e. k_loss_batch at its dispatch edges --------------------------------------------------------------------------
def _loss_market(kind, n_mk=1, seed=20):
    """(S0[n_mk], K[n_mk, M], T, call, market[n_mk, M], p_true[n_mk, 13], binding mask) of a price-objective market:
    kind "bind8": an 8-strike slice at T = 0.05 with binding strikes at 1 and 6 (calls and puts), and 5 strikes at
    T = 0.5 and 1; "bind9": the same with a 9-strike first slice; "slices32" / "slices33": 32 / 33 maturities of
    1-3 strikes.  Model prices of generator-range sets with 1 % noise; per-market spots and strike rows."""
    rng = np.random.default_rng(seed)
    if kind.startswith("bind"):
        n = int(kind[4:])
        K1, c1 = _bind_slice(n, (1, 6))
        K = np.concatenate([K1, np.tile([90.0, 95.0, 100.0, 105.0, 110.0], 2)])
        T = np.concatenate([np.full(n, 0.05), np.full(5, 0.5), np.full(5, 1.0)])
        call = np.concatenate([c1, np.arange(10) % 2 == 0])
        mask = np.concatenate([np.isin(np.arange(n), (1, 6)), np.zeros(10, bool)])
    else:
        n_s = int(kind[6:])
        cnt = 1 + np.arange(n_s) % 3
        T = np.repeat(np.linspace(0.1, 2.0, n_s), cnt)
        K = 100.0 + 5.0 * np.concatenate([np.arange(c) - (c - 1) / 2 for c in cnt]) + rng.uniform(-3, 3, len(T))
        call = np.arange(len(T)) % 2 == 0
        mask = np.zeros(len(T), bool)
    S0 = rng.uniform(80.0, 125.0, n_mk) if n_mk > 1 else np.array([100.0])
    Km = K[None, :] * S0[:, None] / 100.0
    p_true = _params(n_mk, seed + 1)
    market = O.c_price_batch(p_true, S0, Km, T, call, 0.03) * (1 + 0.01 * rng.standard_normal((n_mk, len(T))))
    assert (market > 0).all()
    return S0, Km, T, call, market, p_true, mask


def _states(p_true, per, seed, idx=None):
    """per perturbed states per market (x near the market's own set), and their market index."""
    rng = np.random.default_rng(seed)
    idx = np.repeat(np.arange(len(p_true)), per) if idx is None else idx
    return O.inverse_transform_params(p_true)[idx] + 0.02 * rng.standard_normal((len(idx), 13)), idx.astype(np.int32)


def _oracle_loss(x, idx, S0, K, T, call, market, N):
    out = np.empty(len(x))
    for m in np.unique(idx):
        sel = idx == m
        out[sel] = O.c_loss_batch(x[sel], S0[m], 0.03, K[m], T, call, market[m], N=N)
    return out


def _assert_loss(tag, got, want):
    err = np.abs(got - want) / np.maximum(1.0, np.abs(want))
    print(f"{tag}: worst |f - oracle| / max(1, |f|) {err.max():.2e} (bound {LOSS_ATOL:.0e})")
    assert np.array_equal(got == O.SENTINEL, want == O.SENTINEL) and (err <= LOSS_ATOL).all()


LOSS_CASES = [("bind8", 128, "fused"), ("bind9", 128, "split"), ("slices32", 128, "fused"),
              ("slices33", 128, "split"), ("bind8", 33, "fused"), ("bind8", 257, "fused"), ("bind8", 1000, "fused")]


@pytest.mark.parametrize("kind,N,path", LOSS_CASES)
def test_loss_edges_vs_oracle(ctx, kind, N, path):
    """loss_batch and loss_fd of one market against the C oracle; the FD stencil's 14 losses of two states too."""
    S0, K, T, call, market, p_true, mask = _loss_market(kind)
    x, idx = _states(p_true, 6, 21)
    assert _loss_path(T, len(x) * FD_POINTS) == path and _loss_path(T, len(x)) == path
    _assert_binding(O.transform_params(x), S0[0], K[0], T, 0.03, 10.0, mask)
    mk = ctx.market(S0[0], 0.03, K[0], T, call, market[0], N=N)
    f = mk.loss_batch(x)
    _assert_loss(f"{kind} N={N} ({path}) loss_batch", f, _oracle_loss(x, idx, S0, K, T, call, market, N))
    ff, g, f_all = mk.loss_fd(x[:2], want_all=True)
    assert np.array_equal(ff, f[:2])
    pts = np.concatenate([O.fd_stencil(x[c])[0] for c in range(2)])
    want_all = O.c_loss_batch(pts, S0[0], 0.03, K[0], T, call, market[0], N=N).reshape(2, FD_POINTS)
    _assert_loss(f"{kind} N={N} ({path}) loss_fd stencil", f_all, want_all)
    mk.close()


def test_loss_many_markets_rows(ctx):
    """16 markets of the bind8 shape with per-market spots and strike rows, states routed by market_index in shuffled
    order (fused path): against the oracle market by market, and bit-identical to one-market Markets."""
    S0, K, T, call, market, p_true, mask = _loss_market("bind8", 16, seed=22)
    x, idx = _states(p_true, 3, 23)
    perm = np.random.default_rng(24).permutation(len(x))
    x, idx = x[perm], idx[perm]
    assert _loss_path(T, len(x) * FD_POINTS) == "fused"
    for m in range(16):
        _assert_binding(O.transform_params(x[idx == m]), S0[m], K[m], T, 0.03, 10.0, mask)
    mk = ctx.market(S0, 0.03, K, T, call, market)
    f = mk.loss_batch(x, idx)
    _assert_loss("16 markets loss_batch", f, _oracle_loss(x, idx, S0, K, T, call, market, 128))
    ff, g = mk.loss_fd(x, market_index=idx)
    assert np.array_equal(ff, f)
    for m in range(16):
        sel = idx == m
        one = ctx.market(S0[m], 0.03, K[m], T, call, market[m])
        assert np.array_equal(one.loss_batch(x[sel]), f[sel]), m
        f1, g1 = one.loss_fd(x[sel])
        assert np.array_equal(f1, ff[sel]) and np.array_equal(g1, g[sel]), m
        one.close()
    mk.close()


@pytest.mark.parametrize("kind", ["bind8", "slices32"])
def test_loss_batch_composition_bitwise(ctx, kind):
    """One state's loss and FD gradient: the same bits at B = 1, at a B for which pick_units_per_batch puts several
    units into a block (fused), and at a unit count >= 8192 (split path, same batch kernel)."""
    S0, K, T, call, market, p_true, mask = _loss_market(kind)
    n_slices = len(np.unique(T))
    x, _ = _states(np.repeat(p_true, 600, axis=0), 1, 25)
    mk = ctx.market(S0[0], 0.03, K[0], T, call, market[0])
    B_mid = 7000
    if kind == "bind8":                                      # 3 slices: several units per block whatever the occupancy
        assert all(_pick_units_per_batch(B_mid, n_slices, _sm_count() * b) > 1 for b in range(1, 17))
    else:                                                    # 32 slices: one unit per block
        assert _pick_units_per_batch(B_mid, n_slices, 1) == 1
    xs = np.tile(x, (14, 1))                                  # 8 400 states
    assert _loss_path(T, 1) == _loss_path(T, B_mid) == "fused" and _loss_path(T, len(xs)) == "split"
    l1 = mk.loss_batch(xs[:1])
    l_mid = mk.loss_batch(xs[:B_mid])
    l_big = mk.loss_batch(xs)
    assert np.array_equal(l_mid, l_big[:B_mid]) and l1[0] == l_mid[0]
    assert np.array_equal(l_mid[600:1200], l_mid[:600])
    C_mid = 7000 // FD_POINTS                                 # 7 000 units: fused; 600 states = 8 400 units: split
    assert _loss_path(T, C_mid * FD_POINTS) == "fused" and _loss_path(T, 600 * FD_POINTS) == "split"
    f1, g1 = mk.loss_fd(x[:1])
    f_mid, g_mid = mk.loss_fd(x[:C_mid])
    f_big, g_big = mk.loss_fd(x)
    assert np.array_equal(f_mid, f_big[:C_mid]) and np.array_equal(g_mid, g_big[:C_mid])
    assert f1[0] == f_mid[0] and np.array_equal(g1[0], g_mid[0])
    assert np.array_equal(f_big, l_big[:600])
    mk.close()


def test_fd_counters_grow_and_shrink(ctx):
    """The fused FD kernel's per-state counters: consecutive loss_fd calls with B growing past the counter buffer,
    then shrinking, give identical per-state results."""
    S0, K, T, call, market, p_true, mask = _loss_market("bind8")
    x, _ = _states(np.repeat(p_true, 580, axis=0), 1, 26)
    mk = ctx.market(S0[0], 0.03, K[0], T, call, market[0])
    sizes = [1, 3, 40, 200, 580, 100, 7, 1]
    assert all(_loss_path(T, B * FD_POINTS) == "fused" for B in sizes)
    res = [mk.loss_fd(x[:B]) for B in sizes]
    f_ref, g_ref = res[sizes.index(580)]
    for B, (f, g) in zip(sizes, res):
        assert np.array_equal(f, f_ref[:B]) and np.array_equal(g, g_ref[:B]), B
    mk.close()
