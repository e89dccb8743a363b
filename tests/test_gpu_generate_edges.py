"""The device-resident dataset sweep (csrc/dhj_generate.cuh: k_gen_draws -> pricing kernel -> k_gen_market, driven by
dhj_generate_dev / dhj_generate in dhj_abi.cu) at its structural edges, against the oracle's restatement of the counter
stream (oracle/cos_oracle.py counter_*) and the C pricing oracle:

* grid geometry: 1..32 options, a market tile whose 128 samples do or do not divide by M, even M (row pitch M + 1),
  M = 32 (noise slots up to 23), the batch and the dense pricing kernel with per-sample spots, binding strikes;
* the pricing arguments N, L and r;
* path geometry: paths of 1..500 steps around the 32-step tile of k_gen_draws, ranges that start at a path head,
  inside a tile or at a path's last step, path counts that are not a multiple of the block's 4 warps;
* the 64-bit words of the stream: seeds >= 2^32 (the Philox key's high word) and ranges across 2^32 and 2^40 (the
  counter's high word), produced whole and as ragged shards;
* the host loop of dhj_generate: several chunks over the 3-slot ring, chunks that start inside a path, pinned and
  pageable outputs; the model-only device call; the argument checks.

Every fixture asserts the edge it sits on, so that it cannot drift off it.  Bounds are those of the C4 test
(test_gpu_configs.py): parameters 1e-15 absolute (the same operations), spots 1e-13 relative, noise 1e-13 absolute,
loss 1e-9 absolute; prices 1e-10 relative or COND of the conditioning scale (test_gpu_price_edges.py), for market
prices the same scale times (1 + noise)."""
import ctypes
import re

import numpy as np
import pytest

from oracle import cos_oracle as O
from test_gpu_derivative_edges import _assert_binding
from test_gpu_parity import LOSS_ATOL, PRICE_RTOL
from test_gpu_price_edges import COND, _kernel

pytestmark = pytest.mark.gpu

CHUNK = 131072                # dhj_generate: samples per chunk (less the remainder of whole paths)
SLOTS = 3                     # kSlots (dhj_abi.cu): the ring of staging slots
GEN_WARPS = 4                 # kGenWarps (dhj_generate.cuh): paths per k_gen_draws block
TILE = 32                     # steps drawn per warp round in k_gen_draws
MARKET_BLOCK = 128            # kGenMarketSamples: samples per k_gen_market block
MAX_OPTIONS = 32              # kGenMaxOptions
DHJ_ERR_ARG = -1
PARAMS_ATOL, SPOTS_RTOL, NOISE_ATOL = 1e-15, 1e-13, 1e-13
KEYS = ("params", "spots", "model", "market", "loss")

LO, HI = O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1]
BASE = dict(lo=LO, hi=HI, persistence=0.9, spot0=100.0, ret_mean=0.0003, ret_sd=0.01, noise_sd=0.02,
            strikes_rel=O.GENERATOR_STRIKES_REL, maturities=O.GENERATOR_MATURITIES, r=0.03, N=128, L=10.0)
_ARGS = ("lo", "hi", "persistence", "spot0", "ret_mean", "ret_sd", "noise_sd", "strikes_rel", "maturities", "r")


@pytest.fixture(scope="module")
def ctx():
    import dhj
    c = dhj.Context(0)
    yield c
    c.close()


def _cfg(**over):
    c = dict(BASE, **over)
    c["strikes_rel"] = np.atleast_1d(np.asarray(c["strikes_rel"], dtype=float))
    c["maturities"] = np.atleast_1d(np.asarray(c["maturities"], dtype=float))
    return c


def _M(c):
    return c["strikes_rel"].size * c["maturities"].size


def _host(ctx, seed, first, n, path_len, c, out=None):
    """dhj_generate into host arrays (pageable, or the arrays of `out`)."""
    return ctx.generate(seed, first, n, path_len, *[c[k] for k in _ARGS], N=c["N"], L=c["L"], out=out)


def _dev(ctx, seed, first, n, path_len, c, market=True):
    """dhj_generate_dev into device buffers; returns (host copies, launches).  market=False: the model-only call."""
    import torch
    dev = torch.device("cuda", 0)
    M = _M(c)
    bufs = {k: torch.full(s, np.nan, dtype=torch.float64, device=dev)
            for k, s in (("params", (n, 13)), ("spots", (n,)), ("model", (n, M)), ("market", (n, M)), ("loss", (n,)))}
    n0 = ctx.launch_count
    ctx.generate_dev(seed, first, n, path_len, *[c[k] for k in _ARGS], bufs["params"].data_ptr(),
                     bufs["spots"].data_ptr(), bufs["model"].data_ptr(), bufs["market"].data_ptr() if market else 0,
                     bufs["loss"].data_ptr() if market else 0, torch.cuda.current_stream().cuda_stream,
                     N=c["N"], L=c["L"])
    torch.cuda.synchronize()
    keys = KEYS if market else KEYS[:3]
    return {k: bufs[k].cpu().numpy() for k in keys}, ctx.launch_count - n0


def _oracle(seed, first, n, path_len, c):
    return O.counter_generate(seed, first, n, path_len, r=c["r"], N=c["N"], strikes_rel=c["strikes_rel"],
                              maturities=c["maturities"], L=c["L"], lo=c["lo"], hi=c["hi"],
                              persistence=c["persistence"], spot0=c["spot0"], ret_mean=c["ret_mean"],
                              ret_sd=c["ret_sd"], noise_sd=c["noise_sd"])


def _grid(c, spots):
    """(K[P, M], T[M]) of the sweep's grid at per-sample spots (maturity-major)."""
    K = np.tile(c["strikes_rel"][None, :] * spots[:, None] / 100.0, (1, c["maturities"].size))
    return K, np.repeat(c["maturities"], c["strikes_rel"].size)


def _price_err(got, want, scale, S0):
    """(ok, worst error / scale, worst relative error over prices >= 1e-3 S0) of the price rule of _check."""
    err = np.abs(got - want)
    ok = (err <= PRICE_RTOL * np.abs(want)) | (err <= COND * scale)
    big = np.abs(want) >= 1e-3 * S0[:, None]
    rel = (err[big] / np.abs(want[big])).max() if big.any() else 0.0
    return ok, (err / scale).max(), rel


def _compare(tag, got, seed, first, n, path_len, c):
    """Every output of samples [first, first + n) against the oracle; prints the worst errors next to their bounds and
    returns the oracle's values."""
    want = _oracle(seed, first, n, path_len, c)
    S0 = want["spots"]
    K, T = _grid(c, S0)
    _, b = O.truncation_range_vec(want["params"][:, None, :], S0[:, None], K, T[None, :], c["r"], c["L"])
    scale = np.maximum(S0[:, None], K) * np.maximum(1.0, np.exp(b))
    e_par = np.abs(got["params"] - want["params"]).max()
    e_spot = (np.abs(got["spots"] - S0) / S0).max()
    ok_m, e_m, r_m = _price_err(got["model"], want["model"], scale, S0)
    ok_k, e_k, r_k = _price_err(got["market"], want["market"], scale * (1.0 + want["noise"]), S0)
    with np.errstate(all="ignore"):
        e_noise = np.abs(got["market"] / got["model"] - 1.0 - want["noise"]).max()
    e_loss = np.abs(got["loss"] - want["loss"]).max()
    print(f"{tag}: params {e_par:.1e} (bound {PARAMS_ATOL:.0e}), spots rel {e_spot:.1e} ({SPOTS_RTOL:.0e}), "
          f"model {e_m:.1e} of scale ({COND:.0e}) / {r_m:.1e} rel ({PRICE_RTOL:.0e}), market {e_k:.1e} / {r_k:.1e}, "
          f"noise {e_noise:.1e} ({NOISE_ATOL:.0e}), loss {e_loss:.1e} ({LOSS_ATOL:.0e})")
    assert e_par <= PARAMS_ATOL and e_spot <= SPOTS_RTOL, (e_par, e_spot)
    assert ok_m.all(), (np.argwhere(~ok_m)[:5].tolist(), e_m)
    assert ok_k.all(), (np.argwhere(~ok_k)[:5].tolist(), e_k)
    assert e_noise <= NOISE_ATOL and e_loss <= LOSS_ATOL, (e_noise, e_loss)
    return want


def _slice(d, a, b):
    return {k: v[a:b] for k, v in d.items()}


def _assert_same(a, b, tag=""):
    for k in KEYS:
        if k in a and k in b:
            assert np.array_equal(a[k], b[k]), (tag, k)


# ---- a. grid geometry ------------------------------------------------------------------------------------------------
# (nT, nK, pricing kernel, 128 % M == 0, M even)
GRIDS = [(1, 1, "batch", True, False), (1, 2, "batch", True, True), (3, 1, "batch", False, False),
         (1, 7, "batch", False, False), (1, 8, "batch", True, True), (1, 9, "dense", False, False),
         (3, 5, "batch", False, False), (2, 8, "batch", True, True), (4, 4, "batch", True, True),
         (1, 31, "dense", False, False), (1, 32, "dense", True, True), (32, 1, "batch", True, True),
         (4, 8, "batch", True, True)]


def _grid_cfg(nT, nK):
    if (nT, nK) == (3, 5):                                    # the generator's own grid: the control
        return _cfg()
    Ks = np.linspace(80.0, 120.0, nK) if nK > 1 else [100.0]
    Ts = np.linspace(0.25, 1.5, nT) if nT > 1 else [0.5]
    return _cfg(strikes_rel=Ks, maturities=Ts)


@pytest.mark.parametrize("nT,nK,kernel,divides,even", GRIDS, ids=[f"{g[0]}x{g[1]}" for g in GRIDS])
def test_grid_geometry_vs_oracle(ctx, nT, nK, kernel, divides, even):
    """293 samples (two full 128-sample market tiles and a ragged one) from inside a history, across the next one."""
    c = _grid_cfg(nT, nK)
    M = _M(c)
    _, T = _grid(c, np.array([100.0]))
    assert M == nT * nK <= MAX_OPTIONS and _kernel(T) == kernel
    assert (MARKET_BLOCK % M == 0) == divides and (M % 2 == 0) == even and ((M | 1) != M) == even
    seed, first, n = 1000 + M * 7 + nT, 500 * 3 + 211, 293
    assert n // MARKET_BLOCK == 2 and n % MARKET_BLOCK and first % 500 and (first + n) // 500 > first // 500
    if M == MAX_OPTIONS:
        assert 8 + (M - 1) // 2 == 23                          # the noise's last slot
    got = _host(ctx, seed, first, n, 500, c)
    _compare(f"grid {nT}x{nK} (M={M}, {kernel})", got, seed, first, n, 500, c)


def _binding_grid(kernel):
    """(config, binding mask[M]): K_rel = 30 calls at T = 0.02 among near-the-money strikes."""
    if kernel == "batch":                                     # 8 strikes at T = 0.02 and 1: slice positions 0 and 7
        Ks = np.array([30.0, 93.0, 96.0, 99.0, 102.0, 105.0, 108.0, 30.0])
        c = _cfg(strikes_rel=Ks, maturities=[0.02, 1.0])
        mask = np.concatenate([Ks == 30.0, np.zeros(8, bool)])
    else:                                                     # 20 strikes at T = 0.02: 0, 9 and 19
        Ks = np.linspace(92.0, 108.0, 20)
        Ks[[0, 9, 19]] = 30.0
        c = _cfg(strikes_rel=Ks, maturities=[0.02])
        mask = Ks == 30.0
    return c, mask


@pytest.mark.parametrize("kernel", ["batch", "dense"])
def test_binding_strikes_vs_oracle(ctx, kernel):
    c, mask = _binding_grid(kernel)
    seed, first, n, path_len = 77, 500 * 5 + 400, 293, 500
    got = _host(ctx, seed, first, n, path_len, c)
    K, T = _grid(c, got["spots"])
    assert _kernel(T) == kernel
    _assert_binding(got["params"], got["spots"], K, T, c["r"], c["L"], mask)
    _compare(f"binding grid ({kernel}, M={_M(c)})", got, seed, first, n, path_len, c)


# ---- b. the pricing arguments --------------------------------------------------------------------------------------
# low-diffusion, jump-dominated sets at T = 0.25 and 1: their prices move with N and L well past the bounds
LOW_DIFF = dict(lo=np.array([2e-4, 1.5, 2e-4, 0.03, -0.6, 2e-4, 0.5, 2e-4, 0.03, -0.5, 1.0, -0.3, 0.005]),
                hi=np.array([4e-4, 2.5, 4e-4, 0.06, -0.3, 4e-4, 1.5, 4e-4, 0.05, -0.2, 3.0, 0.25, 0.02]))
PRICING = [(2, 10.0, 0.03, "batch"), (33, 10.0, 0.03, "batch"), (257, 10.0, 0.03, "batch"),
           (1000, 10.0, 0.03, "batch"), (128, 8.0, 0.03, "batch"), (128, 12.0, 0.03, "batch"),
           (128, 10.0, 0.0, "batch"), (128, 10.0, 0.05, "batch"), (257, 8.0, 0.03, "dense"),
           (1000, 12.0, 0.05, "dense")]


@pytest.mark.parametrize("N,L,r,kernel", PRICING, ids=[f"N{p[0]}-L{p[1]:g}-r{p[2]:g}-{p[3]}" for p in PRICING])
def test_pricing_arguments_vs_oracle(ctx, N, L, r, kernel):
    """N, L and r reach the sweep's prices: the oracle at the same (N, L, r) differs from the one at the defaults
    (128, 10, 0.03) by more than 1e5 times the bound somewhere, and the device matches the former."""
    # dense: 12 strikes 92-108, all priced above 1e-9 S0 (at K_rel = 115 a price at the rounding level, 2e-16 S0, can
    # come out as exactly 0, and its market price and loss are then 0 and 0 / 0, as in the reference)
    Ks = O.GENERATOR_STRIKES_REL if kernel == "batch" else np.linspace(92.0, 108.0, 12)
    c = _cfg(maturities=[0.25, 1.0], strikes_rel=Ks, N=N, L=L, r=r, **LOW_DIFF)
    seed, first, n = 4242, 500 * 2 + 333, 300
    assert _kernel(_grid(c, np.array([100.0]))[1]) == kernel
    got = _host(ctx, seed, first, n, 500, c)
    want = _compare(f"pricing N={N} L={L:g} r={r:g} ({kernel})", got, seed, first, n, 500, c)
    default = _oracle(seed, first, n, 500, dict(c, N=128, L=10.0, r=0.03))["model"]
    moved = (np.abs(want["model"] - default) / want["spots"][:, None]).max()
    assert moved > 1e5 * COND, moved


# ---- c. path geometry ----------------------------------------------------------------------------------------------
PATH_LENS = [1, 2, 31, 32, 33, 64, 65, 500]


def _starts(L):
    """first at a path head, inside a 32-step tile and at a path's last step (where the path has them)."""
    s = {"head": 3 * L}
    if L > 2:
        s["tile"] = 3 * L + (37 if L > 40 else L // 2)
    if L > 1:
        s["last"] = 4 * L - 1
    return s


@pytest.mark.parametrize("path_len", PATH_LENS)
def test_path_geometry_vs_oracle(ctx, path_len):
    L = path_len
    seed = 300 + L
    c = _cfg()
    for where, first in _starts(L).items():
        t = first % L
        assert {"head": t == 0, "tile": 0 < t % TILE < TILE - 1 and t < L - 1, "last": t == L - 1}[where], where
        for n in (1, 31, 32, 33, 5 * L + 2):
            paths = (first + n - 1) // L - first // L + 1
            if n == 5 * L + 2:
                assert paths % GEN_WARPS != 0 and paths > GEN_WARPS
            got = _host(ctx, seed, first, n, L, c)
            _compare(f"path_len={L} first at {where} (t={t}) n={n} ({paths} paths)", got, seed, first, n, L, c)


def test_path_exact_invariants(ctx):
    """Device-only identities that hold bit for bit: persistence = 0 gives the path_len = 1 draws, persistence = 1
    repeats each path's head row, ret_sd = 0 gives the sequential product spot0 (1 + ret_mean)^t, noise_sd = 0 gives
    market == model and a zero loss."""
    seed, L, first, n = 41, 65, 65 * 2 + 40, 400
    t = np.arange(first, first + n) % L
    assert t[0] != 0 and (t == 0).sum() >= 5
    c = _cfg()
    raw = _host(ctx, seed, 2 * L, n + 40, 1, c)["params"]              # index 2L.. : every head of the range
    p0 = _host(ctx, seed, first, n, L, _cfg(persistence=0.0))["params"]
    assert np.array_equal(p0, raw[40:])
    p1 = _host(ctx, seed, first, n, L, _cfg(persistence=1.0))["params"]
    heads = (np.arange(first, first + n) // L) * L - 2 * L
    assert np.array_equal(p1, raw[heads])
    s = _host(ctx, seed, first, n, L, _cfg(ret_sd=0.0))["spots"]
    walk = np.empty(L)
    walk[0] = 100.0
    for k in range(1, L):
        walk[k] = walk[k - 1] * (1.0 + 0.0003)
    assert np.array_equal(s, walk[t])
    q = _host(ctx, seed, first, n, L, _cfg(noise_sd=0.0))
    assert np.array_equal(q["market"], q["model"]) and (q["loss"] == 0.0).all()


# ---- d. the 64-bit words of the stream -----------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [2 ** 32 + 7, 2 ** 63 + 5, 2 ** 64 - 1], ids=["2^32+7", "2^63+5", "2^64-1"])
def test_seed_high_word_vs_oracle(ctx, seed):
    assert seed >> 32 != 0 and seed < 2 ** 64
    first, n = 500 * 9 + 420, 700
    c = _cfg()
    got = _host(ctx, seed, first, n, 500, c)
    _compare(f"seed {seed:#x}", got, seed, first, n, 500, c)
    low = _host(ctx, seed & 0xFFFFFFFF, first, n, 500, c)                  # the key's low word alone
    assert (got["params"] != low["params"]).any(axis=1).all()


@pytest.mark.parametrize("edge", [2 ** 32, 2 ** 40], ids=["2^32", "2^40"])
def test_counter_high_word_vs_oracle(ctx, edge):
    """A range across a carry into the counter's high word, with one path straddling it; the same samples as two
    ragged shards cut inside that path are bit-identical."""
    seed, L = 7, 500
    first, n = (edge - 700, 1400) if edge == 2 ** 32 else (edge - 350, 900)
    head = (edge // L) * L
    assert first < head < edge < head + L < first + n                     # the straddling path is in the range
    c = _cfg()
    got = _host(ctx, seed, first, n, L, c)
    _compare(f"counter across {edge:#x}", got, seed, first, n, L, c)
    cut = edge + 17
    a = _host(ctx, seed, first, cut - first, L, c)
    b = _host(ctx, seed, cut, first + n - cut, L, c)
    for k in KEYS:
        assert np.array_equal(np.concatenate([a[k], b[k]]), got[k]), k


# ---- e. the host chunk loop of dhj_generate ----------------------------------------------------------------------
def _chunk(path_len):
    return CHUNK - CHUNK % path_len if path_len < CHUNK else CHUNK


CHUNK_CASES = [(500, 500 * 7 + 123, 4 * 131000 + 12345), (1, 77, 4 * CHUNK + 77), (200000, 123456, 4 * CHUNK + 99)]


def _pinned(n, M):
    """Pinned host outputs, built as bench.py's end-to-end block builds them; the tensors keep the memory alive."""
    import torch
    ts = {k: torch.empty(s, dtype=torch.float64).pin_memory()
          for k, s in (("params", (n, 13)), ("spots", (n,)), ("model", (n, M)), ("market", (n, M)), ("loss", (n,)))}
    assert all(t.is_pinned() for t in ts.values())
    return ts, {k: t.numpy() for k, t in ts.items()}


@pytest.mark.parametrize("path_len,first,n", CHUNK_CASES, ids=[f"path_len={c[0]}" for c in CHUNK_CASES])
def test_host_chunks(ctx, path_len, first, n):
    """Pageable and pinned outputs over at least 4 chunks (the 3-slot ring wraps) equal one generate_dev over the
    range, bit for bit; the oracle on the first and last samples and around every chunk boundary."""
    L, seed = path_len, 555 + path_len
    chunk = _chunk(L)
    n_chunks = -(-n // chunk)
    assert n_chunks >= 4 and n_chunks > SLOTS
    if L > 1:
        assert first % L != 0
    if L > CHUNK:                                             # every chunk after the first starts inside a path
        assert all((first + k * chunk) % L != 0 for k in range(1, n_chunks))
    c = _cfg()
    n0 = ctx.launch_count
    pageable = _host(ctx, seed, first, n, L, c)
    assert ctx.launch_count - n0 == 3 * n_chunks
    keep, pinned_out = _pinned(n, _M(c))
    pinned = _host(ctx, seed, first, n, L, c, out=pinned_out)
    dev, _ = _dev(ctx, seed, first, n, L, c)
    _assert_same(pageable, dev, "pageable")
    _assert_same(pinned, dev, "pinned")
    del keep
    windows = [(0, 1000), (n - 1000, n)]
    windows += [(k * chunk - 1000, min(n, k * chunk + 1000)) for k in range(1, n_chunks)]
    for a, b in windows:
        _compare(f"host chunks path_len={L} samples {a}..{b} (chunk {chunk})", _slice(pageable, a, b), seed,
                 first + a, b - a, L, c)


def test_host_empty_and_single(ctx):
    c = _cfg()
    n0 = ctx.launch_count
    empty = _host(ctx, 5, 1234, 0, 500, c)
    assert ctx.launch_count == n0
    assert {k: v.shape for k, v in empty.items()} == {"params": (0, 13), "spots": (0,), "model": (0, 15),
                                                      "market": (0, 15), "loss": (0,)}
    one = _host(ctx, 5, 1234, 1, 500, c)
    assert ctx.launch_count - n0 == 3
    _compare("host n=1", one, 5, 1234, 1, 500, c)


# ---- f. the model-only device call ---------------------------------------------------------------------------------
@pytest.mark.parametrize("grid", ["3x5", "1x32"])
def test_model_only_generate_dev(ctx, grid):
    """market = loss = NULL: parameters, spots and model prices bit-identical to the full call, one launch fewer."""
    c = _cfg() if grid == "3x5" else _cfg(strikes_rel=np.linspace(80.0, 120.0, 32), maturities=[0.5], N=257)
    seed, L, first, n = 91, 33, 33 * 5 + 9, 1000
    full, n_full = _dev(ctx, seed, first, n, L, c)
    part, n_part = _dev(ctx, seed, first, n, L, c, market=False)
    assert n_full == 3 and n_part == n_full - 1
    _assert_same(part, full, grid)


# ---- g. argument checks ----------------------------------------------------------------------------------------------
def test_grid_size_checks_binding(ctx):
    """Through the binding: a 3 x 11 grid (M = 33) is refused, 4 x 8 (M = 32) accepted; nK = 0, path_len = 0,
    first < 0 and N = 0 are refused; a refused call starts no launch."""
    import dhj
    cases = [(dict(strikes_rel=np.linspace(90.0, 110.0, 11)), {}, "the generator grid must have 1..32 options "
              "(got 3 x 11)"),
             (dict(strikes_rel=np.zeros(0)), {}, "the generator grid must have 1..32 options (got 3 x 0)"),
             ({}, dict(path_len=0), "path_len must be >= 1 (got 0)"),
             ({}, dict(first=-1), "first and n must be >= 0"),
             (dict(N=0), {}, "N must be >= 1 (got 0)")]
    for over, call, message in cases:
        c = _cfg(**over)
        kw = dict(dict(first=0, path_len=500), **call)
        n0 = ctx.launch_count
        with pytest.raises(dhj.NativeError, match=re.escape(message)):
            _host(ctx, 3, kw["first"], 10, kw["path_len"], c)
        assert ctx.launch_count == n0, message
    n0 = ctx.launch_count
    ok = _host(ctx, 3, 0, 10, 500, _cfg(strikes_rel=np.linspace(90.0, 110.0, 8), maturities=[0.25, 0.5, 1.0, 2.0]))
    assert ok["model"].shape == (10, 32) and ctx.launch_count - n0 == 3


def _raw_call(ctx, entry, **over):
    """One direct ctypes call of dhj_generate ("host") or dhj_generate_dev ("dev") with null pointers allowed.
    Returns (rc, message, launches)."""
    import torch
    lib = ctypes.CDLL(ctx._lib._name)
    v = dict(seed=3, first=0, n=10, path_len=500, lo=LO.copy(), hi=HI.copy(), strikes=O.GENERATOR_STRIKES_REL.copy(),
             nK=5, mats=O.GENERATOR_MATURITIES.copy(), nT=3, N=128)
    v.update({k: x for k, x in over.items() if k in v})
    n, M = 10, max(1, v["nK"] * v["nT"])
    shapes = (("params", (n, 13)), ("spots", (n,)), ("model", (n, M)), ("market", (n, M)), ("loss", (n,)))
    if entry == "host":
        outs = {k: np.empty(s) for k, s in shapes}
        ptr = {k: ctypes.c_void_p(a.ctypes.data) for k, a in outs.items()}
    else:
        outs = {k: torch.empty(s, dtype=torch.float64, device=torch.device("cuda", 0)) for k, s in shapes}
        ptr = {k: ctypes.c_void_p(t.data_ptr()) for k, t in outs.items()}
    for k in KEYS:
        if over.get("null") == k:
            ptr[k] = None

    def arr(a):
        return None if a is None else ctypes.c_void_p(a.ctypes.data)
    args = [ctypes.c_void_p(ctx._h.value), ctypes.c_uint64(v["seed"]), ctypes.c_int64(v["first"]),
            ctypes.c_int64(v["n"]), ctypes.c_int32(v["path_len"]), arr(v["lo"]), arr(v["hi"]), ctypes.c_double(0.9),
            ctypes.c_double(100.0), ctypes.c_double(0.0003), ctypes.c_double(0.01), ctypes.c_double(0.02),
            arr(v["strikes"]), ctypes.c_int32(v["nK"]), arr(v["mats"]), ctypes.c_int32(v["nT"]),
            ctypes.c_double(0.03), ctypes.c_int32(v["N"]), ctypes.c_double(10.0)]
    args += [ptr[k] for k in KEYS]
    if entry == "dev":
        args.append(None)
    fn = lib.dhj_generate if entry == "host" else lib.dhj_generate_dev
    fn.restype = ctypes.c_int
    n0 = ctx.launch_count
    rc = fn(*args)
    if entry == "dev":
        torch.cuda.synchronize()
    msg = ctx._lib.dhj_last_error(ctx._h).decode()
    return rc, msg, ctx.launch_count - n0


_RAW_CASES = [
    ("M33", dict(strikes=np.linspace(90.0, 110.0, 11), nK=11), "the generator grid must have 1..32 options "
     "(got 3 x 11)", ("host", "dev")),
    ("nK0", dict(nK=0), "the generator grid must have 1..32 options (got 3 x 0)", ("host", "dev")),
    ("path_len0", dict(path_len=0), "path_len must be >= 1 (got 0)", ("host", "dev")),
    ("first_neg", dict(first=-1), "first and n must be >= 0", ("host", "dev")),
    ("n_neg", dict(n=-1), "first and n must be >= 0", ("host", "dev")),
    ("N0", dict(N=0), "N must be >= 1 (got 0)", ("host", "dev")),
    ("null_lo", dict(lo=None), "null table", ("host", "dev")),
    ("null_strikes", dict(strikes=None), "null table", ("host", "dev")),
    ("null_maturities", dict(mats=None), "null table", ("host", "dev")),
    ("market_without_loss", dict(null="loss"), "market and loss outputs come together (both or neither)", ("dev",)),
    ("null_output", dict(null="market"), "null output array", ("host",)),
]
RAW = [(case, entry, over, message) for case, over, message, entries in _RAW_CASES for entry in entries]


@pytest.mark.parametrize("case,entry,over,message", RAW, ids=[f"{r[0]}-{r[1]}" for r in RAW])
def test_argument_checks_raw(ctx, case, entry, over, message):
    """Direct calls: each refused with DHJ_ERR_ARG and its message, before any launch."""
    rc, msg, launches = _raw_call(ctx, entry, **over)
    assert rc == DHJ_ERR_ARG and msg == message and launches == 0, (rc, msg, launches)


@pytest.mark.parametrize("entry", ["host", "dev"])
def test_argument_checks_raw_accepts_32(ctx, entry):
    """The same direct call with a 4 x 8 grid (M = 32) runs: the refusals above are the checks' doing."""
    rc, msg, launches = _raw_call(ctx, entry, strikes=np.linspace(90.0, 110.0, 8), nK=8,
                                  mats=np.array([0.25, 0.5, 1.0, 2.0]), nT=4)
    assert rc == 0 and launches == 3, (rc, msg)
