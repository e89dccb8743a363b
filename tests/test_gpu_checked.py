"""The kernels under their own checks (lib/libdhj_checked.so = the product sources compiled with -DDHJ_CHECKED).

compute-sanitizer is closed on the B200 pool, so the race / bounds evidence for the warp-synchronous shared-memory
protocol (stages of coefficients handed from the CF lanes to the contraction lanes between two __syncwarp, item
records handed from phase 1 to phase 2) comes from the kernels themselves: every stage carries the epoch it was
written in and the epoch up to which each lane has consumed it; a read before the matching write, a write before the
readers are done, an item used before it was prepared, an index outside a shared array or the caller's output buffer
bumps a device counter (dhj_engine.cuh DHJ_CHECK, dhj_debug_checks).  The checked build must (1) report zero
violations over a workload that reaches every kernel and every rare path (ragged N, strikes with their own (a, b),
puts, more slices than a batch, the fused and the split loss path, the dataset sweep) and (2) produce the same bits as
the product build.
"""
import os

import numpy as np
import pytest

from conftest import PKG
from oracle import cos_oracle as O
from test_gpu_derivative_edges import _bind_slice

pytestmark = pytest.mark.gpu

CHECKED = os.path.join(PKG, "lib", "libdhj_checked.so")


def _workload(ctx):
    rng = np.random.default_rng(77)
    lo, hi = O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1]
    out = {}
    params = rng.uniform(lo, hi, size=(3000, 13))
    spots = rng.uniform(80, 125, size=3000)
    # batch kernel: grid, per-set spots, ragged N, puts
    out["grid"] = ctx.price_grid(params, spots, O.GENERATOR_STRIKES_REL, O.GENERATOR_MATURITIES, 0.03, scale_by_spot=True)
    out["grid_n100"] = ctx.price_grid(params[:500], 100.0, O.GENERATOR_STRIKES_REL, O.GENERATOR_MATURITIES, 0.03, N=100,
                                      is_call=False)
    # binding strikes (own (a, b) passes) in the batch kernel: short maturities, far strikes
    K = np.array([60.0, 80.0, 100.0, 120.0, 150.0, 95.0, 105.0]); T = np.array([0.02, 0.02, 0.02, 0.05, 0.05, 1.0, 1.0])
    out["binding"] = ctx.price_list(params[:400], 100.0, K, T, [1, 0, 1, 0, 1, 1, 0], 0.03)
    # 40 maturities: more slices than one block batch
    out["slices"] = ctx.price_list(params[:50], 100.0, np.full(40, 100.0), np.linspace(0.1, 2.0, 40), np.ones(40), 0.03)
    # dense kernel: regular and binding strikes, two chunks (300 strikes), N = 256
    out["dense"] = ctx.price_grid(params[:64], 100.0, np.linspace(50.0, 150.0, 300), np.array([0.02, 0.25, 1.0]), 0.03, N=256)
    # dense kernel at N = 1000: 449 strikes binding at lane and chunk edges; batch kernel at N = 257: an 8-strike slice
    # binding at 1 and 6 (the extra passes' rotation steps through the pointer shift)
    Kb, cb = _bind_slice(449, (0, 31, 32, 63, 64, 223, 224, 448))
    out["dense_bind"] = ctx.price_list(params[:6], 100.0, Kb, np.full(449, 0.05), cb, 0.03, N=1000)
    Kb, cb = _bind_slice(8, (1, 6))
    out["batch_bind"] = ctx.price_list(params[:200], 100.0, Kb, np.full(8, 0.05), cb, 0.03, N=257)
    # loss: fused kernel (small), split path (large), dense market
    Km = np.tile(O.GENERATOR_STRIKES_REL, 3); Tm = np.repeat(O.GENERATOR_MATURITIES, 5)
    market = out["grid"][0].reshape(-1) * (1 + 0.02 * rng.standard_normal(15))
    mk = ctx.market(float(spots[0]), 0.03, Km * spots[0] / 100.0, Tm, np.ones(15), market)
    x = O.inverse_transform_params(params[:1200]) + 0.05 * rng.standard_normal((1200, 13))
    out["fd_small"] = np.concatenate(mk.loss_fd(x[:40]), axis=None)
    out["fd_large"] = np.concatenate(mk.loss_fd(x), axis=None)
    out["loss"] = mk.loss_batch(x[:700])
    mk.close()
    K2 = np.concatenate([np.linspace(85, 115, 12), [95.0, 100.0, 105.0]]); T2 = np.concatenate([np.full(12, 0.5), np.full(3, 1.0)])
    mk2 = ctx.market(100.0, 0.02, K2, T2, np.ones(15), np.full(15, 5.0))
    out["fd_dense"] = np.concatenate(mk2.loss_fd(x[:20]), axis=None)
    mk2.close()
    # fused loss with 32 maturities (one unit per block); FD on a Market with N = 257
    T32 = np.repeat(np.linspace(0.1, 2.0, 32), 2); K32 = np.tile([95.0, 105.0], 32)
    mk3 = ctx.market(100.0, 0.03, K32, T32, np.arange(64) % 2 == 0, np.full(64, 5.0))
    out["fd_slices32"] = np.concatenate(mk3.loss_fd(x[:30]), axis=None)
    mk3.close()
    mk4 = ctx.market(float(spots[0]), 0.03, Km * spots[0] / 100.0, Tm, np.ones(15), market, N=257)
    out["fd_n257"] = np.concatenate(mk4.loss_fd(x[:40]), axis=None)
    mk4.close()
    # dataset sweep
    g = ctx.generate(3, 250, 2100, 500, lo, hi, 0.9, 100.0, 0.0003, 0.01, 0.02, O.GENERATOR_STRIKES_REL,
                     O.GENERATOR_MATURITIES, 0.03)
    out.update({"gen_" + k: v for k, v in g.items()})
    return out


def test_checked_build_is_clean_and_bit_identical():
    import dhj
    assert os.path.exists(CHECKED), "build it with python __graft_entry__.py build"
    plain = dhj.Context(0)
    enabled, counts = plain.debug_checks()
    assert not enabled and not counts.any()                       # the product build carries no checks
    want = _workload(plain)
    plain.close()
    chk = dhj.Context(0, library=CHECKED)
    enabled, counts = chk.debug_checks()
    assert enabled and not counts.any()
    got = _workload(chk)
    enabled, counts = chk.debug_checks()
    names = ("read-before-write", "write-before-consumed", "shared index", "output index", "item not prepared")
    print("checked build:", dict(zip(names, counts[:5].tolist())), "over", chk.launch_count, "launches")
    assert not counts.any(), dict(zip(names, counts.tolist()))
    chk.close()
    for key in want:
        assert np.array_equal(got[key], want[key], equal_nan=True), key
