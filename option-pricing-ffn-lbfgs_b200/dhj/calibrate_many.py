"""Many independent calibrations at once (BASELINE config C5): every calibration x start is one state of the
batched host optimiser (`BatchLBFGS`, csrc/dhj_lbfgs.cpp), and every optimiser round is ONE launch of the fused
loss / forward-difference kernel over all states that still run (`Market.loss_fd` with a per-state market).

Semantics per market are those of `DoubleHestonJumpCalibrator.calibrate(maxiter, multi_start)`
(/root/reference/src/calibration/lbfgs_calibrator.py:236-336): starts `i % 3` -> literature / perturbed /
ATM-implied initial guess (the perturbed guess draws 13 uniforms from the global NumPy RNG, market by market,
in start order), L-BFGS-B with ftol 1e-9, gtol 1e-6, the strictly lowest final loss wins (first start on ties).
"""
from __future__ import annotations

import time

import numpy as np

import os

from ._native import BatchLBFGS, Context, NativeError, default_context, set_host_threads

PARAM_NAMES = ('v1_0', 'kappa1', 'theta1', 'sigma1', 'rho1', 'v2_0', 'kappa2', 'theta2', 'sigma2', 'rho2',
               'lambda_j', 'mu_j', 'sigma_j')
_LITERATURE = np.array([0.04, 2.5, 0.04, 0.3, -0.7, 0.04, 0.5, 0.04, 0.2, -0.5, 0.15, -0.04, 0.08])


def inverse_transform(p: np.ndarray) -> np.ndarray:
    """Model parameters -> unconstrained x (lbfgs_calibrator.py:89-109), rows of 13."""
    p = np.asarray(p, dtype=np.float64)
    # columns 4, 9 (rho < 0) and 11 (mu_j) are overwritten below: keep them out of the log
    x = np.log(np.where(np.isin(np.arange(13), (4, 9, 11)), 1.0, p))
    x[..., 4] = np.arctanh(np.clip(p[..., 4], -0.999, 0.999))
    x[..., 9] = np.arctanh(np.clip(p[..., 9], -0.999, 0.999))
    x[..., 11] = p[..., 11]
    return x


def transform(x: np.ndarray) -> np.ndarray:
    """Unconstrained x -> model parameters (lbfgs_calibrator.py:62-87)."""
    x = np.asarray(x, dtype=np.float64)
    p = np.exp(x)
    p[..., 4] = np.tanh(x[..., 4])
    p[..., 9] = np.tanh(x[..., 9])
    p[..., 11] = x[..., 11]
    return p


def initial_guesses(spots, strikes, maturities, prices, multi_start=3) -> np.ndarray:
    """x0[n_markets, multi_start, 13] with the reference's three guess types (lbfgs_calibrator.py:179-234).

    Vectorised over markets.  The perturbed guesses (start index % 3 == 1) consume the global NumPy RNG exactly
    as sequential `calibrate` calls would: market-major, then start, then the 13 parameters in dict order, each
    `value * (1 + uniform(-w, w))` with w = 0.15 for rho1, rho2, mu_j and 0.20 otherwise (:202-206)."""
    spots = np.asarray(spots, dtype=np.float64).reshape(-1)
    n = spots.size
    maturities = np.asarray(maturities, dtype=np.float64).reshape(-1)
    strikes = np.broadcast_to(np.asarray(strikes, dtype=np.float64), (n, maturities.size))
    prices = np.asarray(prices, dtype=np.float64).reshape(n, -1)
    p = np.empty((n, multi_start, 13))
    kinds = np.arange(multi_start) % 3
    p[:, kinds == 0] = _LITERATURE
    n1 = int((kinds == 1).sum())
    if n1:
        w = np.where(np.isin(np.arange(13), (4, 9, 11)), 0.15, 0.20)
        draws = np.random.uniform(-w, w, size=(n, n1, 13))                 # same stream order as scalar draws
        pert = _LITERATURE * (1 + draws)
        pert[..., 4] = np.clip(pert[..., 4], -0.95, -0.3)
        pert[..., 9] = np.clip(pert[..., 9], -0.95, -0.3)
        p[:, kinds == 1] = pert
    if (kinds == 2).any():
        ratio = strikes / spots[:, None]
        atm = (ratio > 0.95) & (ratio < 1.05)
        cnt = atm.sum(axis=1)
        with np.errstate(all="ignore"):
            avg_price = np.where(atm, prices, 0.0).sum(axis=1) / cnt
            avg_mat = np.where(atm, maturities[None, :], 0.0).sum(axis=1) / cnt
            iv = np.clip((avg_price / spots) / np.sqrt(avg_mat), 0.01, 0.1)
        iv = np.where(cnt > 0, iv, 0.04)
        g2 = np.empty((n, 13))
        g2[:] = [0.0, 2.0, 0.0, 0.4, -0.6, 0.0, 0.7, 0.0, 0.25, -0.4, 0.12, -0.03, 0.07]
        g2[:, [0, 2, 5, 7]] = iv[:, None]
        p[:, kinds == 2] = g2[:, None, :]
    return inverse_transform(p)


_PIPELINE_MIN_MARKETS = 512         # below this the per-pipeline setup costs more than the overlap returns
_pipeline_contexts: list = []       # second context (own stream and staging) for the second pipeline, made once


def default_pipelines() -> int:
    """Host pipelines for large batches: enough to keep the GPU busy while other pipelines' host optimisers work
    (measured on one B200 with the native lock-step loop, 10 000 markets x 3 starts: 1 pipeline 0.72 s, 2: 0.64,
    4: 0.55, 6: 0.52 — the GPU-side floor is 0.45 s; 1 250 markets: 0.132 / 0.113 / 0.092 / 0.088 s), bounded by this
    process's share of the host's cores (torchrun's LOCAL_WORLD_SIZE ranks share them)."""
    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    ranks_here = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
    return max(1, min(6, cores // (2 * ranks_here)))


def calibrate_many(spots, risk_free_rate, strikes, maturities, is_call, prices, maxiter=300, multi_start=3,
                   x0=None, ctx: Context | None = None, return_all_starts=False, pipelines=None, gradient="fd",
                   objective="price"):
    """Calibrate n markets simultaneously.

    spots[n]; strikes[M] or [n, M]; maturities[M]; is_call[M]; prices[n, M]; optional x0[n, multi_start, 13].
    Returns a dict of arrays: x[n,13], parameters[n,13], final_loss[n], iterations[n], success[n], status[n],
    best_start[n], model_prices[n,M], rounds (launches), seconds; with `return_all_starts` also the per-start
    x / loss / nit / status.

    With `pipelines=k` (default: `default_pipelines()`) and enough markets the set is cut in k parts that run their lock-step loops in k
    threads on k contexts (streams) of the same GPU: while one half's loss launch runs, the other half's host
    optimiser (ask / tell, C++ under a released GIL) works — part of the host share of a round (~20 %) disappears
    from the wall time (10 000 markets: 0.80 -> 0.73 s).  Every optimiser state is independent of the others, so the result does not depend on the split.

    `gradient`: "fd" (default) answers each (f, g) request as the reference does, with scipy's 13 forward differences
    (14 loss evaluations, maxfun 15000 // 14 requests); "analytic" with the exact gradient of the loss (truncation
    range held fixed; one loss evaluation and its Jacobian per request, maxfun 15000 requests as scipy's default
    with a supplied jac).  `evaluations` counts loss evaluations: 14 per request on the FD path, 1 on the analytic.

    `objective`: "price" (default) is the reference's loss; "iv" fits Black–Scholes implied vols (q = 0) instead: per
    market, the mean squared error of the model's implied vols against the quotes' over the quotes that have one,
    + Feller (DESIGN.md §6e; `final_loss` is that objective).  A quote whose implied vol has a status != 0 (e.g. a noised
    price below the intrinsic value) is left out of its market's objective.  The result gains market_vols[n, M] (NaN
    where left out), model_vols[n, M] (at the chosen x) and excluded_quotes[n].  A market with no valid quote is
    dropped before the optimiser runs: its x, parameters, final_loss, model prices and vols are NaN, status is 4
    (the optimiser's "abnormal"), success False and iterations 0; the other markets are unaffected.
    """
    if gradient not in ("fd", "analytic"):
        raise ValueError(f"gradient must be 'fd' or 'analytic' (got {gradient!r})")
    if objective not in ("price", "iv"):
        raise ValueError(f"objective must be 'price' or 'iv' (got {objective!r})")
    t0 = time.time()
    n_all = np.asarray(spots).size
    if pipelines is None:
        pipelines = default_pipelines()
    if pipelines > 1 and ctx is None and n_all >= _PIPELINE_MIN_MARKETS:
        return _calibrate_pipelined(spots, risk_free_rate, strikes, maturities, is_call, prices, maxiter, multi_start,
                                    x0, return_all_starts, t0, int(pipelines), gradient, objective)
    ctx = ctx or default_context()
    spots = np.ascontiguousarray(np.asarray(spots, dtype=np.float64).reshape(-1))
    n = spots.size
    maturities = np.asarray(maturities, dtype=np.float64).reshape(-1)
    prices = np.asarray(prices, dtype=np.float64).reshape(n, maturities.size)
    if x0 is None:
        x0 = initial_guesses(spots, strikes, maturities, prices, multi_start)
    x0 = np.asarray(x0, dtype=np.float64).reshape(n * multi_start, 13)
    iv = objective == "iv"
    market = ctx.market(spots, risk_free_rate, strikes, maturities, is_call, prices)
    if iv:
        try:
            market_vols, market_status = market.set_objective("iv")
        except NativeError:
            # some market has no quote with an implied vol (its objective is undefined): it is dropped and the
            # others run as one batch
            market.close()
            _, st = ctx.implied_vol(prices, spots, strikes, maturities, is_call, risk_free_rate, 0.0,
                                    return_status=True)
            keep = (st == 0).any(axis=1)
            if keep.all():
                raise
            return _with_dropped(spots, risk_free_rate, strikes, maturities, is_call, prices, maxiter, multi_start,
                                 x0.reshape(n, multi_start, 13), ctx, return_all_starts, gradient, keep, t0)
    state_market = np.repeat(np.arange(n, dtype=np.int32), multi_start)
    analytic = gradient == "analytic"
    opt = BatchLBFGS(x0, maxiter=maxiter, ftol=1e-9, gtol=1e-6, maxfun=15000 if analytic else 15000 // 14)
    clock = time.perf_counter
    t_loop0 = clock()
    t_setup = time.time() - t0
    # the lock-step loop (ask -> one loss / FD launch over all running states -> tell) runs natively, GIL released
    if analytic:
        rounds, active_sum, (t_ask, t_loss, t_tell) = opt.minimize_grad(market, state_market)
    else:
        rounds, active_sum, (t_ask, t_loss, t_tell) = opt.minimize_fd(market, state_market, 1e-8)
    t_loop1 = clock()
    xs, fs, nit, nfev, status = opt.result()
    opt.close()
    fs2, xs2 = fs.reshape(n, multi_start), xs.reshape(n, multi_start, 13)
    # strictly lowest loss wins, first start on ties; NaN never wins (lbfgs_calibrator.py:271)
    key = np.where(np.isnan(fs2), np.inf, fs2)
    best = np.argmin(key, axis=1)
    rows = np.arange(n)
    bx = xs2[rows, best]
    model = market.prices(bx, market_index=np.arange(n, dtype=np.int32)) if n else np.empty((0, maturities.size))
    if iv:
        model_vols = market.implied_vols(bx, market_index=np.arange(n, dtype=np.int32))[0]
    market.close()
    out = {
        'x': bx, 'parameters': transform(bx), 'final_loss': fs2[rows, best],
        'iterations': nit.reshape(n, multi_start)[rows, best],
        'status': status.reshape(n, multi_start)[rows, best],
        'success': status.reshape(n, multi_start)[rows, best] <= 1,
        'best_start': best, 'model_prices': model, 'rounds': rounds,
        'evaluations': int(nfev.sum()) * (1 if analytic else 14),
        'seconds': time.time() - t0,
        # where the wall time of the lock-step loop went: device launches incl. copies / host optimiser
        'seconds_loss': t_loss, 'seconds_ask': t_ask, 'seconds_tell': t_tell, 'state_rounds': active_sum,
        'seconds_setup': t_setup, 'seconds_loop': t_loop1 - t_loop0,
    }
    if iv:
        out.update({'market_vols': market_vols, 'model_vols': model_vols,
                    'excluded_quotes': (market_status != 0).sum(axis=1)})
    if return_all_starts:
        out.update({'all_x': xs2, 'all_loss': fs2, 'all_nit': nit.reshape(n, multi_start),
                    'all_status': status.reshape(n, multi_start)})
    return out


def _with_dropped(spots, risk_free_rate, strikes, maturities, is_call, prices, maxiter, multi_start, x0, ctx,
                  return_all_starts, gradient, keep, t0):
    """calibrate_many(objective="iv") when some markets have no valid quote: the others are calibrated as one batch
    and every per-market array is scattered back; the dropped rows are NaN with status 4 (abnormal)."""
    n, M = spots.size, maturities.size
    kept = np.flatnonzero(keep)
    k_all = strikes if np.asarray(strikes).size == M else np.asarray(strikes, dtype=np.float64).reshape(n, M)
    out = {}
    if kept.size:
        sub = calibrate_many(spots[kept], risk_free_rate, k_all if k_all.ndim == 1 else k_all[kept], maturities,
                             is_call, prices[kept], maxiter=maxiter, multi_start=multi_start, x0=x0[kept], ctx=ctx,
                             return_all_starts=return_all_starts, pipelines=1, gradient=gradient, objective="iv")
    else:
        sub = {'rounds': 0, 'evaluations': 0, 'seconds_loss': 0.0, 'seconds_ask': 0.0, 'seconds_tell': 0.0,
               'state_rounds': 0, 'seconds_setup': 0.0, 'seconds_loop': 0.0}
    fill = {'x': (np.nan, (13,)), 'parameters': (np.nan, (13,)), 'final_loss': (np.nan, ()),
            'iterations': (0, ()), 'status': (4, ()), 'success': (False, ()), 'best_start': (0, ()),
            'model_prices': (np.nan, (M,)), 'market_vols': (np.nan, (M,)), 'model_vols': (np.nan, (M,)),
            'excluded_quotes': (M, ())}
    if return_all_starts:
        fill.update({'all_x': (np.nan, (multi_start, 13)), 'all_loss': (np.nan, (multi_start,)),
                     'all_nit': (0, (multi_start,)), 'all_status': (4, (multi_start,))})
    dtypes = {'iterations': np.int32, 'status': np.int32, 'success': bool, 'best_start': np.int64,
              'excluded_quotes': np.int64, 'all_nit': np.int32, 'all_status': np.int32}
    for key, (value, shape) in fill.items():
        dtype = sub[key].dtype if key in sub else dtypes.get(key, np.float64)
        arr = np.full((n,) + shape, value, dtype=dtype)
        if kept.size:
            arr[kept] = sub[key]
        out[key] = arr
    for key, val in sub.items():
        if key not in out:
            out[key] = val
    out['seconds'] = time.time() - t0
    return out


def _calibrate_pipelined(spots, risk_free_rate, strikes, maturities, is_call, prices, maxiter, multi_start, x0,
                         return_all_starts, t0, n_pipes=2, gradient="fd", objective="price"):
    import threading
    spots = np.asarray(spots, dtype=np.float64).reshape(-1)
    n = spots.size
    maturities = np.asarray(maturities, dtype=np.float64).reshape(-1)
    prices = np.asarray(prices, dtype=np.float64).reshape(n, maturities.size)
    strikes = np.asarray(strikes, dtype=np.float64)
    if x0 is None:
        x0 = initial_guesses(spots, strikes, maturities, prices, multi_start)      # ONE draw for all markets
    x0 = np.asarray(x0, dtype=np.float64).reshape(n, multi_start, 13)
    first = default_context()
    while len(_pipeline_contexts) < n_pipes - 1:
        _pipeline_contexts.append(Context(first.device))
    contexts = [first] + _pipeline_contexts[:n_pipes - 1]
    cut = [n * i // n_pipes for i in range(n_pipes + 1)]
    parts, errors = [None] * n_pipes, []

    def work(i):
        lo, hi = cut[i], cut[i + 1]
        try:
            k_local = strikes if strikes.size == maturities.size else strikes.reshape(n, -1)[lo:hi]
            parts[i] = calibrate_many(spots[lo:hi], risk_free_rate, k_local, maturities, is_call, prices[lo:hi],
                                      maxiter=maxiter, multi_start=multi_start, x0=x0[lo:hi], ctx=contexts[i],
                                      return_all_starts=return_all_starts, pipelines=1, gradient=gradient,
                                      objective=objective)
        except BaseException as exc:      # noqa: BLE001  (re-raised in the caller's thread)
            errors.append(exc)

    try:
        cores = len(os.sched_getaffinity(0))
    except AttributeError:
        cores = os.cpu_count() or 1
    # the pipelines' ask / tell loops share this process's part of the host's cores (torchrun's LOCAL_WORLD_SIZE ranks
    # share the host: 2 ranks x 6 pipelines x 5 threads on 32 cores ran 0.68 s where 0.36 s is possible)
    ranks_here = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
    set_host_threads(max(1, cores // (n_pipes * ranks_here)))
    threads = [threading.Thread(target=work, args=(i,)) for i in range(n_pipes)]
    try:
        for t in threads:
            t.start()
        for t in threads:
            t.join()
    finally:
        set_host_threads(0)
    if errors:
        raise errors[0]
    out = {}
    for key, val in parts[0].items():
        if isinstance(val, np.ndarray):
            out[key] = np.concatenate([part[key] for part in parts], axis=0)
    out['rounds'] = max(part['rounds'] for part in parts)
    for key in ('seconds_loss', 'seconds_ask', 'seconds_tell', 'state_rounds', 'seconds_setup', 'seconds_loop'):
        out[key] = [part[key] for part in parts]
    out['launches'] = sum(part['rounds'] for part in parts)
    out['evaluations'] = sum(part['evaluations'] for part in parts)
    out['seconds'] = time.time() - t0
    return out


def calibrate_many_sharded(spots, risk_free_rate, strikes, maturities, is_call, prices, group=None, device=None,
                           **kwargs):
    """One process per GPU: each rank calibrates its contiguous block of markets, results are all-gathered
    (NCCL over NVLink on the GPU box).  Initial guesses are drawn for ALL markets on every rank (same global
    RNG stream everywhere) so the result does not depend on the number of ranks."""
    from .shard import gather_rows, shard_bounds, _dist
    dist = _dist()
    world = dist.get_world_size(group) if dist else 1
    rank = dist.get_rank(group) if dist else 0
    spots = np.asarray(spots, dtype=np.float64).reshape(-1)
    n = spots.size
    maturities = np.asarray(maturities, dtype=np.float64).reshape(-1)
    prices = np.asarray(prices, dtype=np.float64).reshape(n, maturities.size)
    strikes = np.asarray(strikes, dtype=np.float64)
    ms = kwargs.get('multi_start', 3)
    x0 = kwargs.pop('x0', None)
    if x0 is None:
        x0 = initial_guesses(spots, strikes, maturities, prices, ms)
    lo, hi = shard_bounds(n, world, rank)
    k_local = strikes if strikes.size == maturities.size else strikes.reshape(n, -1)[lo:hi]
    local = calibrate_many(spots[lo:hi], risk_free_rate, k_local, maturities, is_call, prices[lo:hi],
                           x0=np.asarray(x0).reshape(n, ms, 13)[lo:hi], **kwargs)
    out = {}
    keys = ('x', 'parameters', 'final_loss', 'iterations', 'status', 'success', 'best_start', 'model_prices')
    if kwargs.get('objective', 'price') == 'iv':                    # forwarded to calibrate_many through **kwargs
        keys += ('market_vols', 'model_vols', 'excluded_quotes')
    for key in keys:
        arr = np.asarray(local[key])
        out[key] = gather_rows(arr.astype(np.float64) if arr.dtype == bool else arr, n, group, device)
    out['success'] = out['success'].astype(bool)
    out['rounds'], out['seconds'] = local['rounds'], local['seconds']
    for key in ('seconds_loss', 'seconds_ask', 'seconds_tell', 'state_rounds', 'evaluations'):
        out[key] = local.get(key)
    return out
