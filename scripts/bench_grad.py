"""Forward-difference against analytic gradient, per (f, g) request and end to end.

    python scripts/bench_grad.py [--out DIR] [--reps 20]

1. Per request on the C5 market (15 calls, N = 128) at C = 3, 500 and 30 000 optimiser states: host wall time of
   one `Market.loss_fd` (one launch: 14 loss evaluations per state) and of one `Market.loss_grad` (expand, Jacobian,
   reduce), each call ending in a device synchronise (median of --reps after a warm-up), and the device time of the
   kernels of one request from torch.profiler (a separate pass; CUDA activities only).
2. C5 end to end (10 000 markets x 3 starts, the inputs of test_c5_calibrate_many_10k) both ways: seconds, rounds,
   loss evaluations and the final-loss distribution.
Prints one JSON object per measurement; the GPU's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "option-pricing-ffn-lbfgs_b200")]

import dhj  # noqa: E402
from oracle import cos_oracle as O  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def c5_inputs(ctx, n=10000):
    lo, hi = O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1]
    data = ctx.generate(7, 0, n, 500, lo, hi, 0.9, 100.0, 0.0003, 0.01, 0.02, O.GENERATOR_STRIKES_REL,
                        O.GENERATOR_MATURITIES, 0.03)
    spots, market = data["spots"], data["market"]
    K = np.tile(O.GENERATOR_STRIKES_REL[None, :] * spots[:, None] / 100.0, (1, 3))
    T = np.repeat(O.GENERATOR_MATURITIES, 5)
    return spots, K, T, market, data["loss"]


def kernel_ms(fn):
    """Device time (ms) of the kernels one call of fn launches, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    total_us = 0.0
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and not ev.name.startswith("Memcpy") and not ev.name.startswith("Memset"):
            total_us += ev.device_time
    return total_us / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--skip-e2e", action="store_true")
    args = ap.parse_args()
    ctx = dhj.default_context()
    gpu = gpu_info()
    rows = []
    spots, K, T, market, loss = c5_inputs(ctx)
    x0 = dhj.initial_guesses(spots, K, T, market, 3).reshape(-1, 13)
    mk = ctx.market(spots, 0.03, K, T, np.ones(15), market)
    for C in (3, 500, 30000):
        x = np.ascontiguousarray(x0[:C])
        idx = np.repeat(np.arange(C // 3 + 1, dtype=np.int32), 3)[:C]
        calls = {"fd": lambda: mk.loss_fd(x, 1e-8, market_index=idx),
                 "analytic": lambda: mk.loss_grad(x, market_index=idx)}
        for name, fn in calls.items():
            fn()
            t = []
            for _ in range(args.reps):
                t0 = time.perf_counter()
                fn()
                t.append(time.perf_counter() - t0)
            try:
                kms = kernel_ms(fn)
            except Exception as exc:  # noqa: BLE001  (profiler unavailable: say so, do not guess)
                kms = f"not measured ({type(exc).__name__})"
            row = {"measure": "request", "states": C, "gradient": name, "wall_ms_median": 1e3 * float(np.median(t)),
                   "wall_ms_min": 1e3 * float(np.min(t)), "kernel_ms": kms, "gpu": gpu}
            rows.append(row)
            print(json.dumps(row), flush=True)
    mk.close()
    if not args.skip_e2e:
        x0 = x0.reshape(-1, 3, 13)
        for name in ("fd", "analytic", "fd", "analytic"):          # alternated: the second pair shows the spread
            t0 = time.perf_counter()
            res = dhj.calibrate_many(spots, 0.03, K, T, np.ones(15), market, maxiter=300, multi_start=3, x0=x0,
                                     gradient=name)
            wall = time.perf_counter() - t0
            fl = res["final_loss"]
            row = {"measure": "c5_end_to_end", "gradient": name, "seconds": wall, "rounds": int(res["rounds"]),
                   "evaluations": int(res["evaluations"]),
                   "final_loss_quantiles_5_50_95": [float(v) for v in np.quantile(fl, [0.05, 0.5, 0.95])],
                   "final_over_true_q99": float(np.quantile(fl / loss, 0.99)), "gpu": gpu}
            rows.append(row)
            print(json.dumps(row), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_grad.json"), "w") as fh:
            json.dump(rows, fh, indent=1)


if __name__ == "__main__":
    main()
