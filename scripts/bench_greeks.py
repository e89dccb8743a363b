"""Greeks in one launch against one pricing launch, on the C2 and C3 shapes.

    python scripts/bench_greeks.py [--out DIR]

1. Kernel time from torch.profiler (CUDA activities; copies excluded) of one `Context.price_greeks` call and of one
   `Context.price_list` call, after a warm-up call of each:
     C2: 1 Mi parameter sets x the 15-option generator grid (calls), N = 128;
     C3: 1 024 parameter sets x 200 strikes x 20 maturities (calls and puts), N = 256.
   Bump-and-revalue needs at least five price_list calls for the same five Greeks (S0 +- h, T + h, r + h, q + h).
2. Host wall time of one `DoubleHeston(...).greeks()` (median of 200 calls after a warm-up).
Prints one JSON object per measurement; the GPU's name and power limit are read in the same run.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "option-pricing-ffn-lbfgs_b200"),
                os.path.join(ROOT, "option-pricing-ffn-lbfgs_b200", "src", "models")]

import dhj  # noqa: E402
from oracle import cos_oracle as O  # noqa: E402
from bench_grad import gpu_info  # noqa: E402


def kernel_times(fn):
    """{kernel name: device ms} of the kernels one call of fn launches, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and not ev.name.startswith("Memcpy") and not ev.name.startswith("Memset"):
            out[ev.name] = out.get(ev.name, 0.0) + ev.device_time / 1e3
    return out


def shapes():
    rng = np.random.default_rng(0)
    lo, hi = O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1]
    c2 = lo + (hi - lo) * rng.random((1 << 20, 13))
    K2, T2 = np.tile(O.GENERATOR_STRIKES_REL, 3), np.repeat(O.GENERATOR_MATURITIES, 5)
    c3 = c2[:1024]
    K3, T3 = np.tile(np.linspace(60.0, 140.0, 200), 20), np.repeat(np.linspace(0.1, 2.0, 20), 200)
    return [("C2", c2, K2, T2, np.ones(15, bool), 128), ("C3", c3, K3, T3, np.arange(4000) % 2 == 0, 256)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ctx = dhj.default_context()
    gpu = gpu_info()
    rows = []
    for name, params, K, T, call, N in shapes():
        calls = {"price_greeks": lambda: ctx.price_greeks(params, 100.0, K, T, call, 0.03, N=N),
                 "price_list": lambda: ctx.price_list(params, 100.0, K, T, call, 0.03, N=N)}
        ms = {}
        for what, fn in calls.items():
            fn()
            t0 = time.perf_counter()
            fn()
            wall = time.perf_counter() - t0
            kt = kernel_times(fn)
            ms[what] = sum(kt.values())
            row = {"measure": "kernel", "shape": name, "call": what, "sets": len(params), "options": len(T), "N": N,
                   "kernel_ms": ms[what], "kernels": kt, "wall_ms": 1e3 * wall, "gpu": gpu}
            rows.append(row)
            print(json.dumps(row), flush=True)
        row = {"measure": "ratio", "shape": name, "greeks_over_price": ms["price_greeks"] / ms["price_list"],
               "acceptance_below": 5.0, "gpu": gpu}
        rows.append(row)
        print(json.dumps(row), flush=True)
    from double_heston import DoubleHeston
    m = DoubleHeston(100.0, 95.0, 0.5, 0.03, 0.04, 2.5, 0.04, 0.3, -0.7, 0.04, 0.5, 0.04, 0.2, -0.5, 0.15, -0.04, 0.08)
    m.greeks()
    t = []
    for _ in range(200):
        t0 = time.perf_counter()
        m.greeks()
        t.append(time.perf_counter() - t0)
    row = {"measure": "double_heston_greeks", "wall_ms_median": 1e3 * float(np.median(t)),
           "wall_ms_min": 1e3 * float(np.min(t)), "gpu": gpu}
    rows.append(row)
    print(json.dumps(row), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_greeks.json"), "w") as fh:
            json.dump(rows, fh, indent=1)


if __name__ == "__main__":
    main()
