"""The implied-volatility calibration objective against the price objective, per (f, g) request and end to end.

    python scripts/bench_iv_calibration.py [--out DIR] [--reps 20] [--skip-e2e]

1. Per request on the C5 market (15 calls, N = 128) at C = 3, 500 and 30 000 optimiser states, for the price and the
   IV objective and both gradients: host wall time of one `Market.loss_fd` / `Market.loss_grad` ending in a device
   synchronise (median of --reps after a warm-up), and the device time of the kernels of one request from
   torch.profiler (a separate pass; CUDA activities only), in total and per kernel.
2. C5 end to end (10 000 markets x 3 starts, the inputs of scripts/bench_grad.py) for both objectives and both
   gradients in the same run: seconds, rounds, loss evaluations, excluded quotes and the median IV RMSE of the fits.
3. k_iv_residual's registers and spills as built (cuobjdump -res-usage of lib/libdhj.so).
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
sys.path[:0] = [ROOT, os.path.join(ROOT, "option-pricing-ffn-lbfgs_b200"), os.path.join(ROOT, "scripts")]

import dhj  # noqa: E402
from bench_grad import c5_inputs, gpu_info  # noqa: E402


def kernels_ms(fn):
    """{kernel name: device ms} of the kernels one call of fn launches, from torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type.name == "CUDA" and not ev.name.startswith(("Memcpy", "Memset")):
            name = ev.name.split("(")[0].split("<")[0].replace("void ", "").replace("dhj::", "")
            out[name] = out.get(name, 0.0) + ev.device_time / 1e3
    return out


def res_usage():
    lib = os.path.join(ROOT, "option-pricing-ffn-lbfgs_b200", "lib", "libdhj.so")
    try:
        text = subprocess.run(["cuobjdump", "-res-usage", lib], capture_output=True, text=True, timeout=120).stdout
    except (OSError, subprocess.SubprocessError) as exc:
        return f"not measured ({type(exc).__name__})"
    lines = text.splitlines()
    for i, line in enumerate(lines):
        if "k_iv_residual" in line and i + 1 < len(lines):
            return lines[i + 1].strip()
    return "not found"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--skip-e2e", action="store_true")
    args = ap.parse_args()
    ctx = dhj.default_context()
    gpu = gpu_info()
    rows = []

    def emit(row):
        row["gpu"] = gpu
        rows.append(row)
        print(json.dumps(row), flush=True)

    emit({"measure": "k_iv_residual_resources", "cuobjdump": res_usage()})
    spots, K, T, market, loss = c5_inputs(ctx)
    x0 = dhj.initial_guesses(spots, K, T, market, 3).reshape(-1, 13)
    _, st = ctx.implied_vol(market, spots, K, T, np.ones(15), 0.03, 0.0, return_status=True)
    emit({"measure": "c5_excluded_quotes", "quotes": int((st != 0).sum()), "markets": int((st != 0).any(axis=1).sum()),
          "of_quotes": int(st.size)})
    markets = {"price": ctx.market(spots, 0.03, K, T, np.ones(15), market),
               "iv": ctx.market(spots, 0.03, K, T, np.ones(15), market)}
    # every C5 market has valid quotes at this seed (c5_excluded_quotes above counts the quotes left out)
    markets["iv"].set_objective("iv")
    for C in (3, 500, 30000):
        x = np.ascontiguousarray(x0[:C])
        idx = np.repeat(np.arange(C // 3 + 1, dtype=np.int32), 3)[:C]
        for obj, mk in markets.items():
            calls = {"fd": lambda mk=mk: mk.loss_fd(x, 1e-8, market_index=idx),
                     "analytic": lambda mk=mk: mk.loss_grad(x, market_index=idx)}
            for name, fn in calls.items():
                fn()
                t = []
                for _ in range(args.reps):
                    t0 = time.perf_counter()
                    fn()
                    t.append(time.perf_counter() - t0)
                try:
                    per = kernels_ms(fn)
                    kms = sum(per.values())
                except Exception as exc:  # noqa: BLE001  (profiler unavailable: say so, do not guess)
                    per, kms = {}, f"not measured ({type(exc).__name__})"
                emit({"measure": "request", "states": C, "objective": obj, "gradient": name,
                      "wall_ms_median": 1e3 * float(np.median(t)), "wall_ms_min": 1e3 * float(np.min(t)),
                      "kernel_ms": kms, "kernels_ms": per})
    for mk in markets.values():
        mk.close()
    if not args.skip_e2e:
        x0 = x0.reshape(-1, 3, 13)
        iv_mk = ctx.market(spots, 0.03, K, T, np.ones(15), market)
        mvol = iv_mk.set_objective("iv")[0]
        for obj, name in (("price", "fd"), ("iv", "fd"), ("price", "analytic"), ("iv", "analytic"),
                          ("price", "fd"), ("iv", "fd"), ("price", "analytic"), ("iv", "analytic")):
            t0 = time.perf_counter()
            res = dhj.calibrate_many(spots, 0.03, K, T, np.ones(15), market, maxiter=300, multi_start=3, x0=x0,
                                     gradient=name, objective=obj)
            wall = time.perf_counter() - t0
            vols = iv_mk.implied_vols(res["x"], market_index=np.arange(len(spots), dtype=np.int32))[0]
            rmse = np.sqrt(np.nanmean((vols - mvol) ** 2, axis=1))
            emit({"measure": "c5_end_to_end", "objective": obj, "gradient": name, "seconds": wall,
                  "rounds": int(res["rounds"]), "evaluations": int(res["evaluations"]),
                  "iv_rmse_median": float(np.median(rmse)),
                  "final_loss_quantiles_5_50_95": [float(v) for v in np.quantile(res["final_loss"], [0.05, 0.5, 0.95])],
                  "status_counts": np.bincount(res["status"], minlength=5).tolist()})
        iv_mk.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_iv_calibration.json"), "w") as fh:
            json.dump(rows, fh, indent=1)


if __name__ == "__main__":
    main()
