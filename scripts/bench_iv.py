"""Implied volatility of COS prices on the device, against the pricing launch that produced them.

    python scripts/bench_iv.py [--out DIR]

1. Kernel time from torch.profiler (CUDA activities; copies excluded) of one `Context.implied_vol_dev` call
   (k_implied_vol) on prices left in HBM by one `Context.price_grid_dev` call, and of that pricing call, after a
   warm-up call of each:
     C2: 1 Mi parameter sets x the 15-option generator grid (calls), N = 128: 15.7 M inversions;
     C3: 1 024 parameter sets x 200 strikes x 20 maturities (calls), N = 256.
2. The solver's evaluations per option on a sample of 20 000 of each shape's prices, from the host emulation of
   dhj_iv.cuh (tests/host_emu/emu_iv.cpp, compiled with g++ into a temporary directory): the device runs the same
   arithmetic up to libm, so the counts are those of the kernel.
3. Host wall time of one `DoubleHeston(...).implied_volatility()` (median of 200 calls after a warm-up).
Prints one JSON object per measurement; the GPU's name and power limit are read in the same run.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
from numpy.ctypeslib import ndpointer

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "option-pricing-ffn-lbfgs_b200"),
                os.path.join(ROOT, "option-pricing-ffn-lbfgs_b200", "src", "models")]

import dhj  # noqa: E402
from oracle import cos_oracle as O  # noqa: E402
from bench_greeks import kernel_times  # noqa: E402
from bench_grad import gpu_info  # noqa: E402


def emulation(tmp):
    out = os.path.join(tmp, "emu_iv.so")
    subprocess.run(["g++", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-I",
                    os.path.join(ROOT, "option-pricing-ffn-lbfgs_b200", "csrc"), "-o", out,
                    os.path.join(ROOT, "tests", "host_emu", "emu_iv.cpp")], check=True)
    lib = ctypes.CDLL(out)
    F, I = ndpointer(np.float64, flags="C_CONTIGUOUS"), ndpointer(np.int32, flags="C_CONTIGUOUS")
    lib.emu_implied_vol.argtypes = [ctypes.c_int64] + [F] * 6 + [I, F, I, I]
    return lib


def iterations(lib, V, K, T, r, n=20000, seed=0):
    """Histogram (list, index = evaluations) and status counts of the solver on a sample of the prices V[P, M]."""
    rng = np.random.default_rng(seed)
    P, M = V.shape
    idx = rng.choice(P * M, min(n, P * M), replace=False)
    m = idx % M
    k = len(idx)
    full = lambda v: np.full(k, float(v))  # noqa: E731
    out, st, it = np.empty(k), np.empty(k, np.int32), np.empty(k, np.int32)
    lib.emu_implied_vol(k, np.ascontiguousarray(V.reshape(-1)[idx]), full(100.0), np.ascontiguousarray(K[m]),
                        np.ascontiguousarray(T[m]), full(r), full(0.0), np.ones(k, np.int32), out, st, it)
    return np.bincount(it[st == 0]).tolist(), np.bincount(st, minlength=5).tolist()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    ctx = dhj.default_context()
    gpu = gpu_info()
    dev = torch.device("cuda", ctx.device)
    rng = np.random.default_rng(0)
    lo, hi = O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1]
    r = 0.03
    shapes = [("C2", 1 << 20, O.GENERATOR_STRIKES_REL, O.GENERATOR_MATURITIES, 128),
              ("C3", 1024, np.linspace(60.0, 140.0, 200), np.linspace(0.1, 2.0, 20), 256)]
    rows = []
    with tempfile.TemporaryDirectory() as tmp:
        emu = emulation(tmp)
        for name, P, strikes, mats, N in shapes:
            params = lo + (hi - lo) * rng.random((P, 13))
            d_params = torch.from_numpy(params).to(dev)
            d_s0 = torch.full((1,), 100.0, dtype=torch.float64, device=dev)
            nK, nT = len(strikes), len(mats)
            d_price = torch.empty((P, nT * nK), dtype=torch.float64, device=dev)
            d_vol = torch.empty_like(d_price)
            d_st = torch.empty((P, nT * nK), dtype=torch.int32, device=dev)
            Kt, Tt = np.tile(strikes, nT), np.repeat(mats, nK)

            def price():
                ctx.price_grid_dev(d_params.data_ptr(), P, d_s0.data_ptr(), 0, strikes, mats, r, 0.0, N, 10.0, False,
                                   True, d_price.data_ptr())

            def invert():
                ctx.implied_vol_dev(d_price.data_ptr(), P, d_s0.data_ptr(), 0, Kt, Tt, True, r, 0.0, d_vol.data_ptr(),
                                    d_st.data_ptr())

            price(); invert()
            torch.cuda.synchronize()
            kp, ki = kernel_times(price), kernel_times(invert)
            st = d_st.cpu().numpy()
            V = d_price.cpu().numpy()
            hist, status = iterations(emu, V, Kt, Tt, r)
            row = {"measure": "kernel", "shape": name, "sets": P, "options": nT * nK, "inversions": P * nT * nK, "N": N,
                   "implied_vol_ms": sum(ki.values()), "pricing_ms": sum(kp.values()),
                   "ratio": sum(ki.values()) / sum(kp.values()), "kernels": {**kp, **ki},
                   "device_status_counts": np.bincount(st.reshape(-1), minlength=5).tolist(),
                   "emulated_iterations_hist": hist, "emulated_sample_status_counts": status,
                   "mean_iterations": float(np.dot(np.arange(len(hist)), hist) / max(1, sum(hist))), "gpu": gpu}
            rows.append(row)
            print(json.dumps(row), flush=True)
            del d_params, d_price, d_vol, d_st
    from double_heston import DoubleHeston
    m = DoubleHeston(100.0, 95.0, 0.5, 0.03, 0.04, 2.5, 0.04, 0.3, -0.7, 0.04, 0.5, 0.04, 0.2, -0.5, 0.15, -0.04, 0.08)
    m.implied_volatility()
    t = []
    for _ in range(200):
        t0 = time.perf_counter()
        m.implied_volatility()
        t.append(time.perf_counter() - t0)
    row = {"measure": "double_heston_implied_volatility", "wall_ms_median": 1e3 * float(np.median(t)),
           "wall_ms_min": 1e3 * float(np.min(t)), "value": float(m.implied_volatility()), "gpu": gpu}
    rows.append(row)
    print(json.dumps(row), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_iv.json"), "w") as fh:
            json.dump(rows, fh, indent=1)


if __name__ == "__main__":
    main()
