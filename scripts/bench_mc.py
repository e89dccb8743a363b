"""Monte Carlo pricing of path-dependent options on the device (dhj_mc_price, csrc/dhj_mc.cuh).

    python scripts/bench_mc.py [--out DIR] [--bias] [--reps R]

Workloads (after one warm-up call of each):
  (a) P = 1 parameter set, 2^24 paths, 252 steps, 252 observations, T = 1, 16 mixed options;
  (b) P = 256 parameter sets from the generator's box (what calibrate_many returns), 2^16 paths each, 63 steps,
      T = 0.25, the same 16 options.
For each: the call's host wall time (median of R synchronous calls; the call ends in a stream synchronise), the kernel
times of k_mc_paths and k_mc_finalize from torch.profiler (CUDA activities) in a run of their own, path-steps per
second of the kernels, the finalize kernel's share, and the FP64 rate: FP64 instructions per step counted from the
SASS of the step loop (static count of the instructions whose line information lies inside the mc_step call of
mc_path; the jump branch, taken with probability ~ lambda dt, is included) times path-steps per second, against the
DFMA instruction rate of dhj_fp64_peak.
--bias: European calls and puts (K = 90, 100, 110) of 16 sets of the generator's box at T = 0.25 and 1, 2^24 paths,
against the COS price (price_list, N = 512) at 64 / 128 / 256 / 512 steps per year: the difference in units of the
standard error that 2^22 paths give (twice that of 2^24).
Prints one JSON object per measurement; the GPU's name and power limit are read in the same run.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "option-pricing-ffn-lbfgs_b200"), os.path.join(ROOT, "scripts")]

import dhj  # noqa: E402
from oracle import cos_oracle as O  # noqa: E402
from bench_greeks import kernel_times  # noqa: E402
from bench_grad import gpu_info  # noqa: E402

LIB = os.path.join(ROOT, "option-pricing-ffn-lbfgs_b200", "lib", "libdhj.so")
MC_SRC = os.path.join(ROOT, "option-pricing-ffn-lbfgs_b200", "csrc", "dhj_mc.cuh")
FP64_OPS = ("DFMA", "DADD", "DMUL", "DSETP", "DMNMX")


def book():
    kind = ["european", "european", "asian", "asian", "up-and-out", "up-and-in", "down-and-out", "down-and-in"] * 2
    call = [1, 0] * 8
    K = [95.0] * 8 + [105.0] * 8
    B = [np.nan] * 4 + [120.0, 120.0, 85.0, 85.0] + [np.nan] * 4 + [130.0, 130.0, 80.0, 80.0]
    return kind, call, K, B


def fp64_per_step():
    """(FP64 instructions, all instructions) of k_mc_paths whose line information lies inside mc_path's call of
    mc_step, from nvdisasm of the library's cubin."""
    call_line = next(i + 1 for i, l in enumerate(open(MC_SRC)) if "mc_step(s, seed, path, step, &st)" in l)
    frame = f'dhj_mc.cuh", line {call_line}'
    with tempfile.TemporaryDirectory() as td:
        subprocess.run(["cuobjdump", "-xelf", "all", LIB], cwd=td, check=True, capture_output=True)
        cubin = next(os.path.join(td, f) for f in sorted(os.listdir(td)) if f.startswith("dhj_abi.") and f.endswith(".cubin"))
        sass = subprocess.run(["nvdisasm", "-gi", cubin], capture_output=True, text=True, check=True).stdout
    fp64 = total = 0
    inside = in_fn = fresh = False
    for line in sass.splitlines():
        if line.startswith("\t.section"):
            in_fn = "k_mc_paths" in line and line.startswith("\t.section\t.text.")
            continue
        if not in_fn:
            continue
        if "//##" in line:               # a run of these lines is one instruction's inline chain, innermost first
            inside = (inside and not fresh) or frame in line
            fresh = False
            continue
        m = re.match(r"\s*/\*[0-9a-f]+\*/\s+(?:@!?U?P\w+\s+)?([A-Z0-9]+)", line)
        if m:
            fresh = True
            if inside:
                total += 1
                fp64 += m.group(1) in FP64_OPS
    return fp64, total


def workload(ctx, name, params, T, n_paths, n_steps, reps, fp64_step, dfma_rate):
    kind, call, K, B = book()
    run = lambda: ctx.mc_price(params, 100.0, T, kind, call, K, 0.03, 0.0, barrier=B, n_paths=n_paths,
                               n_steps=n_steps, seed=1)
    run()
    walls = []
    for _ in range(reps):
        t0 = time.perf_counter()
        run()
        walls.append(time.perf_counter() - t0)
    kt = kernel_times(run)
    paths_ms = sum(v for k, v in kt.items() if "k_mc_paths" in k)
    fin_ms = sum(v for k, v in kt.items() if "k_mc_finalize" in k)
    P = params.reshape(-1, 13).shape[0]
    ps = P * n_paths * n_steps / ((paths_ms + fin_ms) * 1e-3)
    return {"workload": name, "P": P, "n_paths": n_paths, "n_steps": n_steps, "options": len(kind),
            "call_wall_ms_median": 1e3 * float(np.median(walls)), "k_mc_paths_ms": paths_ms,
            "k_mc_finalize_ms": fin_ms, "finalize_share": fin_ms / (paths_ms + fin_ms),
            "path_steps_per_s": ps, "fp64_instr_per_step": fp64_step,
            "fp64_instr_rate_share_of_dfma_peak": fp64_step * ps / dfma_rate}


def bias(ctx):
    rng = np.random.default_rng(17)
    params = rng.uniform(O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1], size=(16, 13))
    K = np.array([90.0, 100.0, 110.0] * 2)
    call = np.array([1, 1, 1, 0, 0, 0])
    rows = []
    for T in (0.25, 1.0):
        cos = ctx.price_list(params, 100.0, K, np.full(6, T), call, O.GENERATOR_RATE, 0.0, N=512)
        for spy in (64, 128, 256, 512):
            steps = max(1, int(round(spy * T)))
            price, err = ctx.mc_price(params, 100.0, T, "european", call, K, O.GENERATOR_RATE, n_paths=1 << 24,
                                      n_steps=steps, seed=123)
            z = (price - cos) / (2.0 * err)            # in units of the 2^22-path standard error
            rows.append({"T": T, "steps_per_year": spy, "n_steps": steps, "mean_d_over_se22": float(z.mean()),
                         "mean_abs_d_over_se22": float(np.abs(z).mean()), "max_abs_d_over_se22": float(np.abs(z).max()),
                         "mean_d": float((price - cos).mean()), "se22_median": float(np.median(2.0 * err)),
                         "d_over_se22": np.round(z, 3).tolist()})
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--bias", action="store_true")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    ctx = dhj.default_context()
    res = [{"gpu": gpu_info()}]
    tflops, _ = ctx.fp64_peak()
    dfma_rate = tflops * 1e12 / 2.0
    fp64, total = fp64_per_step()
    res.append({"fp64_peak_tflops": tflops, "step_fp64_instr": fp64, "step_instr": total})
    rng = np.random.default_rng(0)
    sets = rng.uniform(O.GENERATOR_RANGES[:, 0], O.GENERATOR_RANGES[:, 1], size=(256, 13))
    res.append(workload(ctx, "a", sets[0], 1.0, 1 << 24, 252, args.reps, fp64, dfma_rate))
    res.append(workload(ctx, "b", sets, 0.25, 1 << 16, 63, args.reps, fp64, dfma_rate))
    if args.bias:
        res += bias(ctx)
    for r in res:
        print(json.dumps(r), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_mc.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
