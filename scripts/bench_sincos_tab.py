#!/usr/bin/env python3
"""A/B timing of the pricing engine's table-driven sincos (fm::sincos_tab / cos_tab) against the full-quadrant
sincos_ it replaced on the per-cosine-term path.

Builds libdhj twice into a temporary directory, unchanged and with -DDHJ_SINCOS_QUADRANT (sincos_tab and cos_tab
evaluate sincos_ instead: the engine's arithmetic before the table), then times the C2 and C3 workloads of bench.py
(same parameter sets, same launch, L2 flushed by a 256 MiB write before every timed launch, CUDA events) on the two
builds ALTERNATELY, --pairs times, in one process.  Prints one JSON line: per workload and variant the median ms per
launch and the spread (max - min over the repeats), the relative gain of the table, the largest and the median
relative difference of the prices between the two builds, and the card's name and power limit.

Usage (GPU):  python scripts/bench_sincos_tab.py [--pairs 7] [--steps 10] [--out DIR]"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "option-pricing-ffn-lbfgs_b200"))
import bench  # noqa: E402  (workload definitions and parameter sets of the benchmark)

CSRC = os.path.join(ROOT, "option-pricing-ffn-lbfgs_b200", "csrc")
VARIANTS = {"table": "", "quadrant": " -DDHJ_SINCOS_QUADRANT"}


def build(tmp):
    libs = {}
    for name, define in VARIANTS.items():
        out = os.path.join(tmp, f"libdhj_{name}.so")
        done = subprocess.run(["make", "-s", "-C", CSRC, f"OUT={out}", out, f"NVCC=nvcc{define}"],
                              capture_output=True, text=True)
        if done.returncode != 0:
            raise RuntimeError(f"build of the {name} variant failed:\n{done.stderr[-4000:]}")
        libs[name] = out
    return libs


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:  # noqa: BLE001
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": None, "error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=7)
    ap.add_argument("--steps", type=int, default=10, help="timed launches per variant and repeat")
    ap.add_argument("--out", help="directory for the JSON line (default: stdout only)")
    args = ap.parse_args()
    import torch

    import dhj
    tmp = tempfile.mkdtemp(prefix="dhj_sincos_ab_")
    libs = build(tmp)
    ctxs = {name: dhj.Context(0, library=path) for name, path in libs.items()}
    dev = torch.device("cuda", 0)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    result = {"card": card(), "pairs": args.pairs, "steps": args.steps, "workloads": {}}
    for key in ("c2", "c3"):
        wl = bench.WORKLOADS[key]
        P, N, r = wl["P"], wl["N"], wl["r"]
        strikes, mats = np.array(wl["strikes"]), np.array(wl["maturities"])
        d_params = torch.from_numpy(bench.gen_params(P, 20260101)).to(dev)
        d_s0 = torch.full((1,), 100.0, dtype=torch.float64, device=dev)
        outs = {name: torch.empty((P, mats.size, strikes.size), dtype=torch.float64, device=dev) for name in ctxs}

        def launch(name):
            ctxs[name].price_grid_dev(d_params.data_ptr(), P, d_s0.data_ptr(), 0, strikes, mats, r, 0.0, N, 10.0,
                                      False, True, outs[name].data_ptr(), stream)

        def timed(name):
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
            for e0, e1 in ev:
                flush.zero_()
                e0.record()
                launch(name)
                e1.record()
            torch.cuda.synchronize()
            return sum(e0.elapsed_time(e1) for e0, e1 in ev) / args.steps

        for name in ctxs:                                   # warm-up: module load, first launches
            for _ in range(3):
                launch(name)
        torch.cuda.synchronize()
        ms = {name: [] for name in ctxs}
        for i in range(args.pairs):
            order = list(ctxs) if i % 2 == 0 else list(ctxs)[::-1]      # alternate which variant goes first
            for name in order:
                ms[name].append(timed(name))
        a, b = outs["table"].cpu().numpy(), outs["quadrant"].cpu().numpy()
        rel = np.abs(a - b) / np.maximum(np.abs(b), 1e-300)
        med = {name: float(np.median(v)) for name, v in ms.items()}
        result["workloads"][key] = {
            "name": wl["name"],
            "ms_per_launch": {name: {"median": med[name], "spread": float(max(v) - min(v)), "all": v}
                              for name, v in ms.items()},
            "gain": 1.0 - med["table"] / med["quadrant"],
            "paired_gain": [1.0 - t / q for t, q in zip(ms["table"], ms["quadrant"])],
            "prices_rel_diff": {"max": float(rel.max()), "median": float(np.median(rel))},
        }
    line = json.dumps(result)
    print(line, flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_sincos_tab.json"), "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
