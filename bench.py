#!/usr/bin/env python3
"""bench.py — COS option prices per second (N=128, FP64) on B200, and the reference CPU path beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload c1|c2|c3|c4|c5]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Default workload (BASELINE.json configs[1], "C2"): 1 048 576 random parameter sets in the generator's ranges
(src/data/synthetic_generator.py:75-89 of the reference) x the 15-option grid (5 strikes x 3 maturities),
S0 = 100, r = 0.03, calls, COS N = 128, float64.  One "step" = one pass of the pricing kernel over that
batch.  With N GPUs every rank prices its own, differently seeded, batch of the same size (weak scaling; the
path shards by parameter set with no data-path collective — SURVEY §8e).

Numbers on the JSON line:
  value        prices/s over all ranks, inputs resident in HBM, CUDA-event time of the K steps (max over ranks),
               L2 flushed between steps (untimed);
  e2e          the same metric through the host-buffer C-ABI call (`dhj_price_grid` via `dhj.Context.price_grid`):
               pinned host params in, pinned host prices out, H2D and D2H inside the timed region;
  roofline     bound "fp64" (vector pipe: SURVEY §8d, DESIGN §3).  `achieved` / `frac` are PHYSICAL: FP64 issue
               slots the kernel executes (warp-level DFMA/DMUL/DADD/DSETP instructions per price, from the ncu
               capture of THIS build recorded in profiles/ncu_summary.json — refused as stale if the kernel
               sources changed since) x 2 flop x 32 lanes, against the DFMA peak of this GPU (`dhj_fp64_peak`
               probe, nominal 148 SM x 64 FMA/clk x 2 x clock beside it); <= 1 by construction.  The SURVEY §8d
               contract figure (the reference's formulas: one sincos per strike and k) is kept as
               `achieved_contract` / `frac_contract`; the kernel's recurrences execute fewer flops than that, so it
               exceeds 1.  `hbm` carries the (irrelevant: compute-bound) HBM figure;
  cpu_baseline the UNMODIFIED reference (`DoubleHeston.pricing` from baseline/_ref, installed by
               `__graft_entry__.build()` with pip from /root/reference) on all host cores, bounded sample
               (`kind: "reference"`); the oracle's scalar port only if baseline/_ref is absent (`kind: "port"`);
  calibration  second half of BASELINE.json's metric: seconds per README calibration through the drop-in class, and
               the reference's `compute_loss` timed on this box along its own recorded seed-0 trajectory
               (extrapolated to the 3 206 evaluations of that run; `--workload c1 --impl reference` runs it whole);
  latency      microseconds per `DoubleHeston(...).pricing()` (new strike / maturity on every call) and per
               `compute_loss` through the drop-in classes;
  extra        (default workload, unless --no-extra) the two configs whose scaling is NOT trivially linear, measured
               in the same run so that they appear at every N of the driver's scaling sweep: `c4` — the 100 M-sample
               dataset sweep, STRONG scaling, generated / priced / noised on the device (`dhj_generate_dev`), the
               per-sample losses all-gathered over NCCL inside the timed region; `c5` — 10 000 multi-start-3
               calibrations through `calibrate_many_sharded`, result gather inside the timed region.
`--impl reference` times only the CPU path and prints the same line shape.
`--workload c3|c4|c5|c1` make those configs the headline of the line instead (same keys).
`--steps K` is the number of timed steps of the headline workload (calibrations for c1 / c5); `e2e` and `extra` state
their own step counts.
`--dump-outputs DIR` writes, after the timed steps, what the headline's last timed step returned to its caller as
DIR/<name>.npy (float64, rank 0): c2 / c3 `prices`; c4 `params`, `spots`, `model`, `market`, `loss`; c5 the arrays of
`calibrate_many_sharded`; c1 `parameters`, `model_prices`, `final_loss` of the last calibration.  Outputs larger than
DUMP_BYTES are cut to the same fixed, seeded sample of rows in every array.  The inputs depend on the arguments only,
so two builds run with the same arguments can be compared array for array.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "option-pricing-ffn-lbfgs_b200")
REF_DIR = os.path.join(ROOT, "baseline", "_ref")
sys.path.insert(0, ROOT)
sys.path.insert(0, PKG)

METRIC = "COS option prices/sec (N=128, FP64)"
UNIT = "prices/s"
# SURVEY §8d: FLOP per price = N * (F_CF / nK + F_PAY), F_CF = 1707, F_PAY = 94
F_CF, F_PAY = 1707.0, 94.0
NOMINAL_FP64_TFLOPS = 148 * 64 * 2 * 1.965e9 / 1e12
GRID_K = [90.0, 95.0, 100.0, 105.0, 110.0]
GRID_T = [0.25, 0.5, 1.0]

WORKLOADS = {
    "c1": dict(kind="calibration",
               name="C1: README calibration, 15 options (5K x 3T), N=128, 13 parameters, multi_start=3, maxiter=300"),
    "c2": dict(kind="price", P=1 << 20, strikes=GRID_K, maturities=GRID_T, N=128, r=0.03,
               name="C2: 1Mi random parameter sets x 15-option grid (5K x 3T), N=128, S0=100, r=0.03, calls"),
    "c3": dict(kind="price", P=1024, strikes=list(np.linspace(80.0, 120.0, 200)),
               maturities=list(np.linspace(0.25, 2.0, 20)), N=256, r=0.03,
               name="C3: dense surface 200K x 20T, N=256, 1024 parameter sets per launch"),
    "c4": dict(kind="sweep", P=100_000_000, strikes=GRID_K, maturities=GRID_T, N=128, r=0.03,
               name="C4: synthetic_generator dataset, 100M samples x 15 options (K = K_rel*spot/100), N=128, "
                    "sharded by history (500 samples) over the ranks, counter stream seed 7"),
    "c5": dict(kind="calibrations", markets=10000, starts=3, N=128, r=0.03,
               name="C5: 10 000 independent 15-option multi-start-3 calibrations (maxiter=300), markets = first "
                    "10 000 samples of the C4 dataset, sharded by market over the ranks"),
}

# sampling ranges of the reference's generator (src/data/synthetic_generator.py:75-89)
PARAM_RANGES = np.array([
    (0.025, 0.080), (1.5, 4.5), (0.025, 0.065), (0.20, 0.50), (-0.85, -0.40),
    (0.020, 0.070), (0.30, 1.20), (0.025, 0.070), (0.10, 0.35), (-0.70, -0.20),
    (0.05, 0.25), (-0.08, -0.01), (0.03, 0.12)])
GEN = dict(path_len=500, lo=PARAM_RANGES[:, 0], hi=PARAM_RANGES[:, 1], persistence=0.9, spot0=100.0, ret_mean=0.0003,
           ret_sd=0.01, noise_sd=0.02, strikes_rel=np.array(GRID_K), maturities=np.array(GRID_T), r=0.03)
C4_SEED = 7


def flop_per_price(nK: int, N: int) -> float:
    return N * (F_CF / nK + F_PAY)


def gen_params(P: int, seed: int) -> np.ndarray:
    rng = np.random.default_rng(seed)
    return rng.uniform(PARAM_RANGES[:, 0], PARAM_RANGES[:, 1], size=(P, 13))


def kernel_source_sha() -> str:
    """sha256 over the DEVICE sources (kernels, device math, tables; not the host side of the ABI): ties
    profiles/ncu_summary.json to the build it was captured from."""
    h = hashlib.sha256()
    csrc = os.path.join(PKG, "csrc")
    for f in sorted(os.listdir(csrc)):
        if f.endswith((".cuh", ".inc")):
            h.update(f.encode())
            h.update(open(os.path.join(csrc, f), "rb").read())
    return h.hexdigest()[:16]


DUMP_BYTES = 60 << 20          # --dump-outputs writes at most this much array data (64 MB with room for .npy headers)


def output_sample(arrays: dict, budget: int = DUMP_BYTES, seed: int = 0) -> dict:
    """float64 NumPy copies of `arrays` (NumPy arrays or torch tensors with the same number of rows): whole if they
    fit `budget` bytes, else the same seeded sample of rows, in row order, from each."""
    n = len(next(iter(arrays.values())))
    row_bytes = 8 * sum(int(np.prod(a.shape[1:])) for a in arrays.values())
    keep = budget // max(1, row_bytes)
    idx = None if n <= keep else np.sort(np.random.default_rng(seed).choice(n, size=keep, replace=False))
    out = {}
    for name, a in arrays.items():
        if isinstance(a, np.ndarray):
            a = a if idx is None else a[idx]
        else:                                                   # torch tensor: gather the rows where they live
            import torch
            a = (a if idx is None else a[torch.from_numpy(idx).to(a.device)]).cpu().numpy()
        out[name] = np.ascontiguousarray(a, dtype=np.float64)
    return out


def write_outputs(path: str, arrays: dict) -> None:
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}.npy"), a)


# ------------------------------------------------------------------------------------------------
# CPU path: the unmodified reference from baseline/_ref (else the oracle's scalar port), all cores
# ------------------------------------------------------------------------------------------------
def reference_available() -> bool:
    return os.path.exists(os.path.join(REF_DIR, "src", "models", "double_heston.py"))


def _import_reference():
    """The reference's own modules, imported the way the reference imports them (top-level, sys.path hack:
    lbfgs_calibrator.py:16-18), from the unmodified install under baseline/_ref.  Worker processes only."""
    for sub in ("data", "calibration", "models"):
        p = os.path.join(REF_DIR, "src", sub)
        if p not in sys.path:
            sys.path.insert(0, p)
    import double_heston
    assert os.path.realpath(double_heston.__file__).startswith(os.path.realpath(REF_DIR)), double_heston.__file__
    return double_heston


def _cpu_chunk(job):
    params, strikes, maturities, N, r, use_ref = job
    t0 = time.perf_counter()
    acc = 0.0
    if use_ref:
        DoubleHeston = _import_reference().DoubleHeston
        with np.errstate(all="ignore"):
            for p in params:
                for T in maturities:
                    for K in strikes:
                        acc += DoubleHeston(100.0, K, T, r, *[float(v) for v in p], option_type="call").pricing(N=N)
    else:
        from oracle import cos_oracle as O
        for p in params:
            for T in maturities:
                for K in strikes:
                    acc += O.price_scalar(p, 100.0, K, T, r, True, 0.0, N)
    return len(params) * len(strikes) * len(maturities), acc, time.perf_counter() - t0


def cpu_throughput(wl, sets_per_core: int, pool, cores: int, seed: int, use_ref: bool):
    """prices/s of the reference on `cores` processes; returns (value, n_prices, seconds)."""
    params = gen_params(sets_per_core * cores, seed)
    jobs = [(params[i::cores], wl["strikes"], wl["maturities"], wl["N"], wl["r"], use_ref) for i in range(cores)]
    t0 = time.perf_counter()
    done = pool.map(_cpu_chunk, jobs)
    dt = time.perf_counter() - t0
    n = sum(d[0] for d in done)
    return n / dt, n, dt


def host_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def make_pool(cores):
    import multiprocessing as mp
    return mp.get_context("spawn").Pool(cores)


def cpu_kind(use_ref):
    if use_ref:
        return "reference", ("the unmodified reference: DoubleHeston(...).pricing(N) of baseline/_ref/src/models/double_heston.py "
                             "(pip-installed from /root/reference by __graft_entry__.build()), one process per host core")
    return "port", ("baseline/_ref is absent: oracle/cos_oracle.py price_scalar, the operation-for-operation port of "
                    "src/models/double_heston.py:160-192, one process per host core")


def _ref_loss_timing(job):
    """Worker: the reference's DoubleHestonJumpCalibrator.compute_loss along its own recorded trajectory."""
    spot, r, strike, maturity, market, xs, budget_s = job
    _import_reference()
    import lbfgs_calibrator
    assert os.path.realpath(lbfgs_calibrator.__file__).startswith(os.path.realpath(REF_DIR))
    opts = [{"strike": float(strike[j]), "maturity": float(maturity[j]), "price": float(market[j]), "option_type": "call"}
            for j in range(len(strike))]
    cal = lbfgs_calibrator.DoubleHestonJumpCalibrator(spot, r, opts)
    cal.compute_loss(xs[0])
    t0 = time.perf_counter()
    n = 0
    for x in xs:
        cal.compute_loss(x)
        n += 1
        if time.perf_counter() - t0 > budget_s:
            break
    return n, time.perf_counter() - t0


def _ref_full_calibration(job):
    """Worker: the reference's calibrate(maxiter, multi_start) on the C1 market, np.random.seed(0) — minutes."""
    spot, r, strike, maturity, market, maxiter, multi_start = job
    _import_reference()
    import lbfgs_calibrator
    opts = [{"strike": float(strike[j]), "maturity": float(maturity[j]), "price": float(market[j]), "option_type": "call"}
            for j in range(len(strike))]
    cal = lbfgs_calibrator.DoubleHestonJumpCalibrator(spot, r, opts)
    np.random.seed(0)
    t0 = time.perf_counter()
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        res = cal.calibrate(maxiter=maxiter, multi_start=multi_start)
    return time.perf_counter() - t0, float(res.final_loss), int(res.iterations), str(res.message)


def c1_fixture():
    g = np.load(os.path.join(ROOT, "tests", "golden", "calib_trajectory.npz"))
    return g


def reference_calibration_seconds(budget_s=8.0):
    """Seconds the REFERENCE needs for the README calibration on this box, from a bounded sample: its own
    compute_loss timed along the first evaluations of its recorded seed-0 run (tests/golden/calib_trajectory.npz,
    produced by the unmodified reference: 294 + 826 + 2 086 = 3 206 evaluations), times the run's length."""
    if not reference_available():
        return {"unavailable": "baseline/_ref absent"}
    g = c1_fixture()
    n_total = int(sum(g[f"s{s}_fs"].size for s in range(3)))
    with make_pool(1) as pool:
        n, dt = pool.map(_ref_loss_timing, [(float(g["spot"]), float(g["r"]), g["strike"], g["maturity"], g["market"],
                                             g["s1_xs"], budget_s)])[0]
    return {"value": dt / n * n_total, "unit": "s", "kind": "extrapolated",
            "evaluations_timed": n, "seconds_timed": dt, "evaluations_total": n_total,
            "note": "reference compute_loss (baseline/_ref) timed on this box along its own recorded seed-0 trajectory, "
                    "one core (the reference is sequential), x the 3 206 evaluations of that calibrate(300, 3) run; "
                    "`--workload c1 --impl reference` runs the whole calibration",
            "published_m1_seconds": 117.8, "build_container_seconds": 425.0}


def run_reference_arm(args, wl):
    """--impl reference: the reference's CPU path, bounded sample per step, rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = host_cores()
    use_ref = reference_available()
    kind, note = cpu_kind(use_ref)
    if wl["kind"] == "calibration":
        g = c1_fixture()
        job = (float(g["spot"]), float(g["r"]), g["strike"], g["maturity"], g["market"], 300, 3)
        if not use_ref:
            print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref absent (run __graft_entry__.build())"}))
            return
        with make_pool(1) as pool:
            secs, fl, nit, msg = pool.map(_ref_full_calibration, [job])[0]
        line = {"impl": "reference", "metric": "s per 15-option calibration (maxiter=300, multi_start=3)", "value": secs,
                "unit": "s", "n_gpus": args.gpus, "steps": 1, "warmup": 0, "ms_per_step": secs * 1e3,
                "higher_is_better": False, "scaling": "weak", "vs_baseline": secs / 117.8, "dtype": "f64",
                "data": "synthetic", "config": {"workload": wl["name"]},
                "cpu_baseline": {"value": secs, "unit": "s", "cores": 1, "kind": kind,
                                 "sample": "the whole calibrate(300, 3), np.random.seed(0)", "final_loss": fl,
                                 "iterations": nit, "message": msg},
                "e2e": {"value": secs, "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line), flush=True)
        return
    if wl["kind"] != "price":          # c4 / c5: the CPU arm of a sweep is its pricing (15-option grid, N=128)
        wl = dict(WORKLOADS["c2"], name=wl["name"])
    per_price = 8.0e-3 if wl["N"] <= 128 else 15.0e-3          # s per price per core (BASELINE.md §2, reference)
    n_opt = len(wl["strikes"]) * len(wl["maturities"])
    sets_per_core = max(1, int(round(2.0 / (per_price * n_opt))))       # ~2 s of work per step per core
    with make_pool(cores) as pool:
        for w in range(args.warmup):
            cpu_throughput(wl, sets_per_core, pool, cores, 1000 + w, use_ref)
        n_tot, t_tot = 0, 0.0
        for k in range(args.steps):
            _, n, dt = cpu_throughput(wl, sets_per_core, pool, cores, 2000 + k, use_ref)
            n_tot += n
            t_tot += dt
    value = n_tot / t_tot
    sample = f"{sets_per_core * cores} parameter sets x {n_opt} options per step ({sets_per_core} per core)"
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl["name"], "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample, "note": note},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks sampler
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    REASONS = {0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, device: int):
        self.samples, self.reasons, self.max_mhz, self.ok = [], set(), None, False
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(vis.split(",")[device]) if vis and vis.split(",")[device].isdigit() else device
            self._h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as e:       # noqa: BLE001
            self.error = repr(e)
        self._thread = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self._h)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:        # noqa: BLE001
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        if self.ok:
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self.ok:
            self._thread.join()

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "NVML unavailable"}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def bind_rank_to_cores(local: int, world: int):
    """With several ranks on one host, give each rank its own slice of the cores NVML names as near its GPU (before
    any pinned allocation: first touch decides the memory node).  Returns a description for the JSON line."""
    # opt-in (BENCH_BIND=1): on this pool's 8-GPU hosts every GPU reports the same 32 cores and one memory node, and
    # slicing them per rank made the end-to-end arm 2 % slower (8.98e9 vs 9.15e9 prices/s, profiles/README.md r02)
    if world <= 1 or not os.environ.get("BENCH_BIND"):
        return None
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        idx = int(vis.split(",")[local]) if vis and vis.split(",")[local].isdigit() else local
        h = pynvml.nvmlDeviceGetHandleByIndex(idx)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        near = [c for c in range(n_cpu) if (words[c // 64] >> (c % 64)) & 1]
        allowed = sorted(set(near) & set(os.sched_getaffinity(0))) or sorted(os.sched_getaffinity(0))
        # ranks that share the same near set split it evenly
        per = max(1, len(allowed) // world)
        mine = allowed[(local * per) % len(allowed):][:per] or allowed
        os.sched_setaffinity(0, mine)
        return {"cores": [mine[0], mine[-1]], "n": len(mine), "near_gpu": [near[0], near[-1]] if near else None}
    except Exception as e:      # noqa: BLE001
        return {"error": repr(e)}


# ------------------------------------------------------------------------------------------------
class Bench:
    """Per-process state of the B200 arm: torch device, process group, libdhj context."""

    def __init__(self, args):
        self.args = args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.binding = bind_rank_to_cores(self.local, self.world)
        import torch
        import torch.distributed as dist
        import dhj
        self.torch, self.dist, self.dhj = torch, dist, dhj
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        os.environ.setdefault("DHJ_DEVICE", str(self.local))
        self.ctx = dhj.default_context()
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)        # > 126 MB L2

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x: float) -> float:
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def gather_floats(self, x: float):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world == 1:
            return [float(x)]
        out = self.torch.zeros(self.world, dtype=self.torch.float64, device=self.dev)
        self.dist.all_gather_into_tensor(out, t)
        return [float(v) for v in out.tolist()]

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def roofline_block(per_gpu_prices_per_s, nK, nT, N, kernel_ms, P, fp64_peak, workload_key, kernel_name):
    """Physical FP64-pipe roofline of the dominant kernel (see the module docstring)."""
    fpp = flop_per_price(nK, N)
    contract = per_gpu_prices_per_s * fpp / 1e12
    bytes_alg = P * (13 * 8 + nK * nT * 8)
    sha = kernel_source_sha()
    ncu, stale, traffic = None, None, None
    tpath = os.path.join(ROOT, "profiles", "ncu_summary.json")
    if os.path.exists(tpath):
        try:
            ncu = json.load(open(tpath)).get(workload_key)
        except Exception:      # noqa: BLE001
            ncu = None
    hbm_peak = None
    ppath = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(ppath):
        hbm_peak = json.load(open(ppath)).get("hbm_gbs")
    block = {"bound": "fp64", "unit": "TFLOP/s", "peak": fp64_peak, "kernel": kernel_name, "kernel_ms": kernel_ms,
             "peak_source": "dhj_fp64_peak: DFMA-chain probe on this GPU, one multiplicand uniform (MEASURED_PEAKS.json "
                            "has no FP64 figure)", "nominal_peak": NOMINAL_FP64_TFLOPS,
             "achieved_contract": contract, "frac_contract": contract / fp64_peak, "flop_per_price_contract": fpp,
             "contract_note": "SURVEY §8d: prices/s x FLOP/price of the reference's formulas (one sincos per strike and k); "
                              "the kernel's rotation recurrences execute fewer flops, so this exceeds 1 — it is NOT a "
                              "fraction of the pipe",
             "kernel_source_sha": sha,
             "hbm": {"achieved_gbs": bytes_alg / (kernel_ms * 1e-3) / 1e9, "peak_gbs": hbm_peak,
                     "note": "compute-bound path: algorithmic bytes / kernel time, for information"}}
    if ncu:
        stale = ncu.get("kernel_source_sha") != sha
        slots = ncu.get("fp64_warp_instructions_per_price")               # warp-level FP64 instructions per price
        if slots is None:
            slots = ncu["fp64_warp_instructions"] / (ncu.get("prices_per_launch") or P * nK * nT)
        achieved = per_gpu_prices_per_s * slots * 32 * 2 / 1e12         # an issue slot = 32 lanes x 1 FMA = 64 flop
        flops = per_gpu_prices_per_s * ncu["executed_flop_per_price"] / 1e12
        traffic = ncu.get("dram_bytes_per_launch")
        block.update({
            "achieved": achieved, "frac": achieved / fp64_peak, "traffic": traffic,
            "definition": "achieved = FP64 issue slots executed per second x 64 flop (DFMA, DMUL, DADD, DSETP each hold the "
                          "pipe for one slot); frac = share of the FP64 pipe's peak, <= 1 by construction",
            "fp64_warp_instructions_per_price": slots,
            "executed_flop_per_price": ncu["executed_flop_per_price"], "executed_tflops": flops,
            "executed_flops_frac": flops / fp64_peak,
            "ncu_fp64_pipe_active_pct": ncu.get("fp64_pipe_active_pct"), "ncu_issue_active_pct": ncu.get("issue_active_pct"),
            "ncu_source": ncu.get("capture"), "ncu_capture_is_of_this_build": not stale})
        if stale:
            block["stale_note"] = ("the kernel sources changed after the ncu capture recorded in profiles/ncu_summary.json: "
                                   "instruction counts are of an older build")
    else:
        block.update({"achieved": None, "frac": None, "traffic": None,
                      "note": "no ncu capture recorded for this workload in profiles/ncu_summary.json"})
    return block


def run_price_workload(B: Bench, wl, key, outputs=None):
    """C2 / C3: value (kernel arm), e2e (host-buffer C-ABI call), roofline.  `outputs` (a dict) receives the prices
    of the last timed step."""
    torch, ctx, args = B.torch, B.ctx, B.args
    P, N, r = wl["P"], wl["N"], wl["r"]
    strikes, mats = np.array(wl["strikes"]), np.array(wl["maturities"])
    nK, nT = strikes.size, mats.size
    n_prices = P * nK * nT
    h_params = torch.from_numpy(gen_params(P, 20260101 + B.rank)).pin_memory()
    h_s0 = torch.full((1,), 100.0, dtype=torch.float64).pin_memory()
    h_out = torch.empty((P, nT, nK), dtype=torch.float64).pin_memory()
    d_params, d_s0 = h_params.to(B.dev), h_s0.to(B.dev)
    d_out = torch.empty((P, nT, nK), dtype=torch.float64, device=B.dev)
    stream = torch.cuda.current_stream().cuda_stream

    def step_kernel():
        ctx.price_grid_dev(d_params.data_ptr(), P, d_s0.data_ptr(), 0, strikes, mats, r, 0.0, N, 10.0, False, True,
                           d_out.data_ptr(), stream)

    fp64_peak, _ = ctx.fp64_peak(8192)
    for _ in range(args.warmup):
        step_kernel()
    B.barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches0 = ctx.launch_count
    with ClockSampler(B.local) as clocks:
        B.barrier()
        for e0, e1 in ev:
            B.flush.zero_()                    # L2 flush, outside the timed events
            e0.record()
            step_kernel()
            e1.record()
        B.barrier()
    launches = ctx.launch_count - launches0
    my_ms = sum(e0.elapsed_time(e1) for e0, e1 in ev)
    per_rank_ms = [v / args.steps for v in B.gather_floats(my_ms)]
    total_ms = B.max_over_ranks(my_ms)
    value = B.world * n_prices * args.steps / (total_ms * 1e-3)
    checksum = float(d_out.sum().item())
    checks = B.gather_floats(checksum)             # the ranks' results stay sharded; their checksums travel (NCCL)
    if outputs is not None:
        outputs.update(output_sample({"prices": d_out}))

    # ---- end-to-end arm: host buffers through the C-ABI -------------------------------------------
    np_params, np_s0, np_out = h_params.numpy(), h_s0.numpy(), h_out.numpy()
    for _ in range(max(1, min(args.warmup, 3))):
        ctx.price_grid(np_params, np_s0, strikes, mats, r, 0.0, N, 10.0, False, True, out=np_out)
    e2e_steps = max(3, min(args.steps, 10))
    B.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        ctx.price_grid(np_params, np_s0, strikes, mats, r, 0.0, N, 10.0, False, True, out=np_out)
        _ = float(np_out[0, 0, 0])             # the result is on the host when the call returns
    my_e2e = time.perf_counter() - t0
    B.barrier()
    e2e_s = B.max_over_ranks(my_e2e)
    e2e_per_rank = B.gather_floats(my_e2e / e2e_steps * 1e3)
    e2e_value = B.world * n_prices * e2e_steps / e2e_s
    e2e_match = bool(np.array_equal(np_out, d_out.cpu().numpy()))
    # what the host link gives each rank when every rank copies at once (names the limiter of the e2e arm at N > 1)
    link = {}
    for name, fn, nbytes in (("h2d", lambda: d_params.copy_(h_params, non_blocking=True), h_params.numel() * 8),
                             ("d2h", lambda: h_out.copy_(d_out, non_blocking=True), h_out.numel() * 8)):
        fn(); B.barrier()
        t0 = time.perf_counter()
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        link[name + "_gbs_per_rank"] = [round(nbytes * 3 / v / 1e9, 2) for v in B.gather_floats(time.perf_counter() - t0)]
        B.barrier()

    kernel_ms = total_ms / args.steps
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": B.world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": kernel_ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": wl["name"], "sets_per_gpu": P, "options_per_set": nK * nT, "N": N,
                   "l2": "256 MiB buffer written between timed steps (untimed); inputs+outputs = "
                         f"{P * (13 * 8 + nK * nT * 8) / 2**20:.0f} MiB per step",
                   "sharding": "by parameter set, one batch per rank, no data-path collective; the ranks' checksums are "
                               "all-gathered (NCCL) after the timed steps" if B.world > 1 else "single GPU"},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(P * 13 * 8 + 8),
                "d2h_bytes_per_step": int(n_prices * 8), "steps": e2e_steps, "sets_per_step": P,
                "ms_per_step_per_rank": e2e_per_rank,
                "api": "dhj.Context.price_grid -> dhj_price_grid (pinned host in/out)",
                "bit_identical_to_kernel_arm": e2e_match, "host_link_all_ranks_at_once": link,
                "rank_core_binding": B.binding},
        "gpu_launches": int(launches),
        "roofline": roofline_block(value / B.world, nK, nT, N, kernel_ms, P, fp64_peak, key,
                                   "k_price_batch" if nK <= 8 else "k_price_dense"),
        "ms_per_step_per_rank": per_rank_ms,
        "clocks": clocks.summary(),
        "checksum": checksum, "checksum_all_ranks": float(sum(checks)),
    }
    return line


def run_sweep(B: Bench, wl, steps, warmup, outputs=None):
    """C4: the dataset sweep, STRONG scaling — samples [lo, hi) of the counter stream per rank (whole histories),
    drawn, priced, noised and reduced to losses on the device; the per-sample losses are all-gathered inside the
    timed region (prices and market prices stay sharded, as a dataset writer would leave them).  `outputs` (a dict)
    receives this rank's samples of the last timed step."""
    torch, ctx, dist = B.torch, B.ctx, B.dist
    from dhj.shard import history_shard
    n_total, path_len = wl["P"], GEN["path_len"]
    first, hi_i = history_shard(n_total, path_len, B.world, B.rank)
    n = hi_i - first
    per = -(-(-(-n_total // path_len)) // B.world) * path_len                 # padded block of the gather
    M = 15
    f64 = dict(dtype=torch.float64, device=B.dev)
    bufs = {"params": torch.empty((n, 13), **f64), "spots": torch.empty((n,), **f64),
            "model": torch.empty((n, M), **f64), "market": torch.empty((n, M), **f64),
            "loss": torch.zeros((per,), **f64)}
    all_loss = torch.empty((per * B.world,), **f64) if B.world > 1 else None
    stream = torch.cuda.current_stream().cuda_stream
    gargs = [GEN[k] for k in ("path_len", "lo", "hi", "persistence", "spot0", "ret_mean", "ret_sd", "noise_sd",
                              "strikes_rel", "maturities", "r")]

    def step():
        ctx.generate_dev(C4_SEED, first, n, *gargs, bufs["params"].data_ptr(), bufs["spots"].data_ptr(),
                         bufs["model"].data_ptr(), bufs["market"].data_ptr(), bufs["loss"].data_ptr(), stream)
        if B.world > 1:
            dist.all_gather_into_tensor(all_loss, bufs["loss"])

    for _ in range(warmup):
        step()
    B.barrier()
    launches0 = ctx.launch_count
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    with ClockSampler(B.local) as clocks:
        B.barrier()
        for e0, e1 in ev:
            B.flush.zero_()
            e0.record(); step(); e1.record()
        B.barrier()
    launches = ctx.launch_count - launches0
    my_ms = sum(e0.elapsed_time(e1) for e0, e1 in ev)
    per_rank_ms = [v / steps for v in B.gather_floats(my_ms)]
    total_ms = B.max_over_ranks(my_ms)
    value = n_total * M * steps / (total_ms * 1e-3)
    loss_mean = float((all_loss if B.world > 1 else bufs["loss"][:n]).sum().item()) / n_total
    if outputs is not None:
        outputs.update(output_sample({k: bufs[k][:n] for k in ("params", "spots", "model", "market", "loss")}))
    # the HBM-bound epilogue alone (market prices + per-sample loss): one sweep with it minus one without, no gather
    def timed_once(with_market):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        ctx.generate_dev(C4_SEED, first, n, *gargs, bufs["params"].data_ptr(), bufs["spots"].data_ptr(),
                         bufs["model"].data_ptr(), bufs["market"].data_ptr() if with_market else 0,
                         bufs["loss"].data_ptr() if with_market else 0, stream)
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1)
    ms_with, ms_without = timed_once(True), timed_once(False)
    bytes_out = n * (13 + 1 + 2 * M + 1) * 8
    hbm_peak = None
    ppath = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(ppath):
        hbm_peak = json.load(open(ppath)).get("hbm_gbs")
    # end to end: the same sweep into pinned host arrays (dhj_generate), 4 Mi samples per rank
    n_e2e = min(n, 1 << 22)
    host = {k: torch.empty(s, dtype=torch.float64).pin_memory().numpy()
            for k, s in (("params", (n_e2e, 13)), ("spots", (n_e2e,)), ("model", (n_e2e, M)), ("market", (n_e2e, M)),
                         ("loss", (n_e2e,)))}
    hargs = dict(GEN)
    ctx.generate(C4_SEED, first, min(n_e2e, 1 << 18), **hargs)
    B.barrier()
    t0 = time.perf_counter()
    ctx.generate(C4_SEED, first, n_e2e, out=host, **hargs)
    my_e2e = time.perf_counter() - t0
    B.barrier()
    e2e_s = B.max_over_ranks(my_e2e)
    e2e_match = bool(np.array_equal(host["market"], bufs["market"][:n_e2e].cpu().numpy()))
    return {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": B.world, "steps": steps, "warmup": warmup,
        "ms_per_step": total_ms / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic (generated on the device: counter stream seed %d)" % C4_SEED,
        "config": {"workload": wl["name"], "samples_total": n_total, "samples_this_rank": n, "options_per_set": M,
                   "N": wl["N"], "l2": "256 MiB buffer written between timed steps (untimed); per-rank outputs "
                                       f"{bytes_out / 2**30:.1f} GiB",
                   "sharding": "contiguous blocks of whole histories per rank (dhj.shard.shard_bounds), no data-path "
                               "collective; the per-sample losses are all-gathered over NCCL INSIDE the timed region"},
        "api": "dhj.Context.generate_dev -> dhj_generate_dev (k_gen_draws -> k_price_batch -> k_gen_market)",
        "gpu_launches": int(launches), "ms_per_step_per_rank": per_rank_ms, "mean_loss": loss_mean,
        "clocks": clocks.summary(),
        "hbm": {"bytes_written_per_step_this_rank": bytes_out,
                "achieved_gbs_whole_sweep": bytes_out / (ms_with * 1e-3) / 1e9,
                "epilogue_ms": max(0.0, ms_with - ms_without),
                "epilogue_gbs": n * (2 * M + 1) * 8 / (max(1e-6, ms_with - ms_without) * 1e-3) / 1e9,
                "epilogue_note": "k_gen_market reads the model prices and writes market prices + losses "
                                 f"({n * (2 * M + 1) * 8 / 2**30:.2f} GiB): time of one sweep with it minus one without it",
                "peak_gbs": hbm_peak, "note": "the sweep is FP64-bound (pricing kernel); HBM is idle most of the time"},
        "e2e": {"value": B.world * n_e2e * M / e2e_s, "unit": UNIT, "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": int(n_e2e * (13 + 1 + 2 * M + 1) * 8), "samples_per_rank": n_e2e,
                "api": "dhj.Context.generate -> dhj_generate (pinned host arrays out; nothing goes up: the inputs are "
                       "drawn on the device)", "bit_identical_to_device_arm": e2e_match},
    }


def run_calibrations(B: Bench, wl, steps, warmup, outputs=None):
    """C5: 10 000 markets x 3 starts through calibrate_many_sharded; the gather of the results (NCCL) is inside the
    timed region.  Markets: the first 10 000 samples of the C4 dataset (noisy market prices from the device).
    `outputs` (a dict) receives the per-market arrays of the last timed step."""
    dhj, ctx = B.dhj, B.ctx
    n = wl["markets"]
    data = ctx.generate(C4_SEED, 0, n, **GEN)
    spots, market = data["spots"], data["market"]
    K = np.tile(np.array(GRID_K)[None, :] * spots[:, None] / 100.0, (1, 3))
    T = np.repeat(np.array(GRID_T), 5)
    np.random.seed(1)
    x0 = dhj.initial_guesses(spots, K, T, market, wl["starts"])
    kw = dict(maxiter=300, multi_start=wl["starts"], x0=x0, device=B.dev if B.world > 1 else None)
    for _ in range(max(1, warmup)):                        # buffers of the final shapes, NCCL communicator
        dhj.calibrate_many_sharded(spots, wl["r"], K, T, np.ones(15), market, **dict(kw, maxiter=3))
    times, res = [], None
    launches0 = ctx.launch_count
    for _ in range(steps):
        B.barrier()
        t0 = time.perf_counter()
        res = dhj.calibrate_many_sharded(spots, wl["r"], K, T, np.ones(15), market, **kw)
        my = time.perf_counter() - t0
        times.append(B.max_over_ranks(my))
    launches = ctx.launch_count - launches0
    if outputs is not None:
        outputs.update(output_sample({k: np.asarray(res[k]) for k in ("x", "parameters", "final_loss", "iterations",
                                                                      "status", "success", "best_start",
                                                                      "model_prices")}))
    secs = float(np.median(times))
    fl = res["final_loss"]
    split = {k: res.get(k) for k in ("seconds_loss", "seconds_ask", "seconds_tell", "state_rounds", "evaluations")}
    return {
        "metric": "calibrations/s (15 options, multi_start=3, maxiter=300)", "value": n / secs, "unit": "calibrations/s",
        "n_gpus": B.world, "steps": steps, "warmup": warmup, "ms_per_step": secs * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic (C4 counter stream, first 10 000 samples)",
        "config": {"workload": wl["name"], "markets": n, "starts": wl["starts"],
                   "sharding": "contiguous blocks of markets per rank; every rank runs its own host optimiser and one "
                               "loss launch per round; results all-gathered (NCCL) inside the timed region"},
        "seconds": secs, "seconds_all_steps": times, "rounds_rank0": int(res["rounds"]),
        "gpu_launches": int(launches), "host_device_split_rank0": split,
        "split_note": "seconds_loss = host time inside dhj_loss_fd (copies + launch + wait) per pipeline, seconds_ask / "
                      "seconds_tell = the C++ batch L-BFGS; two pipelines overlap one another above 2 048 markets",
        "final_loss_median": float(np.median(fl)), "final_loss_p95": float(np.percentile(fl, 95)),
        "frac_below_1pct": float(np.mean(fl * 100 < 1.0)), "success_rate": float(np.mean(res["success"])),
        "iterations_median": float(np.median(res["iterations"])),
        "api": "dhj.calibrate_many_sharded -> dhj_lbfgs_ask / dhj_loss_fd / dhj_lbfgs_tell",
    }


def time_readme_calibration(ctx, repeats=5, outputs=None):
    """Second half of BASELINE.json's metric: seconds per 15-option calibration, the README configuration (C1):
    DoubleHestonJumpCalibrator(...).calibrate(maxiter=300, multi_start=3) through the drop-in class on the
    reference suite's market (tests/test_suite.py:274-302).  `outputs` (a dict) receives the last calibration's
    result."""
    for sub in ("models", "calibration"):
        p = os.path.join(PKG, "src", sub)
        if p not in sys.path:
            sys.path.insert(0, p)
    from lbfgs_calibrator import DoubleHestonJumpCalibrator
    from double_heston import DoubleHeston
    g = c1_fixture()
    K, T, mkt = g["strike"], g["maturity"], g["market"]
    opts = [{"strike": K[j], "maturity": T[j], "price": mkt[j], "option_type": "call"} for j in range(15)]
    cal = DoubleHestonJumpCalibrator(float(g["spot"]), float(g["r"]), opts)
    cal.calibrate(maxiter=3, multi_start=1)                                   # warm-up
    times, res, launches = [], None, 0
    for _ in range(repeats):
        np.random.seed(0)
        launches0 = ctx.launch_count
        t0 = time.perf_counter()
        res = cal.calibrate(maxiter=300, multi_start=3)
        times.append(time.perf_counter() - t0)
        launches = ctx.launch_count - launches0
    if outputs is not None:
        outputs.update(output_sample({"parameters": np.array([[res.parameters[k] for k in cal.param_names]]),
                                      "model_prices": res.model_prices[None, :],
                                      "final_loss": np.array([res.final_loss])}))
    # single-call latencies through the drop-in classes: a new (K, T) on every pricing() call
    p = [0.04, 2.0, 0.04, 0.3, -0.5, 0.04, 1.5, 0.04, 0.2, -0.3, 0.1, 0.0, 0.1]
    n_lat = 400
    Ks = 90.0 + 20.0 * np.random.default_rng(0).random(n_lat)
    Ts = 0.25 + np.random.default_rng(1).random(n_lat)
    for i in range(20):
        DoubleHeston(100.0, Ks[i], Ts[i], 0.05, *p, option_type="call").pricing()
    t0 = time.perf_counter()
    for i in range(n_lat):
        DoubleHeston(100.0, Ks[i], Ts[i], 0.05, *p, option_type="call").pricing()
    us_pricing = (time.perf_counter() - t0) / n_lat * 1e6
    x = g["s1_x0"]
    t0 = time.perf_counter()
    for i in range(n_lat):
        cal.compute_loss(x)
    us_loss = (time.perf_counter() - t0) / n_lat * 1e6
    t0 = time.perf_counter()
    for i in range(n_lat):
        cal.compute_loss_and_grad(x)
    us_fg = (time.perf_counter() - t0) / n_lat * 1e6
    calib = {"metric": "s per 15-option calibration (maxiter=300, multi_start=3)", "value": float(np.median(times)),
             "min": float(min(times)), "unit": "s", "higher_is_better": False, "repeats": repeats,
             "final_loss": float(res.final_loss), "iterations": int(res.iterations), "gpu_launches": int(launches),
             "api": "DoubleHestonJumpCalibrator.calibrate -> dhj_loss_fd (one launch per optimiser round)"}
    latency = {"pricing_us": us_pricing, "compute_loss_us": us_loss, "loss_and_fd_gradient_us": us_fg, "calls": n_lat,
               "note": "wall time per call through the drop-in classes, host buffers in and out: DoubleHeston(...).pricing() "
                       "with a new strike and maturity on every call (a new option book each time), compute_loss(x) = 15 "
                       "prices, compute_loss_and_grad(x) = 210 prices + scipy's forward differences"}
    return calib, latency


def run_b200_arm(args, wl, key):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    # CPU baseline first (rank 0, N=1 only), before CUDA is initialised in this process
    cpu_baseline, ref_calibration = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = host_cores()
        use_ref = reference_available()
        kind, note = cpu_kind(use_ref)
        pw = wl if wl["kind"] == "price" else WORKLOADS["c2"]
        per_price = 8.0e-3 if pw["N"] <= 128 else 15.0e-3
        n_opt = len(pw["strikes"]) * len(pw["maturities"])
        sets_per_core = max(1, int(round(12.0 / (per_price * n_opt))))       # ~12 s of work per core
        with make_pool(cores) as pool:
            v, n, dt = cpu_throughput(pw, sets_per_core, pool, cores, 4242, use_ref)
        cpu_baseline = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
                        "sample": f"{sets_per_core * cores} seeded parameter sets x {n_opt} options "
                                  f"({n} prices, {dt:.1f} s wall) of the same workload",
                        "per_core": v / cores, "note": note}
        try:     # best-effort CPU line: the same arithmetic restated in C (oracle/cos_oracle.c), OpenMP over options
            from oracle import cos_oracle as O
            lib = O.c_library()
            pc = gen_params(2500 * cores, 777)
            Kc = np.tile(np.array(pw["strikes"]), len(pw["maturities"]))
            Tc = np.repeat(np.array(pw["maturities"]), len(pw["strikes"]))
            O.c_price_batch(pc[:cores], 100.0, Kc, Tc, np.ones(Kc.size), pw["r"], 0.0, pw["N"])      # warm-up
            t0c = time.perf_counter()
            O.c_price_batch(pc, 100.0, Kc, Tc, np.ones(Kc.size), pw["r"], 0.0, pw["N"])
            dtc = time.perf_counter() - t0c
            cpu_baseline["c_port"] = {"value": pc.shape[0] * Kc.size / dtc, "unit": UNIT,
                                      "threads": int(lib.oracle_threads()), "kind": "port",
                                      "sample": f"{pc.shape[0]} parameter sets x {Kc.size} options, {dtc:.1f} s",
                                      "note": "NOT the reference: oracle/cos_oracle.c, the reference's arithmetic in C99 "
                                              "with OpenMP (a best-effort CPU implementation)"}
        except Exception as e:      # noqa: BLE001
            cpu_baseline["c_port"] = {"unavailable": repr(e)}
        if key in ("c2", "c1"):
            ref_calibration = reference_calibration_seconds()

    B = Bench(args)
    outputs = {} if args.dump_outputs is not None else None
    if wl["kind"] == "price":
        line = run_price_workload(B, wl, key, outputs)
        if key == "c2":
            if rank == 0:
                calib, latency = time_readme_calibration(B.ctx)
                if ref_calibration is not None:
                    calib["reference_seconds"] = ref_calibration
                line["calibration"], line["latency"] = calib, latency
            if not args.no_extra:
                B.barrier()
                extra = {}
                c4 = dict(WORKLOADS["c4"])
                extra["c4"] = run_sweep(B, c4, steps=2, warmup=1)
                extra["c5"] = run_calibrations(B, WORKLOADS["c5"], steps=2, warmup=1)
                line["extra"] = {k: {kk: v[kk] for kk in v if kk not in ("metric", "unit", "dtype", "higher_is_better",
                                                                         "vs_baseline")} | {"metric": v["metric"], "unit": v["unit"]}
                                 for k, v in extra.items()}
    elif wl["kind"] == "sweep":
        line = run_sweep(B, wl, args.steps, max(1, min(args.warmup, 3)), outputs)
    elif wl["kind"] == "calibrations":
        line = run_calibrations(B, wl, args.steps, args.warmup, outputs)
    else:                                                   # c1
        calib, latency = time_readme_calibration(B.ctx, repeats=args.steps, outputs=outputs)
        if ref_calibration is not None:
            calib["reference_seconds"] = ref_calibration
        line = {"metric": calib["metric"], "value": calib["value"], "unit": "s", "n_gpus": B.world, "steps": calib["repeats"],
                "warmup": 1, "ms_per_step": calib["value"] * 1e3, "higher_is_better": False, "scaling": "weak",
                "vs_baseline": calib["value"] / 117.8, "dtype": "f64", "data": "synthetic",
                "config": {"workload": wl["name"], "replicas": "a single calibration does not shard: every rank runs its own"},
                "calibration": calib, "latency": latency, "gpu_launches": calib["gpu_launches"],
                "e2e": {"value": calib["value"], "unit": "s", "h2d_bytes_per_step": 104 * 3 * calib["gpu_launches"] // 3,
                        "d2h_bytes_per_step": 112 * 3 * calib["gpu_launches"] // 3,
                        "note": "calibrate() is already the public API with host buffers in and out"}}
    if rank == 0:
        if cpu_baseline is not None:
            line["cpu_baseline"] = cpu_baseline
        if outputs is not None:
            write_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    B.close()


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of the headline workload")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="default workload only: skip the C4 / C5 blocks")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the headline's outputs of the last timed step to DIR/<name>.npy (--impl b200)")
    args = ap.parse_args(argv)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200: the reference arm keeps no outputs")
    return args


def main():
    args = parse_args()
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        run_reference_arm(args, wl)
    else:
        run_b200_arm(args, wl, args.workload)


if __name__ == "__main__":
    main()
