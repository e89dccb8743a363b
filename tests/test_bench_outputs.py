"""bench.py --dump-outputs: what is written, how large outputs are sampled, and that it is what the timed path computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from conftest import ROOT


def test_small_outputs_are_written_whole_as_float64():
    a = np.arange(12, dtype=np.int32).reshape(4, 3)
    ok = np.array([True, False, True, True])
    out = bench.output_sample({"a": a, "ok": ok})
    assert out["a"].dtype == np.float64 and np.array_equal(out["a"], a)
    assert out["ok"].dtype == np.float64 and np.array_equal(out["ok"], ok)


def test_large_outputs_are_a_fixed_sample_of_rows_within_the_budget():
    n = 10_000
    prices = np.arange(n * 15, dtype=np.float64).reshape(n, 3, 5)
    loss = np.arange(n, dtype=np.float64)
    budget = 8 * 16 * 1000                                          # 1 000 rows of 15 + 1 values
    out = bench.output_sample({"prices": prices, "loss": loss}, budget=budget)
    assert sum(a.nbytes for a in out.values()) <= budget
    rows = out["loss"].astype(np.int64)
    assert rows.size == 1000 and np.all(np.diff(rows) > 0)            # distinct rows, in row order
    assert np.array_equal(out["prices"], prices[rows])               # the same rows in every array
    again = bench.output_sample({"prices": prices, "loss": loss}, budget=budget)
    assert np.array_equal(again["loss"], out["loss"])                # the same sample on every run
    assert bench.DUMP_BYTES + 4096 <= 64 * 10 ** 6


def test_flagship_output_fits_the_budget():
    """C2 prices (1 Mi sets x 15 options, 126 MB) are sampled down to at most DUMP_BYTES."""
    P = bench.WORKLOADS["c2"]["P"]
    assert 15 * 8 * P > bench.DUMP_BYTES >= 15 * 8 * (P // 2)


def test_arguments():
    args = bench.parse_args(["--steps", "7", "--warmup", "0", "--dump-outputs", "out"])
    assert (args.steps, args.warmup, args.dump_outputs) == (7, 0, "out")
    assert bench.parse_args([]).dump_outputs is None
    with pytest.raises(SystemExit):
        bench.parse_args(["--steps", "0"])
    with pytest.raises(SystemExit):
        bench.parse_args(["--impl", "reference", "--dump-outputs", "out"])


@pytest.mark.gpu
def test_dump_is_what_the_timed_path_computed(tmp_path):
    """C3 headline, 2 timed steps: the dumped prices are the whole surface and equal, bit for bit, the host-buffer
    pricing call on the same seeded inputs."""
    out = tmp_path / "dump"
    run = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c3", "--steps", "2",
                          "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(out)],
                         cwd=tmp_path, capture_output=True, text=True, check=True)
    line = json.loads(run.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2
    assert sorted(os.listdir(out)) == ["prices.npy"]
    got = np.load(out / "prices.npy")
    import dhj
    wl = bench.WORKLOADS["c3"]
    ctx = dhj.Context(0)
    want = ctx.price_grid(bench.gen_params(wl["P"], 20260101), 100.0, np.array(wl["strikes"]),      # rank 0's seed
                          np.array(wl["maturities"]), wl["r"], 0.0, wl["N"], 10.0, False, True)
    ctx.close()
    assert got.dtype == np.float64 and got.shape == want.shape
    assert np.array_equal(got, want)
    assert float(got.sum()) == pytest.approx(line["checksum"], rel=1e-12)
