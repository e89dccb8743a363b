"""Bit-for-bit comparison of the price-objective loss paths of two builds of libdhj.so, both loaded in one process.

    python scripts/compare_price_objective.py --baseline path/to/older/libdhj.so [--candidate path/to/libdhj.so]

On the seeded markets of tests/test_gpu_jacobian.py (the c1 and ragged markets of loss_cases.npz and a 24-option
dense market; their states and 20 000 perturbed ones) it runs loss_batch, loss_fd (with f_all) and loss_grad with
each library and reports, per market and batch, whether every output has the same bits.  A baseline built before
an entry point existed loads through stand-ins for the missing symbols (only the loss paths are called).  Exit
status 0 when everything is bit-identical.  Needs a GPU.
"""
import argparse
import ctypes
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "tests"), ROOT, os.path.join(ROOT, "option-pricing-ffn-lbfgs_b200")]

import dhj  # noqa: E402
from dhj._native import EXPORTS  # noqa: E402

_CDLL = ctypes.CDLL


class _OlderLib:
    """a baseline library: symbols it does not export become inert stand-ins so that the binding loads it"""

    def __init__(self, path, *args, **kwargs):
        self._lib = _CDLL(path, *args, **kwargs)

    def __getattr__(self, name):
        try:
            return getattr(self._lib, name)
        except AttributeError:
            if name in EXPORTS:
                self.__dict__[name] = types.SimpleNamespace()
                return self.__dict__[name]
            raise


def outputs(library, baseline):
    from test_gpu_jacobian import _markets
    ctypes.CDLL = _OlderLib if baseline else _CDLL
    try:
        c = dhj.Context(0, library=library)
    finally:
        ctypes.CDLL = _CDLL
    out = []
    for tag, S0, r, K, T, call, mk, x in _markets():
        m = c.market(S0, r, K, T, call, mk)
        rng = np.random.default_rng(1)
        big = x[rng.integers(0, len(x), 20000)] + 1e-3 * rng.standard_normal((20000, 13))
        for xs in (x, big):
            out.append((tag, len(xs), m.loss_batch(xs), *m.loss_fd(xs, want_all=True), *m.loss_grad(xs)))
        m.close()
    c.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--baseline", required=True)
    ap.add_argument("--candidate", default=None, help="default: the in-tree build")
    args = ap.parse_args()
    base = outputs(os.path.abspath(args.baseline), True)
    cand = outputs(args.candidate and os.path.abspath(args.candidate), False)
    ok = True
    for a, b in zip(base, cand):
        same = all(np.array_equal(u, v, equal_nan=True) for u, v in zip(a[2:], b[2:]))
        ok &= same
        print(f"{a[0]} ({a[1]} states): {'bit-identical' if same else 'DIFFERENT'}")
    print("all bit-identical" if ok else "MISMATCH")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
