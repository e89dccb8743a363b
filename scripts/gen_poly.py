#!/usr/bin/env python3
"""Derives the polynomial coefficients used by option-pricing-ffn-lbfgs_b200/csrc/dhj_fastmath.cuh with
mpmath (60 digits): near-minimax fits by Chebyshev-node interpolation followed by a few Remez exchanges.
Prints C initialisers and the achieved maximum error.  Run: python scripts/gen_poly.py"""
import mpmath as mp

mp.mp.dps = 60


def remez(f, a, b, deg, weight=None, iters=12):
    """Minimax polynomial sum c_i x^i for f on [a,b] (absolute error, optionally weighted)."""
    w = weight or (lambda x: mp.mpf(1))
    n = deg + 2
    xs = [(a + b) / 2 + (b - a) / 2 * mp.cos(mp.pi * (n - 1 - i) / (n - 1)) for i in range(n)]
    for _ in range(iters):
        A = mp.matrix(n, n)
        rhs = mp.matrix(n, 1)
        for i, x in enumerate(xs):
            for j in range(deg + 1):
                A[i, j] = x ** j
            A[i, deg + 1] = (-1) ** i / w(x)
            rhs[i] = f(x)
        sol = mp.lu_solve(A, rhs)
        c = [sol[j] for j in range(deg + 1)]
        err = lambda x: (mp.polyval(c[::-1], x) - f(x)) * w(x)
        # new extrema: sample densely, pick local maxima of |err| between sign changes
        grid = [a + (b - a) * mp.mpf(i) / 4000 for i in range(4001)]
        vals = [err(x) for x in grid]
        ext = []
        i = 0
        while i < len(grid):
            j = i
            while j + 1 < len(grid) and (vals[j + 1] > 0) == (vals[i] > 0):
                j += 1
            k = max(range(i, j + 1), key=lambda t: abs(vals[t]))
            ext.append(grid[k])
            i = j + 1
        if len(ext) != n:
            break
        xs = ext
    emax = max(abs(v) for v in vals)
    return c, emax


def show(name, c, emax):
    print(f"// {name}: max error {mp.nstr(emax, 5)}")
    print("{" + ", ".join(mp.nstr(x, 20) for x in c) + "}")


if __name__ == "__main__" and len(__import__("sys").argv) == 1:
    # exp(r) = 1 + r + r^2 * q(r), |r| <= ln2/2 ; q of degree 9 (total degree 11)
    L = mp.log(2) / 2
    q = lambda r: (mp.exp(r) - 1 - r) / r ** 2 if abs(r) > mp.mpf('1e-15') else mp.mpf(1) / 2 + r / 6 + r * r / 24
    c, e = remez(q, -L, L, 9)
    show("exp q(r) deg 9 (abs error of q; times r^2 <= 0.12)", c, e)
    c, e = remez(q, -L, L, 10)
    show("exp q(r) deg 10", c, e)


# ---- coefficients that fit a 32-bit immediate -----------------------------------------------------------------
# An FP64 instruction on sm_100 takes a double constant for free only as a 32-bit immediate (the high word; low
# word zero); any other coefficient costs a constant-bank load.  The highest-order coefficients of a polynomial
# need few bits, so they are rounded to 21 significant bits and the remaining coefficients are refitted around
# them (python scripts/gen_poly.py imm).
def round_hi(x):
    import struct
    b = struct.unpack("<Q", struct.pack("<d", float(x)))[0]
    b = (b + 0x80000000) & 0xFFFFFFFF00000000
    return mp.mpf(struct.unpack("<d", struct.pack("<Q", b))[0])


def refit_with_fixed_top(f, a, b, deg, n_fixed):
    """Minimax coefficients c_0..c_deg of f on [a,b] where the top n_fixed are rounded to a high word, one at a
    time, and the lower ones refitted after each rounding."""
    fixed = []
    for step in range(n_fixed + 1):
        d = deg - len(fixed)
        g = lambda x: f(x) - sum(c * x ** (d + 1 + i) for i, c in enumerate(reversed(fixed)))
        c, e = remez(g, a, b, d)
        if step < n_fixed:
            fixed.append(round_hi(c[-1]))
    return c + list(reversed(fixed)), e


def imm_main():
    Z = (mp.pi / 4) ** 2 * mp.mpf("1.02")
    sq = lambda z: mp.sqrt(z)
    fs = lambda z: ((mp.sin(sq(z)) / sq(z) - 1) / z) if z > mp.mpf("1e-20") else -mp.mpf(1) / 6 + z / 120
    c, e = refit_with_fixed_top(fs, mp.mpf(0), Z, 5, 2)
    show("sin: (sin(r)/r - 1)/z, z = r^2 <= (pi/4)^2, top 2 coefficients 32-bit", c, e)
    fc = lambda z: ((mp.cos(sq(z)) - 1 + z / 2) / z ** 2) if z > mp.mpf("1e-12") else mp.mpf(1) / 24 - z / 720 + z * z / 40320
    c, e = refit_with_fixed_top(fc, mp.mpf(0), Z, 5, 2)
    show("cos: (cos(r) - 1 + z/2)/z^2, top 2 coefficients 32-bit", c, e)
    # sincos_tab: |r| <= pi/512 after the 512-entry table
    Zt = (mp.pi / 512) ** 2 * mp.mpf("1.02")
    c, e = refit_with_fixed_top(fs, mp.mpf(0), Zt, 1, 1)
    show("sincos_tab sin: (sin(r)/r - 1)/z, z <= (pi/512)^2, top coefficient 32-bit (times z: relative error)", c, e * Zt)
    c, e = refit_with_fixed_top(fc, mp.mpf(0), Zt, 1, 1)
    show("sincos_tab cos: (cos(r) - 1 + z/2)/z^2, top coefficient 32-bit (times z^2: absolute error)", c, e * Zt * Zt)
    L = mp.log(2) / 128
    q = lambda r: (mp.exp(r) - 1 - r) / r ** 2 if abs(r) > mp.mpf('1e-15') else mp.mpf(1) / 2 + r / 6 + r * r / 24
    c, e = refit_with_fixed_top(q, -L, L, 3, 1)
    show("exp_tab q(r) deg 3 on |r| <= ln2/128, top coefficient 32-bit (error of q; times r^2 <= 2.9e-5)", c, e)
    for name, v in (("1/7", mp.mpf(1) / 7), ("-1/6", -mp.mpf(1) / 6), ("-1/7", -mp.mpf(1) / 7)):
        print(f"// {name} as a high word: {mp.nstr(round_hi(v), 20)}")


if __name__ == "__main__" and len(__import__("sys").argv) > 1 and __import__("sys").argv[1] == "imm":
    imm_main()
