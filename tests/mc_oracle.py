"""NumPy restatement of the Monte Carlo path scheme and its random stream (csrc/dhj_mc.cuh), vectorised over paths.

Stream "DHJ2": Philox4x32-10 with key (seed lo, seed hi) and counter (path lo, path hi, 4 step + j, 0x44484A32);
j = 0, 1 Box-Muller pairs (Z1, Z1p), (Z2, Z2p); j = 2 U -> N by inversion of the Poisson(lambda dt) CDF (capped at 64);
j = 3 (used when N > 0) z0 of its Box-Muller pair.  The scheme's arithmetic is written in the kernel's operation order,
with NumPy's log / sqrt / sin / cos / exp in place of the library's own (they differ by an ulp or two).
"""
import numpy as np

from oracle.cos_oracle import philox4x32_10

MC_STREAM_TAG = 0x44484A32
MAX_JUMPS = 64
KINDS = ("european", "asian", "up-and-out", "up-and-in", "down-and-out", "down-and-in")
_M32 = np.uint64(0xFFFFFFFF)


def mc_words(seed, path, ctr):
    """(w0, w1) of (path[...], counter word ctr): w0 = x0 | x1 << 32, w1 = x2 | x3 << 32 (uint64)."""
    path = np.asarray(path, dtype=np.uint64)
    c = np.stack([path & _M32, path >> np.uint64(32), np.full(path.shape, ctr, dtype=np.uint64),
                  np.full(path.shape, MC_STREAM_TAG, dtype=np.uint64)], axis=-1)
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    key = np.broadcast_to(np.array([seed & 0xFFFFFFFF, seed >> 32], dtype=np.uint64), path.shape + (2,))
    x = philox4x32_10(c, key).astype(np.uint64)
    return x[..., 0] | (x[..., 1] << np.uint64(32)), x[..., 2] | (x[..., 3] << np.uint64(32))


def uniform(w):
    return (w >> np.uint64(11)).astype(np.float64) * 2.0 ** -53


def box_muller(w0, w1):
    u1 = ((w0 >> np.uint64(11)) + np.uint64(1)).astype(np.float64) * 2.0 ** -53
    R = np.sqrt(-2.0 * np.log(u1))
    ang = 6.283185307179586 * uniform(w1)
    return R * np.cos(ang), R * np.sin(ang)


def poisson_inverse(U, p0, lam_dt):
    """Smallest n with U < F(n), F summed in order p_0 = p0, p_n = p_{n-1} lam_dt / n; capped at MAX_JUMPS."""
    U = np.asarray(U, dtype=np.float64)
    n = np.zeros(U.shape, dtype=np.int64)
    p = np.full(U.shape, p0, dtype=np.float64)
    F = p.copy()
    for k in range(1, MAX_JUMPS + 1):
        go = U >= F
        if not go.any():
            break
        n = np.where(go, k, n)
        p = np.where(go, (p * lam_dt) / np.float64(k), p)
        F = np.where(go, F + p, F)
    return n


def draws(seed, paths, n_steps):
    """The stream's per-step draws for paths[n]: dict of [n_steps, n] arrays Z1, Z1p, Z2, Z2p, U, zj (zj is drawn for
    every path here; the scheme uses it where N > 0)."""
    paths = np.asarray(paths, dtype=np.uint64)
    out = {k: np.empty((n_steps, paths.size)) for k in ("Z1", "Z1p", "Z2", "Z2p", "U", "zj")}
    for s in range(n_steps):
        out["Z1"][s], out["Z1p"][s] = box_muller(*mc_words(seed, paths, 4 * s))
        out["Z2"][s], out["Z2p"][s] = box_muller(*mc_words(seed, paths, 4 * s + 1))
        out["U"][s] = uniform(mc_words(seed, paths, 4 * s + 2)[0])
        out["zj"][s] = box_muller(*mc_words(seed, paths, 4 * s + 3))[0]
    return out


def path_stats(p, S0, r, q, T, n_steps, n_obs, seed=0, paths=None, n_paths=None, d=None):
    """(S_T, sum, max, min) of the observation dates for one parameter set p[13] over paths (default 0..n_paths-1);
    `d` = draws(seed, paths, n_steps) may be passed to share them between sets.  Also returns N (jumps per step) and, per
    path, the number of steps that started with a truncated (negative) variance."""
    if paths is None:
        paths = np.arange(n_paths, dtype=np.uint64)
    if d is None:
        d = draws(seed, paths, n_steps)
    p = np.asarray(p, dtype=np.float64)
    dt = T / n_steps
    rho = np.array([p[4], p[9]])
    rhob = np.sqrt(1.0 - rho * rho)
    lam, mu, sj = p[10], p[11], p[12]
    kbar = np.exp(mu + 0.5 * sj * sj) - 1.0
    drift = r - q - lam * kbar
    lam_dt = lam * dt
    p0 = np.exp(-lam_dt)
    n = len(paths)
    x = np.zeros(n)
    v1, v2 = np.full(n, p[0]), np.full(n, p[5])
    every = n_steps // n_obs
    ssum, mx, mn = np.zeros(n), np.full(n, -np.inf), np.full(n, np.inf)
    ST = np.zeros(n)
    jumps = np.empty((n_steps, n), dtype=np.int64)
    trunc = np.zeros(n, dtype=np.int64)
    with np.errstate(all="ignore"):
        for s in range(n_steps):
            N = poisson_inverse(d["U"][s], p0, lam_dt)
            jumps[s] = N
            Nf = N.astype(np.float64)
            J = np.where(N > 0, Nf * mu + (sj * np.sqrt(Nf)) * d["zj"][s], 0.0)
            trunc += (v1 < 0.0) | (v2 < 0.0)
            a1 = np.where(v1 < 0.0, 0.0, v1)
            a2 = np.where(v2 < 0.0, 0.0, v2)
            sq1, sq2 = np.sqrt(a1 * dt), np.sqrt(a2 * dt)
            x = x + ((drift - 0.5 * (a1 + a2)) * dt + sq1 * (rho[0] * d["Z1"][s] + rhob[0] * d["Z1p"][s])
                     + sq2 * (rho[1] * d["Z2"][s] + rhob[1] * d["Z2p"][s]) + J)
            v1 = v1 + ((p[1] * (p[2] - a1)) * dt + (p[3] * sq1) * d["Z1"][s])
            v2 = v2 + ((p[6] * (p[7] - a2)) * dt + (p[8] * sq2) * d["Z2"][s])
            if (s + 1) % every == 0:
                ST = S0 * np.exp(x)
                ssum = ssum + ST
                mx = np.where(ST > mx, ST, mx)
                mn = np.where(ST < mn, ST, mn)
    return {"ST": ST, "sum": ssum, "max": mx, "min": mn, "N": jumps, "truncated": trunc}


def payoff(st, n_obs, kind, is_call, K, B=np.nan):
    """Payoff of one option on every path of path_stats `st`."""
    kind = KINDS.index(kind) if isinstance(kind, str) else int(kind)
    X = st["sum"] / n_obs if kind == 1 else st["ST"]
    dd = X - K if is_call else K - X
    v = np.where(dd < 0.0, 0.0, dd)
    ind = {0: True, 1: True, 2: st["max"] < B, 3: st["max"] >= B, 4: st["min"] > B, 5: st["min"] <= B}[kind]
    return v * np.where(ind, 1.0, 0.0)


def mc_price(params, S0, r, q, T, n_steps, n_obs, kind, is_call, strike, barrier, seed, n_paths):
    """(price[P, M], stderr[P, M], stats[P]): discounted payoff means and standard errors over paths 0..n_paths-1."""
    params = np.asarray(params, dtype=np.float64).reshape(-1, 13)
    P, M = params.shape[0], len(kind)
    S0 = np.broadcast_to(np.asarray(S0, dtype=np.float64), (P,))
    barrier = [np.nan] * M if barrier is None else barrier
    paths = np.arange(n_paths, dtype=np.uint64)
    d = draws(seed, paths, n_steps)
    disc = np.exp(-r * T)
    price, err, stats = np.empty((P, M)), np.empty((P, M)), []
    for i in range(P):
        st = path_stats(params[i], S0[i], r, q, T, n_steps, n_obs, paths=paths, d=d)
        stats.append(st)
        for m in range(M):
            v = payoff(st, n_obs, kind[m], is_call[m], strike[m], barrier[m])
            price[i, m] = disc * v.mean()
            err[i, m] = disc * np.sqrt(v.var(ddof=1) / n_paths) if n_paths > 1 else np.nan
    return price, err, stats
