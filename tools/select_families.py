"""Seeded synthetic Gram matrices for the selection tests, each designed so that the reference rule
(source/LOD.cc:637-743) takes its decisions with a known margin.  Test infrastructure for tests/test_select_*.py.

A matrix is built from its spectral form: G_o = Q diag(lam) Q^T and g = Q (lam * alpha), so the reference's answer
before truncation is d(0) = -Q alpha, and embedded into an n_coarse x n_coarse G with row / column d holding g.  G is
rounded to fp64, so the designed margins hold only approximately: check_design() evaluates them on the fp64 matrix
with the extended-precision reference, and a margin below its bound is a generator error."""
import zlib

import numpy as np

import select_reference as sr

TRUNCATION_STEPS = (1, 2, 31, 32, 33, 63, 64, 65, 96)   # plus n - 1 and n: across the 32-candidate batches
SCALES = (-200, -60, 60, 200)                          # G -> 2^k G


def orthogonal(n, rng):
    Q, R = np.linalg.qr(rng.standard_normal((n, n)))
    return Q * np.sign(np.diag(R))


def embed(Go, g, d, diag=None):
    """n_coarse x n_coarse G with G[o, o] = Go, G[o, d] = G[d, o] = g (G[d, d] is not read by the selection)."""
    n = Go.shape[0]
    other = [k for k in range(n + 1) if k != d]
    G = np.zeros((n + 1, n + 1))
    G[np.ix_(other, other)] = Go
    G[other, d] = g
    G[d, other] = g
    G[d, d] = np.abs(Go).max() if diag is None else diag
    return G


def from_spectrum(lam, Q, alpha, d):
    Go = (Q * lam) @ Q.T
    Go = (Go + Go.T) / 2
    return embed(Go, Q @ (lam * alpha), d)


def _scaled(Q, alpha, target):
    """alpha scaled so that ||Q alpha||_inf = target."""
    m = np.abs(Q @ alpha).max()
    return alpha * (target / m) if m > 0 else alpha


def _truncated(n, R, lam, Q, rng):
    """alpha for a spectrum in descending order: the n - R largest terms give ||d(R)||_inf = 0.3, and the R smallest
    all push one coordinate i0 the same way, so ||d(r)||_inf >= 0.7 for every r < R."""
    alpha = np.zeros(n)
    k = n - R
    if k > 0:
        alpha[:k] = _scaled(Q[:, :k], rng.standard_normal(k), 0.3)
    i0 = int(np.argmax(np.abs(Q[:, k])))
    alpha[k:] = np.sign(Q[i0, k:]) / abs(Q[i0, k])
    return alpha


def family(name, n, d, seed, R=None):
    """(G, expect): expect holds 'steps' and 'fast' (whether the Cholesky fast path may take it)."""
    rng = np.random.default_rng([seed, n, d, zlib.crc32(name.encode()), R or 0])
    Q = orthogonal(n, rng)
    if name == "fast":        # SPD, cond <= 1e6, ||d||_inf = 0.3
        lam = 10.0 ** (-6 * rng.random(n))
        lam[0] = 1.0
        return from_spectrum(lam, Q, _scaled(Q, rng.standard_normal(n), 0.3), d), dict(steps=0, fast=True)
    if name in ("handoff485", "handoff495"):   # ||d(0)||_inf just below / above the fast path's 0.49 cut
        lam = 10.0 ** (-rng.random(n))
        t = 0.485 if name == "handoff485" else 0.495
        return from_spectrum(lam, Q, _scaled(Q, rng.standard_normal(n), t), d), dict(steps=0, fast=t < 0.49)
    if name == "small_pivot":  # lambda_min = 5e-13 sigma_0 along a direction close to the last coordinate
        lam = 0.9 + 0.1 * rng.random(n)
        lam[-1] = 5e-13
        Q = np.eye(n)
        if n > 1:
            Q[:-1, :-1] = orthogonal(n - 1, rng)
            c, s = np.cos(1e-3), np.sin(1e-3)
            rot = np.eye(n)
            rot[[n - 2, n - 2, n - 1, n - 1], [n - 2, n - 1, n - 2, n - 1]] = [c, -s, s, c]
            Q = Q @ rot
        # ||d||_inf = 0.1: the 0.5 test stays decided although the forward error bound is cond(G_o) eps ||d|| ~ 0.2
        return from_spectrum(lam, Q, _scaled(Q, rng.standard_normal(n), 0.1), d), dict(steps=0, fast=False)
    if name == "indefinite":   # one eigenvalue -1e-8 sigma_0: not SPD, sigma = |lambda| with the sign carried
        lam = 0.1 + 0.9 * rng.random(n)
        lam[0] = 1.0
        lam[rng.integers(1, n) if n > 1 else 0] = -1e-8
        return from_spectrum(lam, Q, _scaled(Q, rng.standard_normal(n), 0.3), d), dict(steps=0, fast=False)
    if name == "truncation":   # well separated spectrum, exactly R truncation steps
        lam = np.logspace(0, -6, n)
        return from_spectrum(lam, Q, _truncated(n, R, lam, Q, rng), d), dict(steps=R, fast=False)
    if name == "clusters":     # kept eigenvalues repeated 2-8 times, three distinct dropped ones below them
        R = min(3, n)
        kept = []
        while len(kept) < n - R:
            m = min(int(rng.integers(2, 9)), n - R - len(kept))
            kept += [10.0 ** (-3 * rng.random())] * m
        lam = np.array(sorted(kept, reverse=True) + [1e-5, 5e-6, 2.5e-6][:R])
        return from_spectrum(lam, Q, _truncated(n, R, lam, Q, rng), d), dict(steps=R, fast=False)
    if name == "zero_load":    # g = 0: d = 0 and c = Minv e_d
        lam = 10.0 ** (-6 * rng.random(n))
        return from_spectrum(lam, Q, np.zeros(n), d), dict(steps=0, fast=True)
    raise ValueError(name)


def cases(n, d, seed=0):
    """Every family at size n for component d: [(label, G, expect)]."""
    out = [(f, *family(f, n, d, seed)) for f in ("fast", "handoff485", "handoff495", "small_pivot", "indefinite",
                                                 "clusters", "zero_load")]
    for R in sorted({r for r in TRUNCATION_STEPS if r <= n} | {max(n - 1, 1), n}):
        out.append((f"truncation{R}", *family("truncation", n, d, seed, R)))
    return out


def check_design(G, d, expect, ref=None):
    """The reference on the fp64 matrix reproduces the design with safe margins; returns the reference."""
    ref = sr.select(G, np.eye(G.shape[0]), d) if ref is None else ref
    assert ref["steps"] == expect["steps"], ("generator error: steps", ref["steps"], expect)
    assert sr.margins_safe(ref), ("generator error: margins", ref["margin_dinf"], ref["margin_thr"])
    if expect["fast"]:
        assert ref["norms"][0] < 0.49 - 1e-3 and ref["lam"].min() > 0
    return ref


def random_minv(ncd, rng):
    """A random symmetric positive definite M^{-1} with condition number <= 10."""
    Q = orthogonal(ncd, rng)
    return (Q * (1.0 + 9.0 * rng.random(ncd))) @ Q.T
