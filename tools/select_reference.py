"""The reference's selection rule (source/LOD.cc:637-743) evaluated in extended precision on a given fp64 Gram matrix.
Test infrastructure for tests/test_select_*.py.

For the component d, G_o is G without row and column d and g = G[o, d].  The reference takes the SVD of G_o with the
singular values below 1e-15 sigma_0 dropped (:667), d = -G_o^+ g (:669-671), and then drops the smallest singular values
one at a time while ||d||_inf >= 0.5 (:703-725); a thresholded direction counts as a step without changing d.  Finally
c = M^{-1} (e_d + sum_k d_k e_other[k]) (:727-743).  G_o is symmetric, so its SVD is its eigen-decomposition with
sigma = |lambda| and the sign carried by U: d = -sum_k v_k (v_k . g) / lambda_k.

Here the eigen-decomposition is computed in numpy's longdouble (64-bit mantissa on x86-64: eps = 1.1e-19): fp64 eigh as a
start, its vectors re-orthonormalised in extended precision, then cyclic Jacobi sweeps (round-robin order, every
rotation of a round applied at once) until no off-diagonal entry is above eps_ld sqrt(|a_pp a_qq|).  Every candidate
d(r) (r = steps, 0..n) is formed directly from the kept terms, so no cancellation from adding terms back in enters.

The returned margins say how far each discrete decision of the rule is from flipping, on this exact fp64 input."""
import numpy as np

LD = np.longdouble
EPS = 2.220446049250313e-16
EPS_LD = float(np.finfo(LD).eps)
PRECISE = EPS_LD <= 1e-18   # False where longdouble is plain double (e.g. aarch64 with 64-bit long double, MSVC)
THRESHOLD = 1e-15           # singular-value threshold relative to sigma_0 (source/LOD.cc:667)
DINF = 0.5                  # truncation test ||d||_inf < 0.5 (source/LOD.cc:703)


def _orthonormalise(Q):
    """Modified Gram-Schmidt, two passes, in the dtype of Q."""
    Q = Q.copy()
    n = Q.shape[1]
    for j in range(n):
        v = Q[:, j]
        for _ in range(2):
            if j:
                v = v - Q[:, :j] @ (Q[:, :j].T @ v)
        Q[:, j] = v / np.sqrt(v @ v)
    return Q


def eigh_ld(A, max_sweeps=60):
    """(lam, V) with A = V diag(lam) V^T in longdouble; A symmetric (fp64 or longdouble)."""
    A = np.asarray(A, dtype=LD)
    n = A.shape[0]
    if n == 1:
        return A[0].copy(), np.ones((1, 1), dtype=LD)
    _, Q = np.linalg.eigh(A.astype(np.float64))
    V = _orthonormalise(Q.astype(LD))
    B = V.T @ A @ V
    B = (B + B.T) / 2
    m = n + (n & 1)
    # round-robin tournament: round k pairs players (k + i) % (m - 1) and (k - i) % (m - 1), i = 1 .. m/2 - 1, and
    # player m - 1 with k; player n (odd n) is a bye
    rounds = []
    for k in range(m - 1):
        a = [k] + [(k + i) % (m - 1) for i in range(1, m // 2)]
        b = [m - 1] + [(k - i) % (m - 1) for i in range(1, m // 2)]
        p, q = np.minimum(a, b), np.maximum(a, b)
        keep = q < n
        rounds.append((p[keep], q[keep]))
    for _ in range(max_sweeps):
        rotated = 0
        for p, q in rounds:
            app, aqq, apq = B[p, p], B[q, q], B[p, q]
            act = np.abs(apq) > EPS_LD * np.sqrt(np.abs(app * aqq))
            if not act.any():
                continue
            rotated += int(act.sum())
            p, q, app, aqq, apq = p[act], q[act], app[act], aqq[act], apq[act]
            tau = (aqq - app) / (2 * apq)
            t = np.where(tau >= 0, 1, -1).astype(LD) / (np.abs(tau) + np.sqrt(1 + tau * tau))
            c = 1 / np.sqrt(1 + t * t)
            s = t * c
            Bp, Bq = B[:, p].copy(), B[:, q].copy()
            B[:, p], B[:, q] = c * Bp - s * Bq, s * Bp + c * Bq
            Bp, Bq = B[p, :].copy(), B[q, :].copy()
            B[p, :], B[q, :] = c[:, None] * Bp - s[:, None] * Bq, s[:, None] * Bp + c[:, None] * Bq
            Vp, Vq = V[:, p].copy(), V[:, q].copy()
            V[:, p], V[:, q] = c * Vp - s * Vq, s * Vp + c * Vq
        if rotated == 0:
            break
    else:
        raise RuntimeError("Jacobi did not converge")
    return np.diag(B).copy(), V


def split(G, d):
    """(G_o, g, other) of component d (source/LOD.cc:637-662)."""
    G = np.asarray(G, dtype=np.float64)
    other = [k for k in range(G.shape[0]) if k != d]
    return G[np.ix_(other, other)], G[other, d], other


def select(G, Minv, d):
    """The reference's selection on the fp64 matrices G, Minv (n_coarse^2) for component d, in longdouble.

    Returns a dict (arrays in float64 unless named *_ld):
      lam, sigma            eigenvalues of G_o in the reference's (descending sigma) order, sigma = |lam|
      V_ld, lam_ld          eigenvectors / eigenvalues of G_o in that order (longdouble)
      ghat_ld               V^T g
      kept_thr              sigma > 1e-15 sigma_0
      cand                  (n + 1, n): cand[r] = d(r), the answer after r truncation steps
      norms                 ||d(r)||_inf
      steps, d, c           the reference's step count, d = d(steps), c = Minv (e_d + sum d_k e_other[k])
      sigma0, kept_min      sigma_0 and the smallest sigma still used (sigma_0 when none is)
      gap                   smallest kept sigma minus largest dropped one (thresholded or truncated); inf: none dropped
      margin_dinf           min over r <= steps of | ||d(r)||_inf - 0.5 |
      margin_thr            min over k of | sigma_k / sigma_0 - 1e-15 |
    """
    Go, g, other = split(G, d)
    n = Go.shape[0]
    lam, V = eigh_ld(Go)
    order = np.argsort(-np.abs(lam), kind="stable")
    lam, V = lam[order], V[:, order]
    sig = np.abs(lam)
    sig0 = sig[0]
    kept_thr = sig > THRESHOLD * sig0
    ghat = V.T @ np.asarray(g, dtype=LD)
    alpha = np.where(kept_thr, ghat / np.where(lam != 0, lam, 1), 0)
    # S[:, k] = sum_{j < k} v_j alpha_j ; d(r) keeps the n - r largest
    S = np.zeros((n, n + 1), dtype=LD)
    S[:, 1:] = np.cumsum(V * alpha, axis=1)
    cand = -S[:, ::-1].T                    # cand[r] = -S[:, n - r]
    norms = np.abs(cand).max(axis=1)
    steps = int(np.argmax(norms < DINF))    # r = n always qualifies (d = 0)
    dsel = cand[steps]
    used = kept_thr & (np.arange(n) < n - steps)
    kept_min = sig[used].min() if used.any() else sig0
    dropped = ~used
    gap = (kept_min - sig[dropped].max()) if (dropped.any() and used.any()) else np.inf
    e = np.zeros(n + 1, dtype=LD)
    e[d] = 1
    e[other] += dsel
    c = np.asarray(Minv, dtype=LD) @ e
    f = lambda x: np.asarray(x, dtype=np.float64)   # noqa: E731
    return dict(lam=f(lam), sigma=f(sig), lam_ld=lam, V_ld=V, ghat_ld=ghat, kept_thr=kept_thr, cand=f(cand),
                norms=f(norms), steps=steps, d=f(dsel), d_ld=dsel, c=f(c), sigma0=float(sig0), kept_min=float(kept_min),
                gap=float(gap), used=used, n=n,
                margin_dinf=float(np.abs(norms[: steps + 1] - DINF).min()),
                margin_thr=float(np.abs(sig / sig0 - THRESHOLD).min()))


def backward_error(G, d, dvec, ref=None):
    """(||P (G_o x + g)||, 8 n eps (||G_o|| ||x|| + ||g||)) in longdouble for the computed x = dvec; P projects onto
    the eigenvectors the reference keeps (the identity when nothing is dropped).  ||G_o|| = sigma_0."""
    Go, g, _ = split(G, d)
    ref = select(G, np.eye(G.shape[0]), d) if ref is None else ref
    x = np.asarray(dvec, dtype=LD)
    r = np.asarray(Go, dtype=LD) @ x + np.asarray(g, dtype=LD)
    if not ref["used"].all():
        Vk = ref["V_ld"][:, ref["used"]]
        r = Vk @ (Vk.T @ r)
    n = Go.shape[0]
    bound = 8 * n * EPS * (ref["sigma0"] * float(np.sqrt(x @ x)) + float(np.linalg.norm(g)))
    return float(np.sqrt(r @ r)), bound


def forward_bound(ref, r=None):
    """Bound on ||d(r) - d_ref(r)|| (default r: the reference's step count) for any backward-stable fp64 evaluation of
    the rule with the same decisions: 10 n eps sigma_0 / min(kept_min, gap) * (||d_ref|| + ||ghat_dropped|| / kept_min).
    The second term is the error of the kept eigenspace (eps sigma_0 / gap) acting on the dropped components of g."""
    n = ref["n"]
    r = ref["steps"] if r is None else r
    sig = ref["sigma"]
    used = ref["kept_thr"] & (np.arange(n) < n - r)
    if not used.any():
        return 0.0
    kept = sig[used].min()
    drop = ~used
    gap = kept - sig[drop].max() if drop.any() else np.inf
    gd = float(np.sqrt(np.sum(np.asarray(ref["ghat_ld"][drop], dtype=np.float64) ** 2))) if drop.any() else 0.0
    scale = float(np.linalg.norm(ref["cand"][r])) + gd / kept
    return 10 * n * EPS * ref["sigma0"] / min(kept, gap) * scale


def margins_safe(ref, dinf_err=None):
    """True when every decision of the rule on this input is decided beyond rounding: the singular-value threshold by
    more than the 8 n eps sigma_0 an fp64 eigen-solver may move an eigenvalue (Weyl), and every ||d(r)||_inf, r <= steps,
    farther from 0.5 than ``dinf_err`` (default: the forward bound of d(r))."""
    n = ref["n"]
    if ref["margin_thr"] <= 8 * n * EPS:
        return False
    for r in range(ref["steps"] + 1):
        err = forward_bound(ref, r) if dinf_err is None else dinf_err
        if abs(ref["norms"][r] - DINF) <= err:
            return False
    return True
