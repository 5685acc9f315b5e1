"""Extended-precision reference of the Gaussian local score, for tests/test_score_precision.py.

score(c | S) = -(N/2) log( [RSS / (N - k - 1)] / [C_cc / (N - 1)] ),  RSS = C_cc - b' A^-1 b,
A = C[S, S], b = C[S, c], from the centred Gram C taken as exact doubles (its own rounding is not charged to
the scorer).  A set whose A is singular, or that reproduces the child exactly (RSS <= 0), scores -inf.

Two evaluations:
* ``mp_score``: mpmath at MP_BITS bits, from scratch (Cholesky of A).  Edge cases and a seeded subset of
  every bulk check.
* ``SetScores``: every single-edge change of one parent set at once, vectorised, in np.longdouble (64-bit
  significand on x86-64) as the reference and in float64 for the conditioning estimate ``err64`` of the
  tolerance model: one factor of the current set, one bordered row per addition (the exact identity
  rss' = rss - e^2/d), the drop-one-regressor identity per deletion (rss' = rss + (y'z)^2 / (y'y)).

Tolerance model, per item:
    |got - ref| <= K * max(err64, (N/2) (k + 2) eps C_cc / RSS) + 4 eps |ref|
``err64`` is the error of a straightforward float64 evaluation of the same set against the reference: it
carries the conditioning of A.  The second term is the cancellation in RSS = C_cc - z'z (k + 2 roundings of
terms as large as C_cc, relative to RSS, times d score / d log RSS = N/2).  The last term is the rounding of
the score itself (the sweep's logarithm is within 2.5 ulp).  K = 16.
"""
from __future__ import annotations

import mpmath
import numpy as np

MP_BITS = 160
K_TOL = 16.0
EPS = np.finfo(np.float64).eps


def mp_score(Cm, c, S, N):
    """(score as float, RSS as float) of child c on the ordered list S; (-inf, 0.0) when degenerate."""
    S = [int(s) for s in S]
    k = len(S)
    with mpmath.workprec(MP_BITS):
        mpf = mpmath.mpf
        L = [[mpf(0)] * k for _ in range(k)]
        z = [mpf(0)] * k
        for i in range(k):
            for m in range(i + 1):
                acc = mpf(float(Cm[S[i], S[m]]))
                for t in range(m):
                    acc -= L[i][t] * L[m][t]
                if m < i:
                    L[i][m] = acc / L[m][m]
                else:
                    if acc <= 0:
                        return -np.inf, 0.0
                    L[i][i] = mpmath.sqrt(acc)
            acc = mpf(float(Cm[S[i], c]))
            for t in range(i):
                acc -= L[i][t] * z[t]
            z[i] = acc / L[i][i]
        ccc = mpf(float(Cm[c, c]))
        rss = ccc - mpmath.fsum(v * v for v in z)
        if rss <= 0:
            return -np.inf, 0.0
        s = -(mpf(N) / 2) * mpmath.log((rss / (N - k - 1)) / (ccc / (N - 1)))
        return float(s), float(rss)


def f64_score(Cm, c, S, N):
    """Straightforward float64 evaluation (numpy Cholesky + triangular solve); nan where it fails."""
    S = list(S)
    k = len(S)
    ccc = float(Cm[c, c])
    if k == 0:
        rss = ccc
    else:
        try:
            L = np.linalg.cholesky(Cm[np.ix_(S, S)])
        except np.linalg.LinAlgError:
            return np.nan
        z = _fwd(L, Cm[S, c])
        rss = ccc - float(z @ z)
    if not rss > 0:
        return np.nan
    return -(N / 2.0) * np.log((rss / (N - k - 1)) / (ccc / (N - 1)))


def _fwd(L, B):
    """L^-1 B by forward substitution (any dtype; B a vector or a matrix of columns)."""
    X = np.zeros_like(B)
    for i in range(L.shape[0]):
        X[i] = (B[i] - L[i, :i] @ X[:i]) / L[i, i]
    return X


def _chol(A):
    n = A.shape[0]
    L = np.zeros_like(A)
    for i in range(n):
        for m in range(i):
            L[i, m] = (A[i, m] - L[i, :m] @ L[m, :m]) / L[m, m]
        d = A[i, i] - L[i, :i] @ L[i, :i]
        if not d > 0:
            return None
        L[i, i] = np.sqrt(d)
    return L


def tolerance(ref, err64, N, k, ccc, rss):
    """The per-item bound of the module docstring (arrays or scalars); k = parent count of the scored set."""
    cancel = (N / 2.0) * (np.asarray(k) + 2.0) * EPS * ccc / np.maximum(rss, 1e-300)
    e64 = np.where(np.isfinite(err64), err64, 0.0)
    return K_TOL * np.maximum(e64, cancel) + 4 * EPS * np.abs(np.where(np.isfinite(ref), ref, 0.0))


class SetScores:
    """Every single-edge change of child c's ordered parent list S (module docstring), at dtype dt."""

    def __init__(self, Cm, c, S, N, dt):
        C = np.asarray(Cm).astype(dt)
        S = [int(s) for s in S]
        k = len(S)
        P = C.shape[0]
        self.k, self.N = k, N
        ccc = C[c, c]
        half = dt(N) / 2
        syy = ccc / (N - 1)
        self.ccc = float(ccc)
        self.add = np.full(P, -np.inf, dtype=dt)
        self.add_rss = np.zeros(P)
        self.add_dsing = np.zeros(P, bool)
        self.dele = np.full(k, -np.inf, dtype=dt)
        self.del_rss = np.zeros(k)
        L = _chol(C[np.ix_(S, S)]) if k else np.zeros((0, 0), dt)
        self.pd = L is not None
        if not self.pd:
            self.base, self.rss = -np.inf, 0.0
            return
        z = _fwd(L, C[S, c]) if k else np.zeros(0, dt)
        rss = ccc - z @ z
        self.pd = bool(rss > 0)
        self.rss = float(rss)
        self.base = float(-half * np.log((rss / (N - k - 1)) / syy)) if self.pd else -np.inf
        if not self.pd:
            return
        # additions: w = L^-1 C[S, j], d = C_jj - w'w, e = C_jc - w'z
        W = _fwd(L, C[S, :]) if k else np.zeros((0, P), dt)
        d = np.diagonal(C) - np.einsum("ij,ij->j", W, W)
        e = C[c, :] - z @ W
        with np.errstate(divide="ignore", invalid="ignore"):
            rn = rss - e * e / d
            ok = (d > 0) & (rn > 0) & (N - k - 2 > 0)
            self.add = np.where(ok, -half * np.log((rn / (N - k - 2)) / syy), -np.inf).astype(dt)
        self.add_rss = np.where(ok, rn, 0.0).astype(np.float64)
        # |d| / C_jj: a candidate (nearly) in the span of S.  Below ~1e-9 the double route cannot tell an
        # exactly singular enlarged Gram from a near-singular one: -inf and a finite value are both right.
        self.add_dsing = np.abs(d / np.diagonal(C)).astype(np.float64) <= 1e-9
        # deletions: y = column e of L^-1
        if k:
            Y = _fwd(L, np.eye(k, dtype=dt))
            yz = Y.T @ z
            yy = np.einsum("ij,ij->j", Y, Y)
            rd = rss + yz * yz / yy
            self.dele = (-half * np.log((rd / (N - k)) / syy)).astype(dt)
            self.del_rss = rd.astype(np.float64)


def prior_value(phi, omega, dist, total_edges):
    """The chain's LogPrior in the same float64 operations (no contraction): -phi*dist - omega*TotalEdges."""
    return np.float64(-phi) * np.float64(dist) - np.float64(omega) * np.float64(total_edges)
