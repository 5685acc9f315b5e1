"""The scorers against an extended-precision reference (tests/score_ref.py): score_nodes (every
score_nodes_kernel instantiation), the all-proposal sweep (every sweep_kernel instantiation, its masks and
its logarithm), and the per-node factors the chains keep for MaxPar > 8 over long runs.

Every comparison uses the context's own centred Gram as exact doubles, and the per-item tolerance model of
score_ref.py: K * max(err64, (N/2)(k+2) eps C_cc / RSS) + 4 eps |ref|, K = 16."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from score_ref import EPS, SetScores, f64_score, mp_score, prior_value, tolerance
from test_chain_resume import RNG_WH, WH_SEEDS, EmuProblem, emu_state_lib  # noqa: F401 (fixture)

CSRC = os.path.join(ROOT, "bayesnetworks_b200", "csrc")
DEGENERATE = 1e-11   # RSS / C_cc below this: the Gram route may call the set degenerate (RSS_FLOOR = 1e-13)
SWEEP_LOG_ULP = 2.5  # the bound sweep_log.cuh states


# ---------------------------------------------------------------------------
# sweep_log: host build against logq, device bits against the host build
# ---------------------------------------------------------------------------
def sweep_log_inputs():
    """Both edges of every binade, +-50 ulp around the sqrt(2) split of the mantissa (several binades),
    1 +- k ulp, a dense grid around 1, 2e6 seeded random normal numbers; and non-normal inputs."""
    xs = []
    e = np.arange(-1022, 1024, dtype=np.float64)
    lo = np.ldexp(1.0, e.astype(int))
    xs += [lo, np.ldexp(2.0 - 2.0**-52, e.astype(int)), np.nextafter(lo, np.inf)]
    split = np.int64(0x3FF6A09E) << 32
    for be in (-1000, -30, -1, 0, 1, 30, 1000):
        base = split + (np.int64(be) << 52)
        xs.append((base + np.arange(-50, 51, dtype=np.int64)).view(np.float64))
    k = np.arange(1, 20001, dtype=np.float64)
    xs += [1.0 + k * 2.0**-52, 1.0 - k * 2.0**-53, np.array([1.0])]
    xs.append(np.linspace(0.999, 1.001, 200001))
    xs.append(np.array([0.999059206]))   # the worst input known: 2.41 ulp
    rng = np.random.default_rng(20261021)
    xs.append(rng.integers(0x0010000000000000, 0x7FF0000000000000, 1_000_000, dtype=np.int64).view(np.float64))
    xs.append(rng.uniform(0.25, 4.0, 1_000_000))
    normal = np.ascontiguousarray(np.concatenate(xs))
    bad = np.array([0.0, -0.0, 5e-324, 2.2250738585072009e-308, -1.0, -2.5e-300, np.inf, -np.inf, np.nan, -np.nan])
    return normal, bad


@pytest.fixture(scope="module")
def sweep_log_host(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("sweep_log") / "libsweep_log_host.so")
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-w", "-x", "c++",
                           f"-I{CSRC}", "-o", so, os.path.join(ROOT, "tests", "emu", "sweep_log_host.cpp"),
                           "-lquadmath"])
    return C.CDLL(so)


def _call(fn, x):
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.empty_like(x)
    dp = C.POINTER(C.c_double)
    fn(x.ctypes.data_as(dp), out.ctypes.data_as(dp), C.c_long(x.size))
    return out


def test_sweep_log_error_bound(sweep_log_host):
    normal, bad = sweep_log_inputs()
    err = _call(sweep_log_host.emu_sweep_log_ulp_err, normal)
    worst = int(np.argmax(err))
    assert err[worst] <= SWEEP_LOG_ULP, (normal[worst], err[worst])
    assert err[worst] > 2.0   # the set reaches the function's worst region (2.41 ulp near x = 1)
    assert _call(sweep_log_host.emu_sweep_log, np.array([1.0]))[0] == 0.0
    assert np.all(np.isnan(_call(sweep_log_host.emu_sweep_log, bad)))


DEVICE_SWEEP_LOG = r"""
#include <cuda_runtime.h>
#include "sweep_log.cuh"
__global__ void k(const double* x, double* y, long n) {
  long i = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (i < n) y[i] = bn::sweep_log(x[i]);
}
extern "C" int dev_sweep_log(const double* x, double* y, long n) {
  double *dx = 0, *dy = 0;
  if (cudaMalloc(&dx, n * 8) || cudaMalloc(&dy, n * 8)) return 1;
  cudaMemcpy(dx, x, n * 8, cudaMemcpyHostToDevice);
  k<<<(unsigned)((n + 255) / 256), 256>>>(dx, dy, n);
  cudaMemcpy(y, dy, n * 8, cudaMemcpyDeviceToHost);
  int rc = cudaGetLastError() != cudaSuccess;
  cudaFree(dx); cudaFree(dy);
  return rc;
}
"""


@pytest.mark.gpu
def test_sweep_log_device_bits(sweep_log_host, tmp_path):
    src = tmp_path / "dev_sweep_log.cu"
    src.write_text(DEVICE_SWEEP_LOG)
    so = str(tmp_path / "libdev_sweep_log.so")
    subprocess.check_call([os.environ.get("NVCC", "nvcc"), "-gencode", "arch=compute_100a,code=sm_100a", "-O3",
                           "-std=c++17", "-Xcompiler", "-fPIC", "--shared", f"-I{CSRC}", "-o", so, str(src)])
    dev = C.CDLL(so)
    normal, bad = sweep_log_inputs()
    x = np.concatenate([normal, bad])
    y = np.empty_like(x)
    dp = C.POINTER(C.c_double)
    assert dev.dev_sweep_log(x.ctypes.data_as(dp), y.ctypes.data_as(dp), C.c_long(x.size)) == 0
    host = _call(sweep_log_host.emu_sweep_log, x)
    same = (y.view(np.int64) == host.view(np.int64)) | (np.isnan(y) & np.isnan(host))
    assert same.all(), x[~same][:5]


# ---------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------
def _hadamard(n):
    H = np.array([[1.0]])
    while H.shape[0] < n:
        H = np.block([[H, H], [H, -H]])
    return H


def _check_scores(got, ref, s64, N, k, ccc, rss, what, undecidable=None):
    """got vs the reference under the tolerance model; -inf exactly where the reference is degenerate (and
    allowed where RSS / C_cc is below DEGENERATE).  `undecidable`: items whose enlarged Gram is singular to
    working precision (SetScores.add_dsing) -- any non-NaN value."""
    got, ref = np.asarray(got, float), np.asarray(ref, float)
    assert not np.isnan(got).any(), (what, np.flatnonzero(np.isnan(got))[:5])
    if undecidable is not None and undecidable.any():
        got, ref, keep = got[~undecidable], ref[~undecidable], ~undecidable
        s64 = np.asarray(s64, float)[keep]
        rss = np.broadcast_to(rss, keep.shape)[keep]
    ref_inf = ~np.isfinite(ref)
    assert np.all(got[ref_inf] == -np.inf), (what, np.flatnonzero(ref_inf & (got != -np.inf))[:5])
    fin = ~ref_inf
    band = fin & (np.asarray(rss) * np.ones_like(ref) <= DEGENERATE * np.asarray(ccc))
    ok_inf = got == -np.inf
    assert not np.any(fin & ok_inf & ~band), (what, np.flatnonzero(fin & ok_inf & ~band)[:5])
    chk = fin & ~ok_inf
    tol = tolerance(ref, np.abs(np.asarray(s64, float) - ref), N, k, ccc, rss)
    bad = chk & ~(np.abs(got - ref) <= tol)
    i = np.flatnonzero(bad)[:3]
    assert not bad.any(), (what, i, got[i], ref[i], np.broadcast_to(tol, ref.shape)[i])
    return int(chk.sum())


# ---------------------------------------------------------------------------
# a. score_nodes at every kernel instantiation
# ---------------------------------------------------------------------------
def _score_nodes_data(N, P, seed):
    """Random columns, near-collinear blocks with chosen condition numbers, Walsh columns (exact Gram
    entries: an exact duplicate and an exact sum of two) and a child that is an exact combination."""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((N, P))
    # near-collinear: column j = column j-1 + delta * fresh noise (condition ~ 1/delta^2)
    for j, delta in ((11, 1e-1), (13, 1e-3), (15, 1e-5)):
        X[:, j] = X[:, j - 1] + delta * rng.standard_normal(N)
    H = _hadamard(N)
    X[:, 0], X[:, 1], X[:, 2] = H[:, 1], H[:, 1], H[:, 2]          # 1 duplicates 0
    X[:, 3] = H[:, 1] + H[:, 2]                                    # exact sum of 0 and 2
    X[:, 4] = H[:, 3]
    X[:, 5] = H[:, 1] - H[:, 3]                                    # exact fit child of [0, 4]
    X[:, 6:9] = X[:, 6:9] + 2.0 * X[:, 20:23]                       # some signal
    return X


@pytest.mark.gpu
@pytest.mark.parametrize("max_par", [8, 16, 64])
def test_score_nodes_every_k(max_par):
    from bayesnetworks_b200 import Context
    N, P = 64, 200   # a Walsh column of length 64 has squared norm 8^2: the exact pivots stay exact
    X = _score_nodes_data(N, P, 3 + max_par)
    mean = X.mean(axis=0)
    Xc = X - mean
    with Context.from_stats(N, mean, Xc.T @ Xc, [1], [2], np.zeros(P, np.int32), max_par=max_par) as ctx:
        Cm = ctx.stats()[3]
        rng = np.random.default_rng(max_par)
        items = []   # (child, list, expect_inf)
        for k in range(0, min(max_par, N - 2) + 1):   # N - k - 1 >= 1
            for rep in range(2):
                c = int(rng.integers(30, P))
                S = [int(q) for q in rng.choice([q for q in range(30, P) if q != c], k, replace=False)]
                items.append((c, S, False))
                items.append((c, S[::-1], False))                 # the same set in another order
        # near-collinear sets (conditions ~1e2, 1e6, 1e10) at several sizes
        for j in (11, 13, 15):
            for extra in (0, 3, min(max_par, N - 2) - 2):
                fill = [int(q) for q in rng.choice(np.arange(30, P), extra, replace=False)]
                items.append((7, [j - 1, j] + fill, False))
                items.append((7, fill + [j, j - 1], False))
        # exactly collinear parent Gram / exact fit: -inf
        items += [(20, [0, 1], True), (20, [1, 0], True), (20, [0, 2, 3], True), (20, [2, 0, 3], True),
                  (5, [0, 4], True), (5, [4, 0], True)]
        if max_par >= 4:
            items += [(20, [0, 1, 30, 31], True), (5, [0, 4, 30, 31], True)]
        n = len(items)
        child = np.array([c for c, _, _ in items], np.int32)
        par = np.full((n, max_par), -1, np.int32)
        npar = np.array([len(S) for _, S, _ in items], np.int32)
        for i, (_, S, _) in enumerate(items):
            par[i, :len(S)] = S
        got = ctx.score_nodes(child, par, npar)
        ref = np.empty(n); rss = np.empty(n); s64 = np.empty(n)
        for i, (c, S, inf) in enumerate(items):
            ref[i], rss[i] = mp_score(Cm, c, S, N)
            s64[i] = f64_score(Cm, c, S, N)
            if inf:
                assert ref[i] == -np.inf and got[i] == -np.inf, (c, S, got[i], ref[i])
        ccc = np.array([Cm[c, c] for c in child])
        _check_scores(got, ref, s64, N, npar, ccc, rss, f"score_nodes max_par={max_par}")
        # the two orders of one set agree within tolerance (the reference is order-free)
        pairs = [(i, i + 1) for i in range(0, 4 * (min(max_par, N - 2) + 1), 2)]
        for a, b in pairs:
            t = 2 * tolerance(ref[a], abs(s64[a] - ref[a]), N, npar[a], ccc[a], rss[a])
            assert abs(got[a] - got[b]) <= t, (items[a], got[a], got[b])
    if max_par < N - 2:
        # k = max_par with one residual degree of freedom (N - k - 1 = 1)
        N1 = max_par + 2
        X1 = np.random.default_rng(max_par + 1).standard_normal((N1, 40))
        m1 = X1.mean(axis=0)
        with Context.from_stats(N1, m1, (X1 - m1).T @ (X1 - m1), [1], [2], np.zeros(40, np.int32),
                                max_par=max_par) as ctx1:
            Cm1 = ctx1.stats()[3]
            par = np.array([list(range(1, 1 + max_par)), list(range(39, 39 - max_par, -1))], np.int32)
            child = np.array([0, 0], np.int32)
            got = ctx1.score_nodes(child, par, np.full(2, max_par, np.int32))
            out = [mp_score(Cm1, 0, list(S), N1) for S in par]
            s64 = [f64_score(Cm1, 0, list(S), N1) for S in par]
            _check_scores(got, [o[0] for o in out], s64, N1, max_par, Cm1[0, 0], np.array([o[1] for o in out]),
                          f"score_nodes dof 1 max_par={max_par}")


# ---------------------------------------------------------------------------
# b. / c. the all-proposal sweep
# ---------------------------------------------------------------------------
def _random_graphs(P, MP, n_graphs, rng, first=None):
    """Acyclic graphs whose nodes take every parent count 0..MP (parents from earlier nodes of a random
    order); `first`: (child, [leading parents]) forced at the front of one node's list in graph 0."""
    par = np.full((n_graphs, P, MP), -1, np.int32)
    npar = np.zeros((n_graphs, P), np.int32)
    for g in range(n_graphs):
        order = rng.permutation(P)
        if first is not None and g == 0:
            c, lead = first
            rest = [q for q in order if q != c and q not in lead]
            order = np.array(list(lead) + rest[:MP + 2] + [c] + rest[MP + 2:])
        for pos, c in enumerate(order):
            # node 1 (an exact duplicate of node 0 in the sweep problems) is a parent of `first` only: with 0
            # elsewhere in a list the set is singular only up to rounding, which no precision decides
            cand = [q for q in order[:pos] if q != 1] if first is not None else order[:pos]
            k = min((pos + g) % (MP + 1), len(cand))
            S = list(rng.choice(cand, k, replace=False)) if k else []
            if first is not None and g == 0 and c == first[0]:
                lead = list(first[1])
                S = lead + [q for q in order[:pos] if q not in lead][:MP - 1 - len(lead)]   # below MP: additions stay unmasked
            par[g, c, :len(S)] = S
            npar[g, c] = len(S)
    return par, npar


def _check_sweep(ctx, par, npar, nt, sim, n_sim, phi, omega, N, rng, items=None, n_mp=25):
    """Every output of the sweep (or of the (g, c) `items`) against the reference; the NaN pattern against
    the documented mask; the natural-order launch bit for bit."""
    base, score, hr = ctx.score_all_proposals(par, npar)
    old = os.environ.get("BN_B200_SWEEP_ORDER")
    os.environ["BN_B200_SWEEP_ORDER"] = "0"
    try:
        b2, s2, h2 = ctx.score_all_proposals(par, npar)
    finally:
        if old is None:
            del os.environ["BN_B200_SWEEP_ORDER"]
        else:
            os.environ["BN_B200_SWEEP_ORDER"] = old
    for a, b in ((base, b2), (score, s2), (hr, h2)):
        assert np.array_equal(a.view(np.int64), b.view(np.int64))
    Cm = ctx.stats()[3]
    G, P, MP = par.shape
    if items is None:
        items = [(g, c) for g in range(G) for c in range(P)]
    checked, seen_k, mp_items = 0, set(), []
    te_g = npar.sum(axis=1)
    ag_g = [int(sum(sim[cc, par[g, cc, e]] for cc in range(P) for e in range(npar[g, cc]))) for g in range(G)]
    for g, c in items:
        k = int(npar[g, c])
        S = [int(q) for q in par[g, c, :k]]
        seen_k.add(k)
        ref = SetScores(Cm, c, S, N, np.longdouble)
        r64 = SetScores(Cm, c, S, N, np.float64)
        ccc = ref.ccc
        te, ag = int(te_g[g]), ag_g[g]
        old_prior = prior_value(phi, omega, (te - ag) + (n_sim - ag), te)
        # base
        if ref.pd:
            _check_scores([base[g, c]], [ref.base], [r64.base if r64.pd else np.nan], N, k, ccc, ref.rss, ("base", g, c))
        else:
            assert base[g, c] == -np.inf, (g, c, base[g, c])
        # additions: mask
        member = np.zeros(P, bool)
        member[S] = True
        can_add = nt[c] != 1 and k < MP
        masked = ~member & ((not can_add) | (np.arange(P) == c) | (nt == 2))
        assert np.all(np.isnan(score[g, c, masked])) and np.all(np.isnan(hr[g, c, masked])), (g, c)
        adds = ~member & ~masked
        assert not np.isnan(score[g, c, ~masked]).any(), (g, c, np.flatnonzero(np.isnan(score[g, c]) & ~masked))
        if ref.pd:
            ra = ref.add.astype(float)
            checked += _check_scores(score[g, c, adds], ra[adds], r64.add[adds], N, k + 1, ccc,
                                     ref.add_rss[adds], ("add", g, c), ref.add_dsing[adds])
        else:
            assert np.all(score[g, c, adds] == -np.inf), (g, c)
            ra = np.full(P, -np.inf)
        # deletions (from scratch when the current set is degenerate)
        if k:
            if ref.pd:
                rd, rd64, rdr = ref.dele.astype(float), r64.dele, ref.del_rss
            else:
                outs = [mp_score(Cm, c, S[:e] + S[e + 1:], N) for e in range(k)]
                rd = np.array([o[0] for o in outs]); rdr = np.array([o[1] for o in outs])
                rd64 = np.array([f64_score(Cm, c, S[:e] + S[e + 1:], N) for e in range(k)])
            checked += _check_scores(score[g, c, S], rd, rd64, N, k - 1, ccc, rdr, ("del", g, c))
        # log Hastings ratios: (new - old) + NewLogPrior - OldLogPrior, IEEE semantics for -inf
        add_p = np.where(sim[c] != 0, prior_value(phi, omega, (te - ag) + (n_sim - ag - 1), te + 1),
                         prior_value(phi, omega, (te + 1 - ag) + (n_sim - ag), te + 1))
        want = np.full(P, np.nan)
        with np.errstate(invalid="ignore"):
            want[adds] = (score[g, c, adds] - base[g, c]) + add_p[adds] - old_prior
            for e, j in enumerate(S):
                a1 = int(sim[c, j])
                newp = prior_value(phi, omega, (te - 1 - (ag - a1)) + (n_sim - (ag - a1)), te - 1)
                want[j] = (score[g, c, j] - base[g, c]) + newp - old_prior
        got_h = hr[g, c]
        nan_w = np.isnan(want)
        assert np.array_equal(nan_w, np.isnan(got_h)), (g, c, np.flatnonzero(nan_w != np.isnan(got_h))[:5])
        fin = np.isfinite(want)
        assert np.array_equal(want[~nan_w & ~fin], got_h[~nan_w & ~fin]), (g, c)
        slack = 8 * EPS * (np.abs(score[g, c]) + abs(base[g, c]) + abs(old_prior) + np.abs(add_p) + 1.0)
        assert np.all(np.abs(got_h[fin] - want[fin]) <= slack[fin]), (g, c)
        # the Hastings ratio against the reference scores (catches a wrong prior term)
        ref_row = ra.copy()
        if k:
            ref_row[S] = rd
        okr = fin & np.isfinite(ref_row)
        if ref.pd and okr.any():
            want_ref = (ref_row - ref.base) + np.where(member, want - (score[g, c] - base[g, c]), add_p - old_prior)
            assert np.all(np.abs(got_h[okr] - want_ref[okr]) <= 1e-6 * (1 + np.abs(want_ref[okr]))), (g, c)
        if len(mp_items) < n_mp and rng.random() < 0.05:
            j = int(rng.choice(np.flatnonzero(adds | member))) if (adds | member).any() else None
            if j is not None:
                mp_items.append((g, c, S, j))
    # a seeded subset re-solved from scratch at MP_BITS bits: kernel and bulk reference
    for g, c, S, j in mp_items:
        T = [q for q in S if q != j] if j in S else S + [j]
        want, rss = mp_score(Cm, c, T, N)
        got = score[g, c, j]
        if np.isfinite(want) and got != -np.inf:
            t = tolerance(want, abs(f64_score(Cm, c, T, N) - want), N, len(T), Cm[c, c], rss)
            assert abs(got - want) <= t, (g, c, j, got, want, t)
    return checked, seen_k


def _sweep_problem(P, N, seed):
    from bayesnetworks_b200.synth import make_dag, simulate_numpy
    dag = make_dag(P, seed=seed)
    X = simulate_numpy(dag, N, seed=seed + 1)
    H = _hadamard(N)
    X[:, 0], X[:, 1], X[:, 2] = H[:, 1], H[:, 1], H[:, 5]     # node 1 duplicates node 0 exactly
    rng = np.random.default_rng(seed)
    nt = np.zeros(P, np.int32)
    nt[rng.choice(np.arange(10, P), P // 12, replace=False)] = 1
    nt[rng.choice(np.flatnonzero(nt == 0)[5:], P // 12, replace=False)] = 2
    prior = make_dag(P, seed=seed + 7)   # a different DAG as the prior: FP > 0 and FN > 0
    src = [p + 1 for c in range(P) for p in prior.parents[c]]
    tgt = [c + 1 for c in range(P) for p in prior.parents[c]]
    return X, nt, src, tgt


@pytest.mark.gpu
@pytest.mark.parametrize("max_par", [8, 16, 64])
def test_sweep_every_output(max_par):
    from bayesnetworks_b200 import Context
    P, N, phi, omega = 300, 256, 0.7, 2.3
    X, nt, src, tgt = _sweep_problem(P, N, 40 + max_par)
    mean = X.mean(axis=0)
    Xc = X - mean
    rng = np.random.default_rng(max_par)
    bad = int(np.flatnonzero(nt == 0)[10])   # a node whose list starts with the exact duplicate pair
    par, npar = _random_graphs(P, max_par, 3, rng, first=(bad, [0, 1]))
    sim = np.zeros((P, P), np.uint8)
    for s, t in zip(src, tgt):
        sim[t - 1, s - 1] = 1
    with Context.from_stats(N, mean, Xc.T @ Xc, src, tgt, nt, max_par=max_par, phi=phi, omega=omega) as ctx:
        base, score, _ = ctx.score_all_proposals(par, npar)
        checked, seen_k = _check_sweep(ctx, par, npar, nt, sim, len(src), phi, omega, N, rng)
    assert seen_k >= set(range(max_par + 1))
    for g in range(3):
        te = int(npar[g].sum())
        ag = int(sum(sim[c, par[g, c, e]] for c in range(P) for e in range(npar[g, c])))
        assert te - ag > 0 and len(src) - ag > 0     # FP > 0, FN > 0
    # the degenerate node: base -inf, additions -inf, deletions of a duplicate finite
    assert base[0, bad] == -np.inf
    k = int(npar[0, bad])
    S = list(par[0, bad, :k])
    assert k < max_par and np.isfinite(score[0, bad, 0]) and np.isfinite(score[0, bad, 1])
    assert np.all(score[0, bad, S[2:]] == -np.inf)
    adds = np.ones(P, bool); adds[S] = False; adds[bad] = False; adds &= nt != 2
    assert adds.sum() > 100 and np.all(score[0, bad, adds] == -np.inf)
    assert checked > 50000


@pytest.mark.gpu
def test_sweep_shipped_dataset(dataset):
    from bayesnetworks_b200 import Context
    X = dataset["X"]
    N, P = X.shape
    phi, omega, MP = 1.0, 6.9, 50
    rng = np.random.default_rng(81)
    par, npar = _random_graphs(P, MP, 3, rng)
    sim = np.zeros((P, P), np.uint8)
    for s, t in zip(dataset["source"], dataset["target"]):
        sim[t - 1, s - 1] = 1
    with Context.from_data(X, dataset["source"], dataset["target"], dataset["node_type"], max_par=MP) as ctx:
        checked, seen_k = _check_sweep(ctx, par, npar, np.asarray(dataset["node_type"]), sim,
                                       len(dataset["source"]), phi, omega, N, rng)
    assert max(seen_k) == MP and checked > 10000


@pytest.mark.gpu
def test_sweep_benchmark_shape():
    """1,000 nodes, MaxPar 8, 64 graphs: the whole NaN mask, and scores / ratios of a seeded sample of
    (graph, child) sets spread over every graph and every parent count."""
    from bayesnetworks_b200 import Context
    from bayesnetworks_b200.synth import make_dag, make_prior, simulate_numpy
    P, N, G, MP = 1000, 2000, 64, 8
    dag = make_dag(P, seed=11)
    g = make_prior(dag, max_par=MP, seed=12)
    X = simulate_numpy(dag, N, seed=13)
    nt = np.asarray(g.node_type_codes(), np.int32)
    rng = np.random.default_rng(64)
    par, npar = _random_graphs(P, MP, G, rng)
    sim = np.zeros((P, P), np.uint8)
    for s, t in zip(g.source, g.target):
        sim[t - 1, s - 1] = 1
    with Context.from_data(X, g.source, g.target, nt, max_par=MP) as ctx:
        base, score, hr = ctx.score_all_proposals(par, npar)
        member = np.zeros((G, P, P), bool)
        for gg in range(G):
            for c in range(P):
                member[gg, c, par[gg, c, :npar[gg, c]]] = True
        full = (npar >= MP)[:, :, None] | (nt == 1)[None, :, None] | (nt == 2)[None, None, :] | np.eye(P, dtype=bool)[None]
        mask = ~member & full
        assert np.array_equal(np.isnan(score), mask) and np.array_equal(np.isnan(hr), mask)
        items = []
        for gg in range(G):
            for k in range(MP + 1):
                cs = np.flatnonzero(npar[gg] == k)
                items += [(gg, int(c)) for c in rng.choice(cs, min(2, cs.size), replace=False)]
        checked, seen_k = _check_sweep(ctx, par, npar, nt, sim, len(g.source), 1.0, 6.9, N, rng, items=items)
    assert seen_k == set(range(MP + 1)) and checked >= 50000


# ---------------------------------------------------------------------------
# d. additions without residual degrees of freedom
# ---------------------------------------------------------------------------
@pytest.mark.gpu
def test_sweep_zero_dof_addition():
    """N = 12, MaxPar 16: a node with N - 2 = 10 parents; an addition leaves N - k - 2 = 0 degrees of
    freedom and scores -inf (the chain's value), never NaN."""
    from bayesnetworks_b200 import Context
    N, P, MP = 12, 30, 16
    rng = np.random.default_rng(0)
    X = rng.standard_normal((N, P))
    for a in (4, 6, 8):   # near-collinear parents: the exact fit's RSS is rounding noise well above the floor
        X[:, a] = X[:, a - 1] + 1e-5 * rng.standard_normal(N)
    mean = X.mean(axis=0)
    Xc = X - mean
    par = np.full((P, MP), -1, np.int32)
    npar = np.zeros(P, np.int32)
    for c, k in ((0, N - 2), (1, N - 3), (2, N - 1)):
        S = list(range(3, 3 + k)) if c == 0 else list(range(15, 15 + k))
        par[c, :k] = S
        npar[c] = k
    with Context.from_stats(N, mean, Xc.T @ Xc, [1], [2], np.zeros(P, np.int32), max_par=MP) as ctx:
        base, score, hr = ctx.score_all_proposals(par, npar)
    member = np.zeros(P, bool); member[par[0, :npar[0]]] = True
    adds = ~member & (np.arange(P) != 0)
    assert not np.isnan(score[0, 0, 1:]).any() and not np.isnan(hr[0, 0, 1:]).any()   # (j = c is masked)
    assert np.all(score[0, 0, adds] == -np.inf)
    assert np.isfinite(base[0, 0]) and np.all(np.isfinite(score[0, 0, member]))
    adds1 = np.ones(P, bool); adds1[par[1, :npar[1]]] = False; adds1[1] = False
    assert np.all(np.isfinite(score[0, 1, adds1]))   # one degree of freedom left: finite


# ---------------------------------------------------------------------------
# the chains' factor cache: long runs on the host build, large parent sets
# ---------------------------------------------------------------------------
def mp_factor(Cm, c, S):
    """(L, z, rss) of the ordered list S at MP_BITS bits, as floats."""
    import mpmath
    from score_ref import MP_BITS
    k = len(S)
    with mpmath.workprec(MP_BITS):
        A = mpmath.matrix([[float(Cm[a, b]) for b in S] for a in S]) if k else None
        L = np.zeros((k, k)); z = np.zeros(k)
        Lm = [[mpmath.mpf(0)] * k for _ in range(k)]
        zm = [mpmath.mpf(0)] * k
        for i in range(k):
            for m in range(i + 1):
                acc = A[i, m] - mpmath.fsum(Lm[i][t] * Lm[m][t] for t in range(m))
                Lm[i][m] = acc / Lm[m][m] if m < i else mpmath.sqrt(acc)
            zm[i] = (mpmath.mpf(float(Cm[S[i], c])) - mpmath.fsum(Lm[i][t] * zm[t] for t in range(i))) / Lm[i][i]
        rss = mpmath.mpf(float(Cm[c, c])) - mpmath.fsum(v * v for v in zm)
        for i in range(k):
            z[i] = float(zm[i])
            for m in range(i + 1):
                L[i, m] = float(Lm[i][m])
        return L, z, float(rss)


def _fac_geom(mp):
    row = lambda i: 2 * (i >> 1) * ((i >> 1) + 1) + (i & 1) * (2 * (i >> 1) + 2)
    zoff = row(mp)
    tail = row(mp) + ((mp + 1) & ~1)
    stride = (tail + 2 + 3) & ~3
    return row, zoff, tail, stride


def check_score_block(block, Cm, fpar, fnpar, N, max_par, bound):
    """The score block of a chain (base[P], then per node: rows of L with 1 / L[i][i] on the diagonal, z,
    rss) against an MP_BITS refactorisation of the final lists: relative errors (base to |base| + 1, L rows
    to sqrt(A_ii), z to sqrt(C_cc), rss to C_cc) within `bound`.  Returns the worst relative error."""
    P = len(fnpar)
    row, zoff, tail, stride = _fac_geom(max(max_par, 8))
    worst = 0.0
    for c in range(P):
        k = int(fnpar[c])
        S = [int(q) for q in fpar[c, :k]]
        ref, rss_ref = mp_score(Cm, c, S, N)
        if not np.isfinite(ref):
            assert block[c] == -np.inf
            continue
        worst = max(worst, abs(block[c] - ref) / (abs(ref) + 1.0))
        if max_par <= 8:
            continue
        F = block[P + c * stride: P + (c + 1) * stride]
        L, z, rss = mp_factor(Cm, c, S)
        for i in range(k):
            sc = np.sqrt(Cm[S[i], S[i]])
            worst = max(worst, np.max(np.abs(F[row(i):row(i) + i] - L[i, :i]), initial=0.0) / sc,
                        abs(1.0 / F[row(i) + i] - L[i, i]) / sc)
        if k:
            worst = max(worst, np.max(np.abs(F[zoff:zoff + k] - z)) / np.sqrt(Cm[c, c]))
        worst = max(worst, abs(F[tail] - rss) / Cm[c, c])
    assert worst <= bound, worst
    return worst


def _synthetic(P, N, max_par, seed):
    from bayesnetworks_b200.synth import make_dag, make_prior, simulate_numpy
    dag = make_dag(P, seed=seed)
    g = make_prior(dag, max_par=max_par, seed=seed + 1)
    X = simulate_numpy(dag, N, seed=seed + 2)
    return X, g


# Bound of the long-run checks: the measured worst over 2e6 iterations is 5.6e-13 (MaxPar 16) and 2.8e-12
# (MaxPar 50) relative, growing about tenfold per hundredfold more accepted deletions (Givens downdates
# accumulate rounding); 1e-10 keeps a factor > 30 of headroom over that and still sits 10x inside the
# 1e-9 parity bar, so a drift that could reach the bar within such a run fails here first.
DRIFT_BOUND = 1e-10


@pytest.mark.parametrize("P,max_par,omega", [(40, 16, 0.2), (70, 50, 0.05)])
def test_factor_drift_long_run(emu_state_lib, P, max_par, omega):
    X, g = _synthetic(P, 500, max_par, 100 + max_par)
    pr = EmuProblem(X, g.source, g.target, g.node_type_codes(), max_par, 100000, RNG_WH, WH_SEEDS, omega=omega)
    out = pr.run(emu_state_lib, 2_000_000)
    dels = int((out["moves"][:, 1] == 2).sum())
    assert dels > 100000
    check_score_block(out["score"], pr.Cm, out["fpar"], out["fnpar"], pr.N, max_par, DRIFT_BOUND)


def test_global_ll_every_iteration(emu_state_lib, oracle):
    """50k iterations, output 1, MaxPar 16: every logged globalLL against the MP_BITS sum of the node
    scores of the graph replayed from the move log; the trajectory (every proposal's score through its
    acceptance) against the oracle's."""
    X, g = _synthetic(40, 500, 16, 116)
    pr = EmuProblem(X, g.source, g.target, g.node_type_codes(), 16, 1, RNG_WH, WH_SEEDS, omega=0.2, init=0)
    out = pr.run(emu_state_lib, 50_000)
    ref = oracle.mcmc(X, g.source, g.target, g.node_type_codes(), max_par=16, omega=0.2, initial_network=0,
                      n_iter=50_000, output=1, rng_kind=RNG_WH, seeds=WH_SEEDS)
    for k in ("iter", "ChangedNode", "movetype", "additions", "deletions", "FN", "FP"):
        assert np.array_equal(out[k], getattr(ref, k)), k
    lists = [list(pr.ppar[c, :pr.pnpar[c]]) for c in range(pr.P)]
    cache = {}

    def node(c):
        key = (c, tuple(lists[c]))
        if key not in cache:
            s, rss = mp_score(pr.Cm, c, lists[c], pr.N)
            cache[key] = (s, (pr.N / 2) * (len(lists[c]) + 2) * EPS * pr.Cm[c, c] / max(rss, 1e-300))
        return cache[key]

    mv = out["moves"]
    mi = 0
    nodes = [node(c) for c in range(pr.P)]
    for it, gll in zip(out["iter"], out["globalLL"]):
        while mi < len(mv) and mv[mi, 0] <= it:
            _, mt, c, j = mv[mi]
            if mt == 1:
                lists[c].append(int(j))
            else:
                lists[c].remove(int(j))
            nodes[c] = node(c)
            mi += 1
        ref = sum(s for s, _ in nodes)
        tol = 16 * sum(t for _, t in nodes) + 1e-12 * abs(ref) + 1e-9
        assert abs(gll - ref) <= tol, (it, gll, ref, tol)
    assert mi == len(mv) and len(mv) > 1000


def _large_k_start(P, max_par, rng, ks):
    """Lists in which the last len(ks) nodes of a random order hold ks parents (earlier nodes), the rest 0-3."""
    order = rng.permutation(P)
    par = np.full((P, max_par), -1, np.int32)
    npar = np.zeros(P, np.int32)
    for pos, c in enumerate(order):
        k = ks[pos - (P - len(ks))] if pos >= P - len(ks) else int(rng.integers(0, 4))
        k = min(k, pos)
        par[c, :k] = rng.choice(order[:pos], k, replace=False)
        npar[c] = k
    return par, npar


def k_occupancy(moves, npar0, n_iter, max_par):
    """From the accepted-move log (rows iter, movetype, child, parent): node-iterations spent at each parent
    count, and accepted moves by the parent count they were proposed at."""
    k = np.asarray(npar0, np.int64).copy()
    since = np.zeros(len(k), np.int64)
    held = np.zeros(max_par + 1, np.int64)
    moved = np.zeros(max_par + 1, np.int64)
    for it, mt, c, _ in moves:
        held[k[c]] += it - since[c]
        moved[k[c]] += 1
        since[c] = it
        k[c] += 1 if mt == 1 else -1
    for c in range(len(k)):
        held[k[c]] += n_iter - since[c]
    return held, moved


# nodes at exactly 31 and 32 parents (the device's warp-cooperative proposal scorer takes sets of 9..32 and
# uses every lane and the last row pair at 31 / 32) and at 33..64 (the streamed scorer, two rows per lane)
LARGE_KS = (30, 30, 31, 31, 31, 32, 32, 32, 33, 36, 40, 47, 52, 58, 63, 64)


def _large_k_problem(max_par):
    """P 100, N 400, a start graph with LARGE_KS nodes; the prior has the same edges (initial_network 0 starts
    the chain from it) and omega 0, phi 2, so that large sets survive and change slowly."""
    rng = np.random.default_rng(max_par)
    X, _ = _synthetic(100, 400, max_par, 200 + max_par)
    par, npar = _large_k_start(100, max_par, rng, [min(k, max_par) for k in LARGE_KS])
    src = [int(par[c, e]) + 1 for c in range(100) for e in range(npar[c])]
    tgt = [c + 1 for c in range(100) for e in range(npar[c])]
    return X, src, tgt, np.zeros(100, np.int32), par, npar


def _assert_large_k_coverage(moves, npar0, n_iter, max_par):
    held, moved = k_occupancy(moves, npar0, n_iter, max_par)
    for k in (31, 32):   # a node at k for a quarter of the run on average, and accepted moves made there
        assert held[k] >= n_iter // 4 and moved[k] >= 10, (k, held[k], moved[k])
    assert held[33:].sum() >= 4 * n_iter and moved[33:].sum() >= 20, (held[33:].sum(), moved[33:].sum())
    assert moved[9:33].sum() >= 20


@pytest.mark.parametrize("max_par", [50, 64])
def test_host_large_parent_sets(emu_state_lib, oracle, max_par):
    """Nodes at 31, 32 and 33..max_par parents on the host build: score_move_stream and factor_downdate at
    large k.  The trajectory against the oracle's, the final score block against a refactorisation."""
    X, src, tgt, nt, par, npar = _large_k_problem(max_par)
    pr = EmuProblem(X, src, tgt, nt, max_par, 1000, RNG_WH, WH_SEEDS, phi=2.0, omega=0.0, init=0)
    out = pr.run(emu_state_lib, 100_000)
    ref = oracle.mcmc(X, src, tgt, nt, max_par=max_par, phi=2.0, omega=0.0, initial_network=0, n_iter=100_000,
                      output=1000, rng_kind=RNG_WH, seeds=WH_SEEDS)
    for k in ("iter", "ChangedNode", "movetype", "additions", "deletions", "FN", "FP"):
        assert np.array_equal(out[k], getattr(ref, k)), k
    assert np.array_equal(out["moves"], ref.accepted_moves())
    _assert_large_k_coverage(out["moves"], npar, 100_000, max_par)
    check_score_block(out["score"], pr.Cm, out["fpar"], out["fnpar"], pr.N, max_par, DRIFT_BOUND)


@pytest.mark.gpu
def test_chain_large_parent_sets_against_oracle():
    """MaxPar 64 chains on the device with nodes at 31, 32 and 33..64 parents: the warp-cooperative scorer at
    k = 31 / 32, the streamed scorer above 32, appended rows and Givens downdates.  Bit-identical integer
    columns, move log and uniforms against the oracle, globalLL within 1e-9, the final score block against
    a refactorisation of the final lists (base within the tolerance model)."""
    from bayesnetworks_b200 import Context
    max_par, n_iter = 64, 20_000
    X, src, tgt, nt, par, npar = _large_k_problem(max_par)
    N = X.shape[0]
    ref = _oracle().mcmc(X, src, tgt, nt, max_par=max_par, phi=2.0, omega=0.0, initial_network=0, n_iter=n_iter,
                         output=1, rng_kind=RNG_WH, seeds=WH_SEEDS)
    with Context.from_data(X, src, tgt, nt, max_par=max_par, phi=2.0, omega=0.0) as ctx:
        r = ctx.run(n_chains=1, n_iter=n_iter, output=1, initial_network=0, rng="wh", seeds=WH_SEEDS,
                    log_moves=True, want_state=True)[0][0]
        Cm = ctx.stats()[3]
    for k in ("iter", "ChangedNode", "movetype", "additions", "deletions", "FN", "FP"):
        assert np.array_equal(r.trace[k], getattr(ref, k)), k
    assert np.array_equal(r.accepted_moves, ref.accepted_moves())
    assert r.uniforms == ref.uniforms
    np.testing.assert_allclose(r.trace["globalLL"], ref.globalLL, rtol=1e-9, atol=1e-9 * N / 2)
    _assert_large_k_coverage(r.accepted_moves, npar, n_iter, max_par)
    block = r.state.score_block
    check_score_block(block, Cm, r.final_parents, r.final_npar, N, max_par, DRIFT_BOUND)
    for c in range(len(npar)):
        S = [int(q) for q in r.final_parents[c, :r.final_npar[c]]]
        want, rss = mp_score(Cm, c, S, N)
        _check_scores([block[c]], [want], [f64_score(Cm, c, S, N)], N, len(S), Cm[c, c], rss, ("block", c))


def _oracle():
    from oracle.oracle import Oracle
    return Oracle()
