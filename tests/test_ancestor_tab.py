"""Posterior ancestor tabulation: anc_freq[d, a] counts the tabulated iterations (those edge_freq counts) after
which the graph has a directed path a -> ... -> d.

The reference (tests/emu/anc_replay.cpp) replays the accepted-move log from the start graph, recomputes the
whole ancestor closure from scratch after every move and integrates each row over the iterations it held.
CPU tests run the host build of the chain core (tests/emu/host_emu_anc.cpp); GPU tests go through the C ABI
(Context.run(tabulate_ancestors=True))."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT
from test_chain_resume import (DROP, N_SPLIT, RNG_RMT, RNG_WH, WH_SEEDS, EmuProblem, _synthetic,  # noqa: F401
                               emu_state_lib)

_ip = C.POINTER(C.c_int)


def _host_lib(name, src):
    out_dir = os.path.join(ROOT, "tests", "emu", "_build")
    so = os.path.join(out_dir, name)
    src = os.path.join(ROOT, "tests", "emu", src)
    csrc = os.path.join(ROOT, "bayesnetworks_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        os.makedirs(out_dir, exist_ok=True)
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-w",
                               "-x", "c++", f"-I{csrc}", "-o", so, src])
    return C.CDLL(so)


class AncLib:
    """host_emu_anc.cpp behind the entry points of host_emu_state.cpp, so that EmuProblem drives it; the
    anc_freq of the last run is in .anc [descendant, ancestor]."""

    def __init__(self, lib):
        self.lib, self.anc = lib, None
        lib.emu_anc_score_state_len.restype = C.c_longlong

    def emu_score_state_len(self, P, max_par):
        return self.lib.emu_anc_score_state_len(P, max_par)

    def emu_run_chain_state(self, P, *args):
        self.anc = np.zeros((P, P), np.int32)
        return self.lib.emu_run_chain_anc(P, *args, self.anc.ctypes.data_as(_ip))


@pytest.fixture(scope="module")
def anc_lib():
    return AncLib(_host_lib("libbn_emu_anc.so", "host_emu_anc.cpp"))


_replay_lib = None


def replay_lib():
    global _replay_lib
    if _replay_lib is None:
        _replay_lib = _host_lib("libanc_replay.so", "anc_replay.cpp")
    return _replay_lib


def replay(par, npar, moves, it0, end, drop, stats=None):
    """anc_freq [descendant, ancestor] (int64) of a chain that starts at iteration it0 from the graph (par,
    npar), accepts `moves` (iter, movetype, child, parent) and stops before iteration `end`.  stats: a
    two-element int64 array that receives the number of moves that changed the closure and the bits they
    flipped."""
    par, npar = np.ascontiguousarray(par, np.int32), np.ascontiguousarray(npar, np.int32)
    mv = np.ascontiguousarray(np.asarray(moves, np.int32).reshape(-1, 4))
    P = len(npar)
    out = np.zeros((P, P), np.int64)
    rc = replay_lib().anc_replay(P, par.shape[1], par.ctypes.data_as(_ip), npar.ctypes.data_as(_ip),
                                 mv.ctypes.data_as(_ip), mv.shape[0], C.c_longlong(it0), C.c_longlong(end), drop,
                                 out.ctypes.data_as(C.POINTER(C.c_longlong)),
                                 None if stats is None else stats.ctypes.data_as(C.POINTER(C.c_longlong)))
    assert rc == 0, rc
    return out


def counted(it0, end, drop):
    return max(end, drop) - max(it0, drop)


def check_invariants(anc, edge, n, node_type):
    """Diagonal = tabulated iterations; anc >= edge; at most one direction of a pair (acyclic); sources have
    no ancestors and sinks no descendants."""
    anc, edge = np.asarray(anc, np.int64), np.asarray(edge, np.int64)
    P = anc.shape[0]
    off = ~np.eye(P, dtype=bool)
    assert (np.diagonal(anc) == n).all()
    assert (anc >= edge).all()
    assert ((anc + anc.T)[off] <= n).all()
    nt = np.asarray(node_type)
    assert (anc[nt == 1] * off[nt == 1] == 0).all()
    assert (anc[:, nt == 2] * off[:, nt == 2] == 0).all()


def run(lib, pr, n_iter, **kw):
    out = pr.run(lib, n_iter, **kw)
    out["anc"] = lib.anc.copy()
    return out


def empty_start(P, max_par):
    return np.full((P, max_par), -1, np.int32), np.zeros(P, np.int32)


def check_against_replay(out, pr, start, it0, end):
    want = replay(start[0], start[1], out["moves"], it0, end, pr.drop)
    assert np.array_equal(out["anc"].astype(np.int64), want)
    check_invariants(out["anc"], out["freq"], counted(it0, end, pr.drop), pr.nt)


# ---------------------------------------------------------------------------
# CPU: the host build of the chain core
# ---------------------------------------------------------------------------
def _same_outputs(a, b):
    for k in ("iter", "ChangedNode", "movetype", "additions", "deletions", "FN", "FP", "globalLL", "moves", "fpar",
              "fnpar", "freq", "nfreq", "score"):
        assert np.array_equal(a[k], b[k]), k
    for k in ("iter", "valid", "total_edges_member", "additions", "deletions", "uniforms"):
        assert getattr(a["state"], k) == getattr(b["state"], k), k
    assert list(a["state"].wh_state) == list(b["state"].wh_state) and list(a["state"].mt) == list(b["state"].mt)


@pytest.mark.parametrize("drop", [0, N_SPLIT // 2])
@pytest.mark.parametrize("kind,seeds", [(RNG_WH, WH_SEEDS), (RNG_RMT, (1234,))])
@pytest.mark.parametrize("max_par", [8, 50])
def test_dataset_matches_replay(anc_lib, emu_state_lib, dataset, max_par, kind, seeds, drop):
    """The shipped dataset (81 nodes), 20,000 iterations: anc_freq equals the replay, and every other output
    equals that of the same run without the tabulation."""
    pr = EmuProblem(dataset["X"], dataset["source"], dataset["target"], dataset["node_type"], max_par, 100, kind,
                    seeds, drop=drop)
    out = run(anc_lib, pr, N_SPLIT)
    assert int((out["moves"][:, 1] == 2).sum()) > 20
    check_against_replay(out, pr, empty_start(pr.P, max_par), 0, N_SPLIT)
    _same_outputs(out, pr.run(emu_state_lib, N_SPLIT))


def _p300(max_par, seed=11):
    from bayesnetworks_b200.synth import make_dag, make_prior, simulate_numpy
    dag = make_dag(300, seed=seed)
    g = make_prior(dag, max_par=max_par, seed=seed + 1)
    return simulate_numpy(dag, 400, seed=seed + 2), g


def test_p300_maxpar16_many_deletions(anc_lib):
    """300 nodes: rows of three 128-bit chunks, chunk boundaries inside a row; MaxPar 16 with hundreds of
    accepted deletions."""
    X, g = _p300(16)
    pr = EmuProblem(X, g.source, g.target, g.node_type_codes(), 16, 50, RNG_WH, (123, 456, 789), drop=3000,
                    omega=0.2)
    out = run(anc_lib, pr, N_SPLIT)
    assert int((out["moves"][:, 1] == 2).sum()) > 200
    assert (out["anc"][:, 128:] > 0).any() and (out["anc"][:, 256:] > 0).any()
    check_against_replay(out, pr, empty_start(pr.P, 16), 0, N_SPLIT)


def _closure_bits(par, npar):
    """Number of (ancestor, descendant) pairs, a != d, of a DAG (Python, from scratch)."""
    P = len(npar)
    memo = {}
    for d in range(P):
        stack = [d]
        while stack:
            x = stack[-1]
            if x in memo:
                stack.pop()
                continue
            ps = [int(q) for q in par[x, :npar[x]]]
            todo = [q for q in ps if q not in memo]
            if todo:
                stack.extend(todo)
                continue
            v = 1 << x
            for q in ps:
                v |= memo[q]
            memo[x] = v
            stack.pop()
    return sum(bin(v).count("1") for v in memo.values()) - P


def test_p300_path_start_deletions_cut_many_bits(anc_lib):
    """A start graph that is one long path 0 -> 1 -> ... -> 299: its deletions cut hundreds of ancestor bits at
    once."""
    X, g = _p300(4, seed=21)
    P = 300
    pr = EmuProblem(X, g.source, g.target, np.zeros(P, np.uint8), 4, 50, RNG_WH, (321, 654, 987), drop=0)
    par, npar = empty_start(P, 4)
    par[1:, 0] = np.arange(P - 1)
    npar[1:] = 1
    out = run(anc_lib, pr, N_SPLIT, start=(par, npar))
    check_against_replay(out, pr, (par, npar), 0, N_SPLIT)
    # the largest drop of the closure over one accepted deletion, from scratch
    cur, npc, bits, lost = par.copy(), npar.copy(), _closure_bits(par, npar), 0
    for it, typ, c, j in out["moves"][:200]:
        if typ == 1:
            cur[c, npc[c]] = j
            npc[c] += 1
        else:
            e = list(cur[c, :npc[c]]).index(j)
            cur[c, e:npc[c] - 1] = cur[c, e + 1:npc[c]].copy()
            npc[c] -= 1
            cur[c, npc[c]] = -1
        nb = _closure_bits(cur, npc)
        lost = max(lost, bits - nb)
        bits = nb
    assert lost >= 300


def _segments(lib, pr, n_iter, points, start=None):
    bounds = [0] + sorted(set(int(q) for q in points if 0 < q < n_iter)) + [n_iter]
    segs, prev = [], None
    for a, b in zip(bounds[:-1], bounds[1:]):
        if prev is None:
            r = run(lib, pr, b - a, start=start)
        else:
            r = run(lib, pr, b - a, start=(prev["fpar"], prev["fnpar"]), st_in=prev["state"], score_in=prev["score"])
        assert r["state"].iter == b
        r["it0"], r["start"] = a, (start if prev is None else (prev["fpar"], prev["fnpar"]))
        segs.append(r)
        prev = r
    return segs


@pytest.mark.parametrize("max_par,kind,seeds", [(8, RNG_WH, WH_SEEDS), (50, RNG_RMT, (99,))])
def test_segments_add_up(anc_lib, dataset, max_par, kind, seeds):
    """Split inside the opening `TotalEdges < 3` phase (1, 2), just before, at and after `drop`, and later:
    the segments' anc_freq sum to the uninterrupted run's, and each segment matches its own replay."""
    pr = EmuProblem(dataset["X"], dataset["source"], dataset["target"], dataset["node_type"], max_par, 10, kind,
                    seeds, drop=DROP)
    full = run(anc_lib, pr, N_SPLIT)
    segs = _segments(anc_lib, pr, N_SPLIT, [1, 2, DROP - 1, DROP, DROP + 1, 12345])
    assert np.array_equal(sum(s["anc"].astype(np.int64) for s in segs), full["anc"])
    for s in segs:
        start = s["start"] if s["start"] is not None else empty_start(pr.P, max_par)
        check_against_replay(s, pr, start, s["it0"], int(s["state"].iter))


def test_segments_add_up_p300_path(anc_lib):
    X, g = _p300(16)
    P = 300
    pr = EmuProblem(X, g.source, g.target, np.zeros(P, np.uint8), 16, 50, RNG_WH, (5, 6, 7), drop=4000, omega=0.2)
    par, npar = empty_start(P, 16)
    par[1:, 0] = np.arange(P - 1)
    npar[1:] = 1
    full = run(anc_lib, pr, N_SPLIT, start=(par, npar))
    segs = _segments(anc_lib, pr, N_SPLIT, [3999, 4000, 9000], start=(par, npar))
    assert np.array_equal(sum(s["anc"].astype(np.int64) for s in segs), full["anc"])
    check_against_replay(full, pr, (par, npar), 0, N_SPLIT)


def test_ancestor_posterior_hand_made():
    from bayesnetworks_b200 import ancestor_posterior
    # chain 1: 10 iterations, 0 -> 1 in 4 of them, 0 -> 1 -> 2 in 2; chain 2: 30 iterations, 0 -> 2 in 6
    a = np.array([[10, 0, 0], [4, 10, 0], [2, 2, 10]], np.int32)
    b = np.array([[30, 0, 0], [0, 30, 0], [6, 0, 30]], np.int32)
    got = ancestor_posterior([a, b])
    want = np.array([[1, 0, 0], [0.1, 1, 0], [0.2, 0.05, 1]])
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-15)
    # int64 pooling: the sum of two chains overflows int32
    big = np.diag(np.full(2, 2**31 - 1)).astype(np.int32)
    big[1, 0] = 2**31 - 1
    np.testing.assert_array_equal(ancestor_posterior([big, big]), [[1, 0], [1, 1]])
    with pytest.raises(ValueError):
        ancestor_posterior([np.zeros((2, 3), np.int32)])


# ---------------------------------------------------------------------------
# GPU: the CUDA chains through the C ABI
# ---------------------------------------------------------------------------
def _gpu_pair(ctx, **kw):
    """The same run with and without the tabulation: every other output must be the same."""
    on = ctx.run(log_moves=True, tabulate=True, tabulate_ancestors=True, **kw)[0]
    off = ctx.run(log_moves=True, tabulate=True, **kw)[0]
    for a, b in zip(on, off):
        for k in a.trace:
            assert np.array_equal(a.trace[k], b.trace[k]), k
        for k in ("accepted_moves", "edge_freq", "npar_freq", "final_parents", "final_npar", "mt_state"):
            x, y = getattr(a, k), getattr(b, k)
            assert (x is None and y is None) or np.array_equal(x, y), k
        for k in ("uniforms", "valid_iters", "proposed", "reject", "n_nonpd", "total_edges"):
            assert getattr(a, k) == getattr(b, k), k
        assert b.anc_freq is None
    return on


def _gpu_check(res, node_type, n_iter, drop, max_par, start=None):
    for r in res:
        par, npar = start if start is not None else empty_start(len(r.final_npar), max_par)
        want = replay(par, npar, r.accepted_moves, 0, n_iter, drop)
        assert np.array_equal(r.anc_freq.astype(np.int64), want)
        check_invariants(r.anc_freq, r.edge_freq, counted(0, n_iter, drop), node_type)


@pytest.mark.gpu
@pytest.mark.parametrize("P", [896, 1000, 1025])
def test_gpu_dense_shapes_match_replay(P):
    """The dense fixtures' inputs (MaxPar 8, thousands of accepted moves), eight chains in one launch: on
    both sides of the 8-chunk ancestor path (897..1,024 nodes)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_dense_parity import CASES, MAX_PAR, dense_inputs
    from bayesnetworks_b200 import Context
    X, g, nt = dense_inputs(P)
    _, _, phi, omega, _ = CASES[f"p{P}_mid"]
    seeds = np.array([(100 + 7 * c, 200 + 11 * c, 300 + 13 * c) for c in range(8)], np.int32)
    with Context.from_data(X, g.source, g.target, nt, max_par=MAX_PAR, phi=phi, omega=omega) as ctx:
        res = _gpu_pair(ctx, n_chains=8, n_iter=N_SPLIT, output=100, rng="wh", seeds=seeds, drop=7000)
    assert min(int((r.accepted_moves[:, 1] == 2).sum()) for r in res) > 1000
    _gpu_check(res, nt, N_SPLIT, 7000, MAX_PAR)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["config3_maxpar50", "large_p_global_memory"])
def test_gpu_other_shapes_match_replay(shape):
    """Config 3 (100 nodes x 10,000 samples) at MaxPar 50; the 2,500-node shape whose state partly lives in
    global memory."""
    from bayesnetworks_b200 import Context
    if shape == "config3_maxpar50":
        X, g, nt = _synthetic(100, 10000, 50, 42)
        mp, n_iter, nc, kw = 50, N_SPLIT, 4, dict(output=10, omega=0.3)
    else:
        X, g, nt = _synthetic(2500, 120, 4, 9)
        mp, n_iter, nc, kw = 4, N_SPLIT, 2, dict(output=50, omega=0.3)
    omega = kw.pop("omega", 6.9)
    with Context.from_data(X, g.source, g.target, nt, max_par=mp, omega=omega) as ctx:
        res = _gpu_pair(ctx, n_chains=nc, n_iter=n_iter, rng="wh", drop=1000, **kw)
    assert min(len(r.accepted_moves) for r in res) > 100
    _gpu_check(res, nt, n_iter, 1000, mp)


@pytest.mark.gpu
def test_gpu_segments_add_up():
    """Eight chains on the shipped dataset, resumed at iterations 1, DROP and 12,345, with start= / want_state=:
    the segments' anc_freq sum to the uninterrupted run's."""
    from bayesnetworks_b200 import Context
    z = np.load(os.path.join(ROOT, "tests", "golden", "network_p3sim8.npz"))
    seeds = np.array([(1000 + 7 * c, 2000 + 11 * c, 3000 + 13 * c) for c in range(8)], np.int32)
    kw = dict(n_chains=8, output=10, rng="wh", drop=DROP, log_moves=True, tabulate=True, tabulate_ancestors=True,
              want_state=True)
    with Context.from_data(z["X"], z["source"], z["target"], z["node_type"], max_par=8) as ctx:
        full = ctx.run(n_iter=N_SPLIT, seeds=seeds, **kw)[0]
        parts, start, done = [], None, 0
        for b in (1, DROP, 12345, N_SPLIT):
            r = ctx.run(n_iter=b - done, seeds=seeds if start is None else None, start=start, **kw)[0]
            parts.append(r)
            start, done = [x.state for x in r], b
    for c in range(8):
        total = sum(p[c].anc_freq.astype(np.int64) for p in parts)
        assert np.array_equal(total, full[c].anc_freq)
        assert np.array_equal(np.concatenate([p[c].accepted_moves for p in parts]), full[c].accepted_moves)
    _gpu_check(full, z["node_type"], N_SPLIT, DROP, 8)
