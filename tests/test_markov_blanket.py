"""Posterior Markov blanket tabulation: mb_freq[i, j] counts the tabulated iterations (those edge_freq counts) after
which i -> j, j -> i, or some node has both i and j as parents.

The reference (tests/emu/mb_replay.cpp) replays the accepted-move log from the start graph, recomputes every
node's blanket from scratch after every move (parents, children and the children's other parents) and integrates
each row over the iterations it held.  It does not use the witness counts the chain keeps.  CPU tests run the
host build of the chain core (tests/emu/host_emu_mb.cpp); GPU tests go through the C ABI
(Context.run(tabulate_markov_blankets=True))."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import ROOT
from test_ancestor_tab import AncLib, _host_lib, _p300, empty_start
from test_ancestor_tab import replay as anc_replay
from test_best_graph import BestLib, EmuBestGraph
from test_chain_resume import (DROP, N_SPLIT, RNG_RMT, RNG_WH, WH_SEEDS, EmuProblem, _synthetic,  # noqa: F401
                               emu_state_lib)

_ip = C.POINTER(C.c_int)


class MbLib:
    """host_emu_mb.cpp behind the entry points of host_emu_state.cpp, so that EmuProblem drives it.  After a run,
    .mb holds mb_freq [P, P] (None when `mb` is off), .anc the ancestor tabulation and .best the best graph (a
    dict) when `anc` / `best` are on."""

    def __init__(self, lib):
        self.lib, self.mb_on, self.anc_on, self.best_on = lib, True, False, False
        self.mb = self.anc = self.best = None
        lib.emu_mb_score_state_len.restype = C.c_longlong

    def emu_score_state_len(self, P, max_par):
        return self.lib.emu_mb_score_state_len(P, max_par)

    def emu_run_chain_state(self, P, max_par, *args):
        self.mb = np.zeros((P, P), np.int32) if self.mb_on else None
        self.anc = np.zeros((P, P), np.int32) if self.anc_on else None
        par = np.full((P, max_par), -7, np.int32)
        npar = np.full(P, -7, np.int32)
        b = EmuBestGraph()
        ptr = lambda a: None if a is None else a.ctypes.data_as(_ip)  # noqa: E731
        rc = self.lib.emu_run_chain_mb(P, max_par, *args, ptr(self.mb), ptr(self.anc),
                                       ptr(par) if self.best_on else None, ptr(npar) if self.best_on else None,
                                       C.byref(b) if self.best_on else None)
        self.best = None
        if self.best_on:
            self.best = dict(parents=par, npar=npar, log_post=b.log_post, log_lik=b.log_lik, log_prior=b.log_prior,
                             iter=int(b.iter), total_edges=int(b.total_edges), found=int(b.found))
        return rc


@pytest.fixture(scope="module")
def mb_lib():
    return MbLib(_host_lib("libbn_emu_mb.so", "host_emu_mb.cpp"))


_replay_lib = None


def replay(par, npar, moves, it0, end, drop, stats=None):
    """mb_freq [i, j] (int64) of a chain that starts at iteration it0 from the graph (par, npar), accepts `moves`
    (iter, movetype, child, parent) and stops before iteration `end`.  stats: a two-element int64 array that
    receives the number of moves that changed some blanket and the (i, j) entries they flipped."""
    global _replay_lib
    if _replay_lib is None:
        _replay_lib = _host_lib("libmb_replay.so", "mb_replay.cpp")
    par, npar = np.ascontiguousarray(par, np.int32), np.ascontiguousarray(npar, np.int32)
    mv = np.ascontiguousarray(np.asarray(moves, np.int32).reshape(-1, 4))
    P = len(npar)
    out = np.zeros((P, P), np.int64)
    rc = _replay_lib.mb_replay(P, par.shape[1], par.ctypes.data_as(_ip), npar.ctypes.data_as(_ip),
                               mv.ctypes.data_as(_ip), mv.shape[0], C.c_longlong(it0), C.c_longlong(end), drop,
                               out.ctypes.data_as(C.POINTER(C.c_longlong)),
                               None if stats is None else stats.ctypes.data_as(C.POINTER(C.c_longlong)))
    assert rc == 0, rc
    return out


def counted(it0, end, drop):
    return max(end, drop) - max(it0, drop)


def check_invariants(mb, edge, n, node_type, max_par):
    """Symmetric; diagonal = tabulated iterations; 0 <= mb <= n; off the diagonal mb >= edge + edge.T (equal at
    MaxPar 1); a sink's row holds its parents only."""
    mb, edge = np.asarray(mb, np.int64), np.asarray(edge, np.int64)   # edge: [child, parent]
    P = mb.shape[0]
    off = ~np.eye(P, dtype=bool)
    both = edge + edge.T
    assert np.array_equal(mb, mb.T)
    assert (np.diagonal(mb) == n).all()
    assert (mb >= 0).all() and (mb <= n).all()
    assert (mb[off] >= both[off]).all()
    if max_par == 1:
        assert np.array_equal(mb[off], both[off])
    sinks = np.flatnonzero(np.asarray(node_type) == 2)
    assert np.array_equal(mb[sinks][off[sinks]], edge[sinks][off[sinks]])


def run(lib, pr, n_iter, **kw):
    out = pr.run(lib, n_iter, **kw)
    out["mb"] = None if lib.mb is None else lib.mb.copy()
    out["anc"] = None if lib.anc is None else lib.anc.copy()
    out["best"] = lib.best
    return out


def check_against_replay(out, pr, start, it0, end, stats=None):
    want = replay(start[0], start[1], out["moves"], it0, end, pr.drop, stats)
    assert np.array_equal(out["mb"].astype(np.int64), want)
    check_invariants(out["mb"], out["freq"], counted(it0, end, pr.drop), pr.nt, pr.max_par)


def _same_outputs(a, b):
    for k in ("iter", "ChangedNode", "movetype", "additions", "deletions", "FN", "FP", "globalLL", "moves", "fpar",
              "fnpar", "freq", "nfreq", "score"):
        assert np.array_equal(a[k], b[k]), k
    for k in ("iter", "valid", "total_edges_member", "additions", "deletions", "uniforms"):
        assert getattr(a["state"], k) == getattr(b["state"], k), k
    assert list(a["state"].wh_state) == list(b["state"].wh_state) and list(a["state"].mt) == list(b["state"].mt)


def _witness_events(par, npar, moves):
    """Python walk of the moves with per-pair witness counts (test coverage only, not the reference): the
    number of moves that removed a witness from a pair that kept at least one."""
    wit = {}
    lists = [list(par[c, :npar[c]]) for c in range(len(npar))]

    def bump(a, b, d):
        key = (min(a, b), max(a, b))
        wit[key] = wit.get(key, 0) + d
        return wit[key]
    for c, pc in enumerate(lists):
        for e, j in enumerate(pc):
            bump(j, c, 1)
            for q in pc[:e]:
                bump(j, q, 1)
    kept = 0
    for _, typ, c, j in moves:
        pc = lists[c]
        if typ == 1:
            bump(j, c, 1)
            for q in pc:
                bump(j, q, 1)
            pc.append(j)
        else:
            pc.remove(j)
            hit = bump(j, c, -1) > 0
            for q in pc:
                hit |= bump(j, q, -1) > 0
            kept += hit
    return kept


# ---------------------------------------------------------------------------
# CPU: the host build of the chain core
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("drop", [0, N_SPLIT // 2])
@pytest.mark.parametrize("kind,seeds", [(RNG_WH, WH_SEEDS), (RNG_RMT, (1234,))])
@pytest.mark.parametrize("max_par", [8, 50])
def test_dataset_matches_replay(mb_lib, emu_state_lib, dataset, max_par, kind, seeds, drop):
    """The shipped dataset (81 nodes), 20,000 iterations: mb_freq equals the replay, and every other output
    equals that of the same run without the tabulation."""
    pr = EmuProblem(dataset["X"], dataset["source"], dataset["target"], dataset["node_type"], max_par, 100, kind,
                    seeds, drop=drop)
    out = run(mb_lib, pr, N_SPLIT)
    assert int((out["moves"][:, 1] == 2).sum()) > 20
    stats = np.zeros(2, np.int64)
    check_against_replay(out, pr, empty_start(pr.P, max_par), 0, N_SPLIT, stats)
    assert stats[0] > 20
    _same_outputs(out, pr.run(emu_state_lib, N_SPLIT))


def test_maxpar1_is_edges_both_ways(mb_lib):
    """300 nodes at MaxPar 1: no node has two parents, so the blanket is the edge in either direction."""
    X, g = _p300(1, seed=31)
    _, first = np.unique(g.target, return_index=True)   # a prior graph with at most one parent per node
    pr = EmuProblem(X, g.source[first], g.target[first], g.node_type_codes(), 1, 100, RNG_WH, WH_SEEDS, drop=3000)
    out = run(mb_lib, pr, N_SPLIT)
    assert int((out["moves"][:, 1] == 2).sum()) > 5
    check_against_replay(out, pr, empty_start(pr.P, 1), 0, N_SPLIT)


def test_p300_maxpar16_many_deletions(mb_lib):
    """300 nodes at MaxPar 16 with hundreds of accepted deletions."""
    X, g = _p300(16)
    pr = EmuProblem(X, g.source, g.target, g.node_type_codes(), 16, 50, RNG_WH, (123, 456, 789), drop=3000,
                    omega=0.2)
    out = run(mb_lib, pr, N_SPLIT)
    assert int((out["moves"][:, 1] == 2).sum()) > 200
    check_against_replay(out, pr, empty_start(pr.P, 16), 0, N_SPLIT)


def test_random_start(mb_lib, dataset):
    """InitialNetwork 1: the start graph is drawn inside chain_init (a zero-iteration run returns it)."""
    pr = EmuProblem(dataset["X"], dataset["source"], dataset["target"], dataset["node_type"], 8, 100, RNG_WH,
                    (77, 88, 99), drop=500, init=1)
    start = run(mb_lib, pr, 0)
    assert int(start["fnpar"].sum()) > 20
    assert (start["mb"] == 0).all()
    out = run(mb_lib, pr, N_SPLIT)
    check_against_replay(out, pr, (start["fpar"], start["fnpar"]), 0, N_SPLIT)


def test_full_node_deleted_down(mb_lib, dataset):
    """A start graph with node 80 at MaxPar 50 parents (1,225 spouse pairs), which the chain then deletes."""
    P, mp = 81, 50
    pr = EmuProblem(dataset["X"], dataset["source"], dataset["target"], np.zeros(P, np.uint8), mp, 100, RNG_WH,
                    (31, 41, 59), drop=0, omega=9.0)
    par, npar = empty_start(P, mp)
    par[80, :] = np.arange(mp)
    npar[80] = mp
    out = run(mb_lib, pr, N_SPLIT, start=(par, npar))
    assert int(((out["moves"][:, 1] == 2) & (out["moves"][:, 2] == 80)).sum()) >= 20
    assert out["fnpar"][80] <= mp - 20
    check_against_replay(out, pr, (par, npar), 0, N_SPLIT)
    # the first tabulated iteration saw every spouse pair
    assert (out["mb"][:mp, :mp] > 0).all()


def test_pair_with_several_witnesses(mb_lib, dataset):
    """0 and 1 share the children 10..15 and 0 -> 1: losing one witness must not take the pair out of the
    blanket."""
    P, mp = 81, 8
    pr = EmuProblem(dataset["X"], dataset["source"], dataset["target"], np.zeros(P, np.uint8), mp, 100, RNG_WH,
                    (2, 3, 5), drop=0, omega=9.0)
    par, npar = empty_start(P, mp)
    par[1, 0], npar[1] = 0, 1
    for c in range(10, 16):
        par[c, :2], npar[c] = (0, 1), 2
    out = run(mb_lib, pr, N_SPLIT, start=(par, npar))
    assert _witness_events(par, npar, out["moves"]) > 0
    check_against_replay(out, pr, (par, npar), 0, N_SPLIT)


def test_drop_on_an_accepted_move(mb_lib, dataset):
    probe = EmuProblem(dataset["X"], dataset["source"], dataset["target"], dataset["node_type"], 8, 100, RNG_WH,
                       WH_SEEDS, drop=0)
    mv = run(mb_lib, probe, N_SPLIT)["moves"]
    t = int(mv[len(mv) // 2, 0])
    pr = EmuProblem(dataset["X"], dataset["source"], dataset["target"], dataset["node_type"], 8, 100, RNG_WH,
                    WH_SEEDS, drop=t)
    out = run(mb_lib, pr, N_SPLIT)
    assert int(out["moves"][len(mv) // 2, 0]) == t
    check_against_replay(out, pr, empty_start(pr.P, 8), 0, N_SPLIT)


def test_end_before_drop(mb_lib, dataset):
    """No tabulated iteration: all zero, and the posterior is NaN."""
    from bayesnetworks_b200 import markov_blanket_posterior
    pr = EmuProblem(dataset["X"], dataset["source"], dataset["target"], dataset["node_type"], 8, 100, RNG_WH,
                    WH_SEEDS, drop=N_SPLIT + 5)
    out = run(mb_lib, pr, N_SPLIT)
    assert len(out["moves"]) > 0 and (out["mb"] == 0).all()
    assert np.isnan(markov_blanket_posterior([out["mb"]])).all()
    check_against_replay(out, pr, empty_start(pr.P, 8), 0, N_SPLIT)


@pytest.mark.parametrize("max_par,kind,seeds", [(8, RNG_WH, WH_SEEDS), (50, RNG_RMT, (99,))])
def test_segments_add_up(mb_lib, dataset, max_par, kind, seeds):
    """Split inside the opening `TotalEdges < 3` phase (1, 2), just before, at and after `drop`, and later: the
    segments' mb_freq sum to the uninterrupted run's, and each segment matches its own replay."""
    pr = EmuProblem(dataset["X"], dataset["source"], dataset["target"], dataset["node_type"], max_par, 10, kind,
                    seeds, drop=DROP)
    full = run(mb_lib, pr, N_SPLIT)
    bounds = [0, 1, 2, DROP - 1, DROP, DROP + 1, 12345, N_SPLIT]
    segs, prev = [], None
    for a, b in zip(bounds[:-1], bounds[1:]):
        if prev is None:
            r = run(mb_lib, pr, b - a)
            start = empty_start(pr.P, max_par)
        else:
            start = (prev["fpar"], prev["fnpar"])
            r = run(mb_lib, pr, b - a, start=start, st_in=prev["state"], score_in=prev["score"])
        assert r["state"].iter == b
        check_against_replay(r, pr, start, a, b)
        segs.append(r)
        prev = r
    assert np.array_equal(sum(s["mb"].astype(np.int64) for s in segs), full["mb"])


def test_with_ancestors_and_best_graph(mb_lib, dataset):
    """All three on in one run: each equals its run alone, and every other output is unchanged."""
    pr = EmuProblem(dataset["X"], dataset["source"], dataset["target"], dataset["node_type"], 8, 100, RNG_WH,
                    WH_SEEDS, drop=4000)
    alone = run(mb_lib, pr, N_SPLIT)
    mb_lib.anc_on = mb_lib.best_on = True
    try:
        both = run(mb_lib, pr, N_SPLIT)
        mb_lib.mb_on = False
        without = run(mb_lib, pr, N_SPLIT)
    finally:
        mb_lib.mb_on, mb_lib.anc_on, mb_lib.best_on = True, False, False
    assert np.array_equal(both["mb"], alone["mb"])
    _same_outputs(both, alone)
    _same_outputs(both, without)
    assert np.array_equal(both["anc"], without["anc"])
    for k, v in both["best"].items():
        assert np.array_equal(v, without["best"][k]), k
    assert both["best"]["found"] == 1
    want = anc_replay(*empty_start(pr.P, 8), both["moves"], 0, N_SPLIT, pr.drop)
    assert np.array_equal(both["anc"].astype(np.int64), want)
    # the ancestor and best-graph host builds agree too
    anc_lib = AncLib(_host_lib("libbn_emu_anc.so", "host_emu_anc.cpp"))
    assert np.array_equal(run_other(anc_lib, pr)["anc"], both["anc"])
    best_lib = BestLib(_host_lib("libbn_emu_best.so", "host_emu_best.cpp"))
    pr.run(best_lib, N_SPLIT)
    assert best_lib.best["log_post"] == both["best"]["log_post"]
    assert np.array_equal(best_lib.best["parents"], both["best"]["parents"])


def run_other(lib, pr):
    out = pr.run(lib, N_SPLIT)
    out["anc"] = lib.anc.copy()
    return out


def test_markov_blanket_posterior_hand_made():
    from bayesnetworks_b200 import markov_blanket_posterior
    # chain 1: 10 iterations, 0 -> 1 in 4 of them; chain 2: 30 iterations, 0 and 2 parents of 1 in 6
    a = np.array([[10, 4, 0], [4, 10, 0], [0, 0, 10]], np.int32)
    b = np.array([[30, 6, 6], [6, 30, 6], [6, 6, 30]], np.int32)
    got = markov_blanket_posterior([a, b])
    want = np.array([[1, 0.25, 0.15], [0.25, 1, 0.15], [0.15, 0.15, 1]])
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-15)
    # int64 pooling: the sum of two chains overflows int32
    big = np.full((2, 2), 2**31 - 1, np.int32)
    np.testing.assert_array_equal(markov_blanket_posterior([big, big]), [[1, 1], [1, 1]])
    # a row without tabulated iterations is NaN
    assert np.isnan(markov_blanket_posterior([np.zeros((2, 2), np.int32)])).all()
    with pytest.raises(ValueError):
        markov_blanket_posterior([np.zeros((2, 3), np.int32)])


# ---------------------------------------------------------------------------
# GPU: the CUDA chains through the C ABI
# ---------------------------------------------------------------------------
def _gpu_pair(ctx, **kw):
    """The same run with and without the tabulation, with want_state=True and as a default run: every other
    output must be the same."""
    on = ctx.run(log_moves=True, tabulate=True, tabulate_markov_blankets=True, want_state=True, **kw)[0]
    for off in (ctx.run(log_moves=True, tabulate=True, want_state=True, **kw)[0],
                ctx.run(log_moves=True, tabulate=True, **kw)[0]):
        for a, b in zip(on, off):
            for k in a.trace:
                assert np.array_equal(a.trace[k], b.trace[k]), k
            for k in ("accepted_moves", "edge_freq", "npar_freq", "final_parents", "final_npar", "mt_state"):
                x, y = getattr(a, k), getattr(b, k)
                assert (x is None and y is None) or np.array_equal(x, y), k
            for k in ("uniforms", "valid_iters", "proposed", "reject", "n_nonpd", "total_edges"):
                assert getattr(a, k) == getattr(b, k), k
            assert b.mb_freq is None
            if b.state is not None:
                assert np.array_equal(a.state.score_block, b.state.score_block)
                for k in ("iter", "valid", "total_edges_member", "additions", "deletions", "uniforms"):
                    assert getattr(a.state, k) == getattr(b.state, k), k
    return on


def _gpu_check(res, node_type, n_iter, drop, max_par, start=None):
    for r in res:
        par, npar = start if start is not None else empty_start(len(r.final_npar), max_par)
        want = replay(par, npar, r.accepted_moves, 0, n_iter, drop)
        assert np.array_equal(r.mb_freq.astype(np.int64), want)
        check_invariants(r.mb_freq, r.edge_freq, counted(0, n_iter, drop), node_type, max_par)


@pytest.mark.gpu
@pytest.mark.parametrize("P", [896, 1000, 1025])
def test_gpu_dense_shapes_match_replay(P):
    """The dense fixtures' inputs (MaxPar 8, thousands of accepted moves), eight chains in one launch."""
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
@pytest.mark.parametrize("shape", ["config3_maxpar50", "large_p_global_memory", "maxpar1"])
def test_gpu_other_shapes_match_replay(shape):
    """Config 3 (100 nodes x 10,000 samples) at MaxPar 50; the 2,500-node shape whose state partly lives in
    global memory; MaxPar 1, where the blanket is the edge either way."""
    from bayesnetworks_b200 import Context
    if shape == "config3_maxpar50":
        X, g, nt = _synthetic(100, 10000, 50, 42)
        mp, nc, kw = 50, 4, dict(output=10, omega=0.3)
    elif shape == "maxpar1":
        X, g, nt = _synthetic(300, 400, 1, 5)
        _, first = np.unique(g.target, return_index=True)   # a prior graph with at most one parent per node
        mp, nc, kw = 1, 4, dict(output=10, omega=2.0)
    else:
        X, g, nt = _synthetic(2500, 120, 4, 9)
        mp, nc, kw = 4, 2, dict(output=50, omega=0.3)
    omega = kw.pop("omega")
    src, tgt = (g.source[first], g.target[first]) if shape == "maxpar1" else (g.source, g.target)
    with Context.from_data(X, src, tgt, nt, max_par=mp, omega=omega) as ctx:
        res = _gpu_pair(ctx, n_chains=nc, n_iter=N_SPLIT, rng="wh", drop=1000, **kw)
    assert min(len(r.accepted_moves) for r in res) > 100
    _gpu_check(res, nt, N_SPLIT, 1000, mp)


@pytest.mark.gpu
def test_gpu_segments_add_up():
    """Eight chains on the shipped dataset, resumed at iterations 1, DROP and 12,345: the segments' mb_freq sum
    to the uninterrupted run's."""
    from bayesnetworks_b200 import Context
    z = np.load(os.path.join(ROOT, "tests", "golden", "network_p3sim8.npz"))
    seeds = np.array([(1000 + 7 * c, 2000 + 11 * c, 3000 + 13 * c) for c in range(8)], np.int32)
    kw = dict(n_chains=8, output=10, rng="wh", drop=DROP, log_moves=True, tabulate=True,
              tabulate_markov_blankets=True, want_state=True)
    with Context.from_data(z["X"], z["source"], z["target"], z["node_type"], max_par=8) as ctx:
        full = ctx.run(n_iter=N_SPLIT, seeds=seeds, **kw)[0]
        parts, start, done = [], None, 0
        for b in (1, DROP, 12345, N_SPLIT):
            r = ctx.run(n_iter=b - done, seeds=seeds if start is None else None, start=start, **kw)[0]
            parts.append(r)
            start, done = [x.state for x in r], b
    for c in range(8):
        total = sum(p[c].mb_freq.astype(np.int64) for p in parts)
        assert np.array_equal(total, full[c].mb_freq)
        assert np.array_equal(np.concatenate([p[c].accepted_moves for p in parts]), full[c].accepted_moves)
    _gpu_check(full, z["node_type"], N_SPLIT, DROP, 8)


@pytest.mark.gpu
def test_gpu_with_ancestors_and_best_graph():
    """The three chain-kernel summaries in one run: each equals its run alone."""
    from bayesnetworks_b200 import Context
    z = np.load(os.path.join(ROOT, "tests", "golden", "network_p3sim8.npz"))
    seeds = np.array([(5 + c, 6 + 2 * c, 7 + 3 * c) for c in range(4)], np.int32)
    kw = dict(n_chains=4, n_iter=N_SPLIT, output=10, rng="wh", drop=DROP, seeds=seeds, log_moves=True, tabulate=True)
    with Context.from_data(z["X"], z["source"], z["target"], z["node_type"], max_par=16) as ctx:
        all3 = ctx.run(tabulate_markov_blankets=True, tabulate_ancestors=True, track_best=True, **kw)[0]
        mb = ctx.run(tabulate_markov_blankets=True, **kw)[0]
        rest = ctx.run(tabulate_ancestors=True, track_best=True, **kw)[0]
    for a, b, c in zip(all3, mb, rest):
        assert np.array_equal(a.mb_freq, b.mb_freq)
        assert np.array_equal(a.anc_freq, c.anc_freq)
        assert a.best.log_post == c.best.log_post and np.array_equal(a.best.parents, c.best.parents)
        for k in a.trace:
            assert np.array_equal(a.trace[k], b.trace[k]) and np.array_equal(a.trace[k], c.trace[k]), k
    _gpu_check(all3, z["node_type"], N_SPLIT, DROP, 16)


@pytest.mark.gpu
def test_gpu_device_outputs():
    """bn_run with device_outputs = 1 and torch device buffers gives the host path's counts."""
    import torch
    from bayesnetworks_b200 import Context, _lib
    from bayesnetworks_b200.api import check
    z = np.load(os.path.join(ROOT, "tests", "golden", "network_p3sim8.npz"))
    nc, n_iter, out_every, P = 4, N_SPLIT, 100, z["X"].shape[1]
    seeds = np.array([(11 + c, 22 + c, 33 + c) for c in range(nc)], np.int32)
    with Context.from_data(z["X"], z["source"], z["target"], z["node_type"], max_par=8) as ctx:
        host = ctx.run(n_chains=nc, n_iter=n_iter, output=out_every, rng="wh", seeds=seeds, drop=DROP,
                       tabulate_markov_blankets=True)[0]
        cap = (n_iter + out_every - 1) // out_every
        dev = torch.device("cuda", 0)
        d_ints = torch.zeros((7, nc, cap), dtype=torch.int32, device=dev)
        d_gll = torch.zeros((nc, cap), dtype=torch.float64, device=dev)
        d_rows = torch.zeros(nc, dtype=torch.int32, device=dev)
        d_mb = torch.full((nc, P, P), -1, dtype=torch.int32, device=dev)
        d_par = torch.zeros((nc, P, 8), dtype=torch.int32, device=dev)
        d_npar = torch.zeros((nc, P), dtype=torch.int32, device=dev)
        ip = lambda t: C.cast(C.c_void_p(t.data_ptr()), _lib._ip)  # noqa: E731
        col = lambda k: C.cast(C.c_void_p(d_ints.data_ptr() + 4 * k * nc * cap), _lib._ip)  # noqa: E731
        tr = _lib.Trace(cap, ip(d_rows), col(0), col(1), col(2), C.cast(C.c_void_p(d_gll.data_ptr()), _lib._dp),
                        col(3), col(4), col(5), col(6))
        args = _lib.RunArgs()
        args.n_chains, args.rng_kind = nc, 0
        args.seeds = seeds.ctypes.data_as(_lib._ip)
        args.initial_network, args.drop = 2, DROP
        args.n_iter, args.output_every, args.device_outputs = n_iter, out_every, 1
        args.mb_freq = ip(d_mb)
        stats = (_lib.ChainStats * nc)()
        ms = C.c_float(0)
        torch.cuda.synchronize()
        check(_lib.lib().bn_run(ctx._h, C.byref(args), C.byref(tr), ip(d_par), ip(d_npar), C.cast(stats, C.c_void_p),
                                C.byref(ms)))
        torch.cuda.synchronize()
        mb = d_mb.cpu().numpy()
        fpar = d_par.cpu().numpy()
    for c in range(nc):
        assert np.array_equal(mb[c], host[c].mb_freq)
        assert np.array_equal(fpar[c], host[c].final_parents)
    assert (np.diagonal(mb, axis1=1, axis2=2) == counted(0, n_iter, DROP)).all()
