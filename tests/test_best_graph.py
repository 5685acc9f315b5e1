"""Best graph visited: for each chain, the graph with the highest log_lik + log_prior among the graphs
edge_freq counts (a graph created at t and replaced at t' counts iff t' > D = max(drop, iter0); the final one
iff end > D), the first to reach the maximum winning ties.

The reference, `replay` below, is independent of the tracking code: it replays the accepted-move log from
the start graph, takes each created graph's log_lik from the trace row of its creation iteration (runs
with output = 1: an accepted iteration is always logged, and its row sees the post-move graph), the start
graph's from a trace row before the first accepted move or from the start's score block summed in the
chain's order, and the log prior from the replayed TotalEdges / Nagree with the chain's operation order
(float64, round to nearest, no contraction).  CPU tests run the host build of the chain core
(tests/emu/host_emu_best.cpp); GPU tests go through the C ABI (Context.run(track_best=True))."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from test_chain_resume import (DROP, N_SPLIT, RNG_RMT, RNG_WH, WH_SEEDS, EmuProblem, _synthetic,  # noqa: F401
                               emu_state_lib)

_ip = C.POINTER(C.c_int)


class EmuBestGraph(C.Structure):
    _fields_ = [("log_post", C.c_double), ("log_lik", C.c_double), ("log_prior", C.c_double),
                ("iter", C.c_longlong), ("total_edges", C.c_int), ("found", C.c_int)]


class BestLib:
    """host_emu_best.cpp behind the entry points of host_emu_state.cpp, so that EmuProblem drives it; the best
    graph of the last run is in .best (a dict), or None when `track` is off."""

    def __init__(self, lib):
        self.lib, self.best, self.track = lib, None, True
        lib.emu_best_score_state_len.restype = C.c_longlong

    def emu_score_state_len(self, P, max_par):
        return self.lib.emu_best_score_state_len(P, max_par)

    def emu_run_chain_state(self, P, max_par, *args):
        if not self.track:
            self.best = None
            return self.lib.emu_run_chain_best(P, max_par, *args, None, None, None)
        par = np.full((P, max_par), -7, np.int32)
        npar = np.full(P, -7, np.int32)
        b = EmuBestGraph()
        rc = self.lib.emu_run_chain_best(P, max_par, *args, par.ctypes.data_as(_ip), npar.ctypes.data_as(_ip),
                                         C.byref(b))
        self.best = dict(parents=par, npar=npar, log_post=b.log_post, log_lik=b.log_lik, log_prior=b.log_prior,
                         iter=int(b.iter), total_edges=int(b.total_edges), found=int(b.found))
        return rc


@pytest.fixture(scope="module")
def best_lib():
    out_dir = os.path.join(ROOT, "tests", "emu", "_build")
    so = os.path.join(out_dir, "libbn_emu_best.so")
    src = os.path.join(ROOT, "tests", "emu", "host_emu_best.cpp")
    csrc = os.path.join(ROOT, "bayesnetworks_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        os.makedirs(out_dir, exist_ok=True)
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-w",
                               "-x", "c++", f"-I{csrc}", "-o", so, src])
    return BestLib(C.CDLL(so))


# ---------------------------------------------------------------------------
# The reference
# ---------------------------------------------------------------------------
def chain_sum(scores, lanes):
    """globalLL of a score vector as the chain sums it: lane l adds nodes l, l + lanes, ... in order, then a
    butterfly over the lanes (one lane on the host build, 32 on the device)."""
    acc = [0.0] * lanes
    for c, v in enumerate(scores):
        acc[c % lanes] += float(v)
    o = lanes // 2
    while o:
        acc = [acc[i] + acc[i ^ o] for i in range(lanes)]
        o //= 2
    return acc[0]


def log_prior(phi, omega, te, ag, n_sim):
    """prior_value(phi, omega, FP + FN, TotalEdges) of chain_core.cuh, in float64."""
    dist = (te - ag) + (n_sim - ag)
    return float(np.float64(-phi) * np.float64(dist) - np.float64(omega) * np.float64(te))


def replay(par, npar, moves, it0, end, drop, t_iter, t_gll, sim, n_sim, phi, omega, start_ll=None):
    """The best graph (dict as BestLib.best) of a chain that starts at iteration it0 from (par, npar), accepts
    `moves` (iter, movetype, child, parent) and stops before iteration `end`; t_iter / t_gll: its trace
    (output = 1); sim[child, parent]: the prior graph, n_sim its list entries (NsimEdges); start_ll: the start
    graph's log_lik, if known."""
    par, npar = np.array(par, np.int32), np.array(npar, np.int32)
    P, MP = par.shape
    row = {int(i): float(g) for i, g in zip(t_iter, t_gll)}
    te = int(npar.sum())
    ag = int(sum(sim[c, par[c, e]] for c in range(P) for e in range(npar[c])))
    D = max(drop, it0)
    first = int(moves[0][0]) if len(moves) else end
    ll = start_ll
    if ll is None:  # a logged iteration before the first accepted move saw the start graph
        before = [i for i in row if it0 <= i < first]
        ll = row[before[0]] if before else None
    born = it0
    best = dict(parents=np.full((P, MP), -1, np.int32), npar=np.zeros(P, np.int32), log_post=-np.inf,
                log_lik=-np.inf, log_prior=-np.inf, iter=-1, total_edges=0, found=0)

    def visit(t):
        if t <= D:
            return
        assert ll is not None, "the start graph's log_lik is needed but unknown"
        lpr = log_prior(phi, omega, te, ag, n_sim)
        lp = ll + lpr
        if not best["found"] or lp > best["log_post"]:
            best.update(parents=par.copy(), npar=npar.copy(), log_post=lp, log_lik=ll, log_prior=lpr,
                        iter=max(born, D), total_edges=te, found=1)

    for t, typ, c, j in np.asarray(moves, np.int64).reshape(-1, 4):
        t, c, j = int(t), int(c), int(j)
        visit(t)
        if typ == 1:
            par[c, npar[c]] = j
            npar[c] += 1
            te += 1
            ag += int(sim[c, j])
        else:
            e = list(par[c, :npar[c]]).index(j)
            par[c, e:npar[c] - 1] = par[c, e + 1:npar[c]].copy()
            npar[c] -= 1
            par[c, npar[c]] = -1
            te -= 1
            ag -= int(sim[c, j])
        ll, born = row[t], t
    visit(end)
    return best


def same_best(got, want):
    """Exact equality: lists in order, npar, the bits of the three scores, iter, TotalEdges, found."""
    assert int(got["found"]) == int(want["found"])
    assert np.array_equal(got["parents"], want["parents"]) and np.array_equal(got["npar"], want["npar"])
    for k in ("log_post", "log_lik", "log_prior"):
        assert np.float64(got[k]).tobytes() == np.float64(want[k]).tobytes(), (k, got[k], want[k])
    assert int(got["iter"]) == int(want["iter"]) and int(got["total_edges"]) == int(want["total_edges"])


def empty_start(P, max_par):
    return np.full((P, max_par), -1, np.int32), np.zeros(P, np.int32)


# ---------------------------------------------------------------------------
# CPU: the host build of the chain core
# ---------------------------------------------------------------------------
def run(lib, pr, n_iter, **kw):
    out = pr.run(lib, n_iter, **kw)
    out["best"] = lib.best
    return out


def emu_replay(out, pr, start, it0, end, score_in=None):
    start_ll = None if score_in is None else chain_sum(score_in[:pr.P], 1)
    return replay(start[0], start[1], out["moves"], it0, end, pr.drop, out["iter"], out["globalLL"], pr.sim,
                  pr.n_sim, pr.phi, pr.omega, start_ll=start_ll)


def _same_outputs(a, b):
    for k in ("iter", "ChangedNode", "movetype", "additions", "deletions", "FN", "FP", "globalLL", "moves", "fpar",
              "fnpar", "freq", "nfreq", "score"):
        assert np.array_equal(a[k], b[k]), k
    for k in ("iter", "valid", "total_edges_member", "additions", "deletions", "uniforms"):
        assert getattr(a["state"], k) == getattr(b["state"], k), k
    assert list(a["state"].wh_state) == list(b["state"].wh_state) and list(a["state"].mt) == list(b["state"].mt)


@pytest.mark.parametrize("drop", [0, DROP])
@pytest.mark.parametrize("kind,seeds", [(RNG_WH, WH_SEEDS), (RNG_RMT, (1234,))])
@pytest.mark.parametrize("max_par", [8, 50])
def test_dataset_matches_replay(best_lib, emu_state_lib, dataset, max_par, kind, seeds, drop):
    """The shipped dataset (81 nodes), 20,000 iterations: the best graph equals the replay's, and every other
    output equals that of the same run without the tracking."""
    pr = EmuProblem(dataset["X"], dataset["source"], dataset["target"], dataset["node_type"], max_par, 1, kind,
                    seeds, drop=drop)
    out = run(best_lib, pr, N_SPLIT)
    assert out["best"]["found"] == 1 and out["best"]["iter"] >= drop
    same_best(out["best"], emu_replay(out, pr, empty_start(pr.P, max_par), 0, N_SPLIT))
    _same_outputs(out, pr.run(emu_state_lib, N_SPLIT))


def test_tracking_off_same_outputs(best_lib, emu_state_lib, dataset):
    """The host build with its best pointers null is the plain chain, and output = 100 (rows seldom cache the
    log_lik the tracking computes) changes nothing either."""
    pr = EmuProblem(dataset["X"], dataset["source"], dataset["target"], dataset["node_type"], 8, 100, RNG_WH,
                    WH_SEEDS, drop=DROP)
    on = run(best_lib, pr, N_SPLIT)
    best_lib.track = False
    try:
        off = run(best_lib, pr, N_SPLIT)
    finally:
        best_lib.track = True
    assert off["best"] is None and on["best"]["found"] == 1
    _same_outputs(on, off)
    _same_outputs(on, pr.run(emu_state_lib, N_SPLIT))


def test_p300_maxpar16_many_deletions(best_lib):
    """300 nodes at MaxPar 16: hundreds of accepted deletions, whose scores come from Givens downdates."""
    X, g, nt = _synthetic(300, 400, 16, 11)
    pr = EmuProblem(X, g.source, g.target, nt, 16, 1, RNG_WH, (123, 456, 789), drop=3000, omega=0.2)
    out = run(best_lib, pr, N_SPLIT)
    assert int((out["moves"][:, 1] == 2).sum()) > 200
    same_best(out["best"], emu_replay(out, pr, empty_start(pr.P, 16), 0, N_SPLIT))
    assert out["best"]["total_edges"] > 0


def _problem(dataset, drop, max_par=8, kind=RNG_WH, seeds=WH_SEEDS):
    return EmuProblem(dataset["X"], dataset["source"], dataset["target"], dataset["node_type"], max_par, 1, kind,
                      seeds, drop=drop)


def test_no_tabulated_iteration(best_lib, dataset):
    """end <= D: found = 0, lists -1 / 0, -inf scores, iter -1 -- a fresh run that ends at drop, and a
    resumed segment that ends before drop."""
    pr = _problem(dataset, DROP)
    out = run(best_lib, pr, DROP)
    b = out["best"]
    assert b["found"] == 0 and b["iter"] == -1 and b["total_edges"] == 0
    assert (b["parents"] == -1).all() and (b["npar"] == 0).all()
    assert b["log_post"] == -np.inf and b["log_lik"] == -np.inf and b["log_prior"] == -np.inf
    a = run(best_lib, pr, 1000)
    seg = run(best_lib, pr, 2000, start=(a["fpar"], a["fnpar"]), st_in=a["state"], score_in=a["score"])
    assert seg["best"]["found"] == 0 and (seg["best"]["parents"] == -1).all()
    from bayesnetworks_b200 import best_graph
    from bayesnetworks_b200.api import BestGraph
    assert best_graph([BestGraph(parents=b["parents"], npar=b["npar"], log_post=b["log_post"], log_lik=b["log_lik"],
                                 log_prior=b["log_prior"], iter=b["iter"], found=False)]) is None


def test_no_move_after_drop_gives_held_graph(best_lib, dataset):
    """No accepted move after D: the graph held at D wins with iter == D.  A fresh run whose drop lies behind
    its last accepted move gives its final graph; a resumed segment without an accepted move gives its start
    graph (its log_lik from the score block)."""
    pr = _problem(dataset, 0)
    full = run(best_lib, pr, N_SPLIT)
    last = int(full["moves"][-1, 0])
    assert last + 10 < N_SPLIT
    pr2 = _problem(dataset, last + 5)
    out = run(best_lib, pr2, N_SPLIT)
    assert out["best"]["iter"] == last + 5
    assert np.array_equal(out["best"]["parents"], out["fpar"]) and np.array_equal(out["best"]["npar"], out["fnpar"])
    same_best(out["best"], emu_replay(out, pr2, empty_start(pr2.P, 8), 0, N_SPLIT))
    # the longest gap between accepted moves: a segment inside it accepts nothing
    it = full["moves"][:, 0]
    k = int(np.argmax(np.diff(it)))
    a, b = int(it[k]) + 1, int(it[k + 1])
    assert b - a >= 3
    first = run(best_lib, pr, a)
    seg = run(best_lib, pr, b - a - 1, start=(first["fpar"], first["fnpar"]), st_in=first["state"],
              score_in=first["score"])
    assert len(seg["moves"]) == 0
    sb = seg["best"]
    assert sb["found"] == 1 and sb["iter"] == a
    assert np.array_equal(sb["parents"], first["fpar"]) and np.array_equal(sb["npar"], first["fnpar"])
    same_best(sb, emu_replay(seg, pr, (first["fpar"], first["fnpar"]), a, b - 1, score_in=first["score"]))


def test_drop_at_an_accepted_move(best_lib, dataset):
    """drop = the iteration of an accepted move: the graph it replaces is not a candidate (it was never held
    after a tabulated iteration)."""
    pr0 = _problem(dataset, 0)
    full = run(best_lib, pr0, N_SPLIT)
    t = int(full["moves"][len(full["moves"]) // 2, 0])
    pr = _problem(dataset, t)
    out = run(best_lib, pr, N_SPLIT)
    assert np.array_equal(out["moves"], full["moves"])
    want = emu_replay(out, pr, empty_start(pr.P, 8), 0, N_SPLIT)
    same_best(out["best"], want)
    assert out["best"]["iter"] >= t
    # and the replay's candidate rule is what decides: counted from t - 1 on, the replaced graph is one
    with_it = emu_replay(out, _problem(dataset, t - 1), empty_start(pr.P, 8), 0, N_SPLIT)
    assert with_it["log_post"] >= want["log_post"]


def _as_best(d):
    from bayesnetworks_b200.api import BestGraph
    return BestGraph(parents=d["parents"], npar=d["npar"], log_post=d["log_post"], log_lik=d["log_lik"],
                     log_prior=d["log_prior"], iter=d["iter"], found=bool(d["found"]))


def _segments(lib, pr, n_iter, points):
    bounds = [0] + sorted(set(int(q) for q in points if 0 < q < n_iter)) + [n_iter]
    segs, prev = [], None
    for a, b in zip(bounds[:-1], bounds[1:]):
        if prev is None:
            r = run(lib, pr, b - a)
        else:
            r = run(lib, pr, b - a, start=(prev["fpar"], prev["fnpar"]), st_in=prev["state"], score_in=prev["score"])
        assert r["state"].iter == b
        r["it0"], r["end"], r["prev"] = a, b, prev
        segs.append(r)
        prev = r
    return segs


def _check_segments(pr, full, segs):
    from bayesnetworks_b200 import best_graph
    got = best_graph([_as_best(s["best"]) for s in segs])
    fb = full["best"]
    same_best(dict(parents=got.parents, npar=got.npar, log_post=got.log_post, log_lik=got.log_lik,
                   log_prior=got.log_prior, iter=got.iter, total_edges=int(got.npar.sum()), found=int(got.found)), fb)
    for s in segs:
        p = s["prev"]
        start = empty_start(pr.P, pr.max_par) if p is None else (p["fpar"], p["fnpar"])
        same_best(s["best"], emu_replay(s, pr, start, s["it0"], s["end"], score_in=None if p is None else p["score"]))


@pytest.mark.parametrize("max_par,kind,seeds", [(8, RNG_WH, WH_SEEDS), (50, RNG_RMT, (99,))])
def test_segments_combine(best_lib, dataset, max_par, kind, seeds):
    """Splits inside the opening `TotalEdges < 3` phase, around drop, later, and one inside the interval in
    which the uninterrupted run's best graph was held: best_graph over the segments in order is the
    uninterrupted run's best, and each segment matches its own replay."""
    pr = EmuProblem(dataset["X"], dataset["source"], dataset["target"], dataset["node_type"], max_par, 1, kind,
                    seeds, drop=DROP)
    full = run(best_lib, pr, N_SPLIT)
    it = full["moves"][:, 0]
    b_it = full["best"]["iter"]
    after = it[it > b_it]
    held_to = int(after[0]) if after.size else N_SPLIT
    assert held_to - b_it >= 2
    inside = (b_it + held_to) // 2    # the best graph is a candidate on both sides of this split
    assert b_it < inside < held_to
    segs = _segments(best_lib, pr, N_SPLIT, [1, 2, DROP - 1, DROP, DROP + 1, 12345, inside])
    _check_segments(pr, full, segs)
    # the graph held across `inside` is the best of both segments that share it; the earlier one is reported
    from bayesnetworks_b200 import best_graph
    k = [s["it0"] for s in segs].index(inside)
    assert segs[k]["best"]["log_post"] == full["best"]["log_post"]
    assert best_graph([_as_best(s["best"]) for s in segs]).iter == b_it


def test_segments_combine_p300_maxpar16(best_lib):
    X, g, nt = _synthetic(300, 400, 16, 11)
    pr = EmuProblem(X, g.source, g.target, nt, 16, 1, RNG_WH, (5, 6, 7), drop=4000, omega=0.2)
    full = run(best_lib, pr, N_SPLIT)
    segs = _segments(best_lib, pr, N_SPLIT, [3999, 4000, 9000, 15000])
    _check_segments(pr, full, segs)


def test_best_graph_hand_made():
    from bayesnetworks_b200 import best_graph
    from bayesnetworks_b200.api import BestGraph
    par = np.array([[-1], [0], [-1]], np.int32)
    npar = np.array([0, 1, 0], np.int32)
    mk = lambda lp, it, found=True: BestGraph(parents=par, npar=npar, log_post=lp, log_lik=lp + 1, log_prior=-1.0,  # noqa: E731
                                               iter=it, found=found)
    a, b, c, d = mk(-5.0, 10), mk(-3.0, 20), mk(-3.0, 30), mk(0.0, -1, found=False)
    assert best_graph([a, b, c, d]) is b          # first of the maximum; found = False skipped
    assert best_graph([d]) is None
    assert b.edges() == [(0, 1)]
    st = b.as_start()
    assert np.array_equal(st.parents, par) and np.array_equal(st.npar, npar) and not st.resumed
    with pytest.raises(ValueError):
        best_graph([np.zeros(3)])


def test_ctypes_mirror_matches_header(tmp_path):
    """_lib.RunArgs / BestGraphC have the layout of bn_run_args / bn_best_graph in include/bn_b200.h."""
    from bayesnetworks_b200 import _lib
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "bn_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu %zu %zu %zu\\n", sizeof(bn_run_args), '
                   'offsetof(bn_run_args, best_parents), offsetof(bn_run_args, best_n_par), offsetof(bn_run_args, best), '
                   'sizeof(bn_best_graph), offsetof(bn_best_graph, iter), offsetof(bn_best_graph, found)); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.check_call(["gcc", "-std=c99", f"-I{os.path.join(ROOT, 'include')}", "-o", str(exe), str(src)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    R, B = _lib.RunArgs, _lib.BestGraphC
    assert got == [C.sizeof(R), R.best_parents.offset, R.best_n_par.offset, R.best.offset, C.sizeof(B),
                   B.iter.offset, B.found.offset]


# ---------------------------------------------------------------------------
# GPU: the CUDA chains through the C ABI
# ---------------------------------------------------------------------------
def _sim(source, target, P):
    """sim[child, parent] of a 1-based prior edge list, and its NsimEdges (list entries)."""
    sim = np.zeros((P, P), np.uint8)
    for s_, t_ in zip(source, target):
        sim[t_ - 1, s_ - 1] = 1
    return sim, len(source)


def _bd(b):
    return dict(parents=b.parents, npar=b.npar, log_post=b.log_post, log_lik=b.log_lik, log_prior=b.log_prior,
                iter=b.iter, total_edges=int(b.npar.sum()) if b.found else 0, found=int(b.found))


def _gpu_pair(ctx, **kw):
    """The same run with and without the tracking: every other output must be the same."""
    on = ctx.run(log_moves=True, tabulate=True, track_best=True, **kw)[0]
    off = ctx.run(log_moves=True, tabulate=True, **kw)[0]
    for a, b in zip(on, off):
        for k in a.trace:
            assert np.array_equal(a.trace[k], b.trace[k]), k
        for k in ("accepted_moves", "edge_freq", "npar_freq", "final_parents", "final_npar", "mt_state", "anc_freq"):
            x, y = getattr(a, k), getattr(b, k)
            assert (x is None and y is None) or np.array_equal(x, y), k
        for k in ("uniforms", "valid_iters", "proposed", "reject", "n_nonpd", "total_edges"):
            assert getattr(a, k) == getattr(b, k), k
        assert b.best is None and a.best is not None
    return on


def _gpu_check(res, sim, n_iter, drop, max_par, phi, omega):
    sim, n_sim = sim
    for r in res:
        par, npar = empty_start(len(r.final_npar), max_par)
        want = replay(par, npar, r.accepted_moves, 0, n_iter, drop, r.trace["iter"], r.trace["globalLL"], sim,
                      n_sim, phi, omega)
        same_best(_bd(r.best), want)


@pytest.mark.gpu
@pytest.mark.parametrize("P", [896, 1000, 1025])
def test_gpu_dense_shapes_match_replay(P):
    """The dense fixtures' inputs (MaxPar 8), eight chains in one launch, drop mid-run."""
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_dense_parity import CASES, MAX_PAR, dense_inputs
    from bayesnetworks_b200 import Context
    X, g, nt = dense_inputs(P)
    _, _, phi, omega, _ = CASES[f"p{P}_mid"]
    seeds = np.array([(100 + 7 * c, 200 + 11 * c, 300 + 13 * c) for c in range(8)], np.int32)
    with Context.from_data(X, g.source, g.target, nt, max_par=MAX_PAR, phi=phi, omega=omega) as ctx:
        res = _gpu_pair(ctx, n_chains=8, n_iter=N_SPLIT, output=1, rng="wh", seeds=seeds, drop=7000)
    assert min(int((r.accepted_moves[:, 1] == 2).sum()) for r in res) > 1000
    _gpu_check(res, _sim(g.source, g.target, P), N_SPLIT, 7000, MAX_PAR, phi, omega)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["config3_maxpar50", "large_p_global_memory"])
def test_gpu_other_shapes_match_replay(shape):
    """Config 3 (100 nodes x 10,000 samples) at MaxPar 50; the 2,500-node shape whose state partly lives in
    global memory."""
    from bayesnetworks_b200 import Context
    if shape == "config3_maxpar50":
        X, g, nt = _synthetic(100, 10000, 50, 42)
        mp, nc = 50, 4
    else:
        X, g, nt = _synthetic(2500, 120, 4, 9)
        mp, nc = 4, 2
    with Context.from_data(X, g.source, g.target, nt, max_par=mp, omega=0.3) as ctx:
        res = _gpu_pair(ctx, n_chains=nc, n_iter=N_SPLIT, output=1, rng="wh", drop=1000)
    assert min(len(r.accepted_moves) for r in res) > 100
    _gpu_check(res, _sim(g.source, g.target, X.shape[1]), N_SPLIT, 1000, mp, 1.0, 0.3)


@pytest.mark.gpu
def test_gpu_flag_with_ancestor_tabulation():
    """track_best next to tabulate_ancestors: anc_freq and every other output as without the tracking."""
    from bayesnetworks_b200 import Context
    z = np.load(os.path.join(ROOT, "tests", "golden", "network_p3sim8.npz"))
    with Context.from_data(z["X"], z["source"], z["target"], z["node_type"], max_par=8) as ctx:
        res = _gpu_pair(ctx, n_chains=4, n_iter=N_SPLIT, output=1, rng="wh", drop=DROP, tabulate_ancestors=True)
    for r in res:
        assert r.anc_freq is not None
    _gpu_check(res, _sim(z["source"], z["target"], z["X"].shape[1]), N_SPLIT, DROP, 8, 1.0, 6.9)


@pytest.mark.gpu
def test_gpu_segments_combine_and_rescore():
    """Eight chains on the shipped dataset resumed at 1, DROP, 12,345 (state + score block): best_graph over the
    segments is the uninterrupted run's best, bit for bit.  Rescoring that graph with score_nodes and a numpy
    prior agrees with log_lik / log_prior to 1e-9, and it seeds new chains."""
    from bayesnetworks_b200 import Context, best_graph
    z = np.load(os.path.join(ROOT, "tests", "golden", "network_p3sim8.npz"))
    P = z["X"].shape[1]
    sim, n_sim = _sim(z["source"], z["target"], P)
    seeds = np.array([(1000 + 7 * c, 2000 + 11 * c, 3000 + 13 * c) for c in range(8)], np.int32)
    kw = dict(n_chains=8, output=1, rng="wh", drop=DROP, log_moves=True, track_best=True, want_state=True)
    with Context.from_data(z["X"], z["source"], z["target"], z["node_type"], max_par=8) as ctx:
        full = ctx.run(n_iter=N_SPLIT, seeds=seeds, **kw)[0]
        parts, start, done = [], None, 0
        for b in (1, DROP, 12345, N_SPLIT):
            r = ctx.run(n_iter=b - done, seeds=seeds if start is None else None, start=start, **kw)[0]
            parts.append(r)
            start, done = [x.state for x in r], b
        for c in range(8):
            got = best_graph([p[c] for p in parts])
            same_best(_bd(got), _bd(full[c].best))
        bg = best_graph(full)
        assert bg is not None and all(bg.log_post >= r.best.log_post for r in full)
        sc = ctx.score_nodes(np.arange(P), bg.parents, bg.npar)
        te = int(bg.npar.sum())
        ag = int(sum(sim[c, bg.parents[c, e]] for c in range(P) for e in range(bg.npar[c])))
        np.testing.assert_allclose(sc.sum(), bg.log_lik, rtol=1e-9, atol=0)
        np.testing.assert_allclose(-1.0 * ((te - ag) + (n_sim - ag)) - 6.9 * te, bg.log_prior,
                                   rtol=1e-9, atol=0)
        seeded = ctx.run(n_chains=1, n_iter=100, output=10, start=[bg.as_start()], track_best=True)[0][0]
        assert seeded.best.found
    _gpu_check(full, (sim, n_sim), N_SPLIT, DROP, 8, 1.0, 6.9)


@pytest.mark.gpu
def test_gpu_partial_pointers_refused():
    from bayesnetworks_b200 import BnError, Context, _lib
    z = np.load(os.path.join(ROOT, "tests", "golden", "network_p3sim8.npz"))
    P = z["X"].shape[1]
    with Context.from_data(z["X"], z["source"], z["target"], z["node_type"], max_par=4) as ctx:
        L = _lib.lib()
        cap = 10
        cols = [np.zeros(cap, np.int32) for _ in range(7)]
        gll = np.zeros(cap)
        n_rows = np.zeros(1, np.int32)
        tr = _lib.Trace(cap, n_rows.ctypes.data_as(_ip), *[cols[k].ctypes.data_as(_ip) for k in range(3)],
                        gll.ctypes.data_as(_lib._dp), *[cols[k].ctypes.data_as(_ip) for k in range(3, 7)])
        bpar = np.zeros((P, 4), np.int32)
        bnpar = np.zeros(P, np.int32)
        bst = _lib.BestGraphC()
        for missing in ("best_parents", "best_n_par", "best"):
            a = _lib.RunArgs()
            a.n_chains, a.rng_kind, a.initial_network, a.n_iter, a.output_every = 1, 0, 2, 100, 10
            if missing != "best_parents":
                a.best_parents = bpar.ctypes.data_as(_ip)
            if missing != "best_n_par":
                a.best_n_par = bnpar.ctypes.data_as(_ip)
            if missing != "best":
                a.best = C.cast(C.pointer(bst), C.c_void_p)
            with pytest.raises(BnError) as e:
                _lib.check(L.bn_run(ctx._h, C.byref(a), C.byref(tr), None, None, None, None))
            assert e.value.status == _lib.BN_ERR_BAD_ARG and f"{missing} is NULL" in str(e.value)
