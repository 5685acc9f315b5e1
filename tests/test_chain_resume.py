"""Resumable chains: a run of N iterations split into segments, each started from the state the previous
segment returned (graph, bn_chain_state scalars, stream state, score block), computes the same bits as one
run of N iterations -- trace columns, move log, summed tabulations, final graph, stream state.

CPU tests run the host build of the chain core (tests/emu/host_emu_state.cpp); GPU tests go through the
C ABI (Context.run(start=..., want_state=True))."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, centered_stats, prior_lists

INT_COLS = ("iter", "ChangedNode", "movetype", "additions", "deletions", "FN", "FP")
COLS = INT_COLS + ("globalLL",)
RNG_WH, RNG_RMT, RNG_REPLAY = 0, 1, 2
WH_SEEDS = (10437, 13568, 30524)
INT_MAX = 2**31 - 1


class EmuChainState(C.Structure):
    _fields_ = [("iter", C.c_longlong), ("valid", C.c_int), ("total_edges_member", C.c_int),
                ("additions", C.c_int), ("deletions", C.c_int), ("wh_state", C.c_int * 3),
                ("uniforms", C.c_longlong), ("mt", C.c_int * 625)]


@pytest.fixture(scope="module")
def emu_state_lib():
    """Host (one-lane) build of the chain core with the supplied-start entry point, tests only."""
    out_dir = os.path.join(ROOT, "tests", "emu", "_build")
    so = os.path.join(out_dir, "libbn_emu_state.so")
    src = os.path.join(ROOT, "tests", "emu", "host_emu_state.cpp")
    csrc = os.path.join(ROOT, "bayesnetworks_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        os.makedirs(out_dir, exist_ok=True)
        subprocess.check_call(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", "-w",
                               "-x", "c++", f"-I{csrc}", "-o", so, src])
    lib = C.CDLL(so)
    lib.emu_score_state_len.restype = C.c_longlong
    return lib


def _rmt_seed_state(seed):
    """R's set.seed() scrambling (MT words; the position is 624)."""
    s = np.uint32(seed)
    out = np.zeros(625, np.uint32)
    with np.errstate(over="ignore"):
        for _ in range(50):
            s = np.uint32(69069) * s + np.uint32(1)
        for j in range(625):
            s = np.uint32(69069) * s + np.uint32(1)
            out[j] = s
    return out[1:].copy()


class EmuProblem:
    """One dataset + chain settings for the host build."""

    def __init__(self, X, src, tgt, nt, max_par, output, kind, seeds, drop=0, phi=1.0, omega=6.9, init=2,
                 replay=None):
        self.N, self.P = X.shape
        _, self.Cm = centered_stats(X)
        self.ppar, self.pnpar = prior_lists(src, tgt, self.P, max_par)
        self.sim = np.zeros((self.P, self.P), np.uint8)
        for s_, t_ in zip(src, tgt):
            self.sim[t_ - 1, s_ - 1] = 1
        self.n_sim = len(src)
        self.nt = np.asarray(nt).astype(np.uint8)
        self.max_par, self.output, self.kind, self.drop = max_par, output, kind, drop
        self.phi, self.omega, self.init = phi, omega, init
        self.sd = np.zeros(3, np.int32)
        self.sd[:len(seeds)] = seeds
        self.mt = _rmt_seed_state(seeds[0]) if kind == RNG_RMT else np.zeros(624, np.uint32)
        self.replay = None if replay is None else np.ascontiguousarray(replay, dtype=np.float64)

    def run(self, lib, n_iter, start=None, st_in=None, score_in=None, replay_from=0):
        P, mp = self.P, self.max_par
        cap = (n_iter + self.output - 1) // self.output + 1
        ti = [np.zeros(cap, np.int32) for _ in range(7)]
        gll = np.zeros(cap)
        moves = np.zeros((max(n_iter, 1), 4), np.int32)
        freq = np.zeros((P, P), np.int32)
        nfreq = np.zeros((P, mp + 1), np.int32)
        fpar = np.zeros((P, mp), np.int32)
        fnpar = np.zeros(P, np.int32)
        cnt = np.zeros(12, np.int64)
        st_out = EmuChainState()
        slen = int(lib.emu_score_state_len(P, mp))
        score_out = np.zeros(slen)
        dp, ip, up = C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_ubyte)
        rp = None if self.replay is None else self.replay[replay_from:]
        spar = snpar = None
        if start is not None:
            spar, snpar = np.ascontiguousarray(start[0], np.int32), np.ascontiguousarray(start[1], np.int32)
        rc = lib.emu_run_chain_state(
            P, mp, self.N, self.Cm.ctypes.data_as(dp), self.nt.ctypes.data_as(up), self.sim.ctypes.data_as(up),
            self.n_sim, C.c_double(self.phi), C.c_double(self.omega), self.init, self.drop, n_iter, self.output,
            self.ppar.ctypes.data_as(ip), self.pnpar.ctypes.data_as(ip), self.kind, self.sd.ctypes.data_as(ip),
            self.mt.ctypes.data_as(C.POINTER(C.c_uint)), None if rp is None else rp.ctypes.data_as(dp),
            C.c_long(0 if rp is None else len(rp)), cap,
            *[ti[k].ctypes.data_as(ip) for k in range(3)], gll.ctypes.data_as(dp),
            *[ti[k].ctypes.data_as(ip) for k in range(3, 7)], moves.shape[0], moves.ctypes.data_as(ip),
            freq.ctypes.data_as(ip), nfreq.ctypes.data_as(ip), fpar.ctypes.data_as(ip), fnpar.ctypes.data_as(ip),
            cnt.ctypes.data_as(C.POINTER(C.c_long)),
            None if spar is None else spar.ctypes.data_as(ip), None if snpar is None else snpar.ctypes.data_as(ip),
            None if st_in is None else C.byref(st_in), C.byref(st_out),
            None if score_in is None else score_in.ctypes.data_as(dp), score_out.ctypes.data_as(dp))
        assert rc == 0
        n = int(cnt[8])
        out = dict(zip(INT_COLS, [ti[0][:n], ti[1][:n], ti[2][:n], ti[3][:n], ti[4][:n], ti[5][:n], ti[6][:n]]))
        out.update(globalLL=gll[:n], moves=moves[:int(cnt[9])], fpar=fpar, fnpar=fnpar, freq=freq, nfreq=nfreq,
                   state=st_out, score=score_out)
        return out

    def split(self, lib, n_iter, points, with_scores=True):
        """Segments [0, p1), [p1, p2), ... [pk, n_iter), each from the state the previous one returned."""
        bounds = [0] + sorted(set(int(q) for q in points if 0 < q < n_iter)) + [n_iter]
        segs, prev = [], None
        for a, b in zip(bounds[:-1], bounds[1:]):
            if prev is None:
                r = self.run(lib, b - a)
            else:
                r = self.run(lib, b - a, start=(prev["fpar"], prev["fnpar"]), st_in=prev["state"],
                             score_in=prev["score"] if with_scores else None, replay_from=prev["state"].uniforms)
            assert r["state"].iter == b
            segs.append(r)
            prev = r
        return segs


def _joined(segs):
    out = {k: np.concatenate([s[k] for s in segs]) for k in COLS}
    out["moves"] = np.concatenate([s["moves"] for s in segs])
    out["freq"] = sum(s["freq"].astype(np.int64) for s in segs)
    out["nfreq"] = sum(s["nfreq"].astype(np.int64) for s in segs)
    return out


def _same_state(a, b):
    for k in ("iter", "valid", "total_edges_member", "additions", "deletions", "uniforms"):
        assert getattr(a, k) == getattr(b, k), k
    assert list(a.wh_state) == list(b.wh_state)
    assert list(a.mt) == list(b.mt)


def _assert_split_equals_full(full, segs, gll_exact=True):
    j = _joined(segs)
    for k in INT_COLS:
        assert np.array_equal(j[k], full[k]), k
    if gll_exact:
        assert np.array_equal(j["globalLL"], full["globalLL"])
    else:
        np.testing.assert_allclose(j["globalLL"], full["globalLL"], rtol=1e-9, atol=0)
    assert np.array_equal(j["moves"], full["moves"])
    assert np.array_equal(j["freq"], full["freq"])
    assert np.array_equal(j["nfreq"], full["nfreq"])
    assert np.array_equal(segs[-1]["fpar"], full["fpar"]) and np.array_equal(segs[-1]["fnpar"], full["fnpar"])
    _same_state(segs[-1]["state"], full["state"])


N_SPLIT = 20000
DROP = 5000


# ---------------------------------------------------------------------------
# CPU: the host build of the chain core
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("output", [1, 100])
@pytest.mark.parametrize("kind,seeds", [(RNG_WH, WH_SEEDS), (RNG_RMT, (1234,))])
@pytest.mark.parametrize("max_par", [8, 50])
def test_split_run_equals_full_run(emu_state_lib, dataset, max_par, kind, seeds, output):
    """The shipped dataset, 20,000 iterations: split inside the opening `TotalEdges < 3` phase (1, 2, 5),
    at a non-multiple of `output`, around `drop`, right after an accepted deletion; and in ten equal
    segments."""
    pr = EmuProblem(dataset["X"], dataset["source"], dataset["target"], dataset["node_type"], max_par, output,
                    kind, seeds, drop=DROP)
    full = pr.run(emu_state_lib, N_SPLIT)
    dels = full["moves"][(full["moves"][:, 1] == 2) & (full["moves"][:, 0] > 100), 0]
    assert dels.size > 0
    points = [1, 2, 5, 7777, DROP - 1, DROP + 1, int(dels[0]) + 1]
    _assert_split_equals_full(full, pr.split(emu_state_lib, N_SPLIT, points))
    _assert_split_equals_full(full, pr.split(emu_state_lib, N_SPLIT, range(2000, N_SPLIT, 2000)))


def _dense16():
    from bayesnetworks_b200.synth import make_dag, make_prior, simulate_numpy
    dag = make_dag(40, seed=5)
    g = make_prior(dag, max_par=16, seed=6)
    return simulate_numpy(dag, 500, seed=7), g


def test_factor_path_many_deletions(emu_state_lib):
    """MaxPar 16 (per-node Cholesky factors, Givens downdates on accepted deletions), five segments: bit
    for bit with the score block; without it the factors are refactorised, so the integer columns stay
    and globalLL agrees to rounding."""
    X, g = _dense16()
    pr = EmuProblem(X, g.source, g.target, g.node_type_codes(), 16, 7, RNG_WH, (123, 456, 789), omega=0.2)
    full = pr.run(emu_state_lib, N_SPLIT)
    assert int((full["moves"][:, 1] == 2).sum()) > 200
    points = range(4000, N_SPLIT, 4000)
    _assert_split_equals_full(full, pr.split(emu_state_lib, N_SPLIT, points))
    _assert_split_equals_full(full, pr.split(emu_state_lib, N_SPLIT, points, with_scores=False), gll_exact=False)


@pytest.mark.parametrize("max_par", [8, 50])
def test_start_from_prior_graph_equals_initial_network_0(emu_state_lib, dataset, max_par):
    """A fresh chain from the prior's lists is the InitialNetwork = 0 chain with the same seeds."""
    args = (dataset["X"], dataset["source"], dataset["target"], dataset["node_type"], max_par, 10, RNG_WH, WH_SEEDS)
    a = EmuProblem(*args, init=0).run(emu_state_lib, 5000)
    pr = EmuProblem(*args, init=2)
    b = pr.run(emu_state_lib, 5000, start=(pr.ppar, pr.pnpar))
    for k in COLS + ("moves", "fpar", "fnpar"):
        assert np.array_equal(a[k], b[k]), k
    _same_state(a["state"], b["state"])


def test_replayed_stream_split(emu_state_lib, dataset):
    """A replayed stream: each segment gets the rest of the buffer from the uniforms already consumed."""
    u = np.random.default_rng(3).random(200000)
    pr = EmuProblem(dataset["X"], dataset["source"], dataset["target"], dataset["node_type"], 8, 10, RNG_REPLAY,
                    (1,), replay=u)
    full = pr.run(emu_state_lib, 10000)
    _assert_split_equals_full(full, pr.split(emu_state_lib, 10000, [3, 2500, 6001]))


def test_chain_state_checkpoint_roundtrip(tmp_path):
    from bayesnetworks_b200 import ChainState
    rng = np.random.default_rng(1)
    st = ChainState.from_edges([(3, 0), (1, 0), (2, 4)], n_nodes=6, max_par=4)
    assert st.parents[0, :2].tolist() == [3, 1] and st.npar.tolist() == [2, 0, 0, 0, 1, 0] and not st.resumed
    full = ChainState(parents=st.parents, npar=st.npar, n_samples=500, rng=RNG_RMT, iter=12345, valid=0,
                      total_edges_member=17, additions=40, deletions=33, uniforms=987654321012,
                      mt_state=rng.integers(-2**31, 2**31, 625).astype(np.int32), score_block=rng.random(50))
    for s in (st, full):
        path = str(tmp_path / "ckpt.npz")
        s.save(path)
        t = ChainState.load(path)
        for k in ("parents", "npar", "wh_state", "mt_state", "score_block"):
            a, b = getattr(s, k), getattr(t, k)
            assert (a is None and b is None) or np.array_equal(a, b), k
        for k in ("n_samples", "rng", "iter", "valid", "total_edges_member", "additions", "deletions", "uniforms"):
            assert getattr(s, k) == getattr(t, k), k


# ---------------------------------------------------------------------------
# GPU: the CUDA chains through the C ABI
# ---------------------------------------------------------------------------
def _ctx_run(ctx, **kw):
    return ctx.run(log_moves=True, tabulate=True, want_state=True, **kw)[0]


def _gpu_join(parts):
    out = {k: np.concatenate([p.trace[k] for p in parts]) for k in COLS}
    out["moves"] = np.concatenate([p.accepted_moves for p in parts])
    out["freq"] = sum(p.edge_freq.astype(np.int64) for p in parts)
    out["nfreq"] = sum(p.npar_freq.astype(np.int64) for p in parts)
    return out


def _gpu_same(full, parts, gll_exact=True):
    j = _gpu_join(parts)
    for k in INT_COLS:
        assert np.array_equal(j[k], full.trace[k]), k
    if gll_exact:
        assert np.array_equal(j["globalLL"], full.trace["globalLL"])
    else:
        np.testing.assert_allclose(j["globalLL"], full.trace["globalLL"], rtol=1e-9, atol=0)
    assert np.array_equal(j["moves"], full.accepted_moves)
    assert np.array_equal(j["freq"], full.edge_freq) and np.array_equal(j["nfreq"], full.npar_freq)
    a, b = parts[-1].state, full.state
    assert np.array_equal(a.parents, b.parents) and np.array_equal(a.npar, b.npar)
    for k in ("iter", "valid", "total_edges_member", "additions", "deletions", "uniforms"):
        assert getattr(a, k) == getattr(b, k), k
    for k in ("wh_state", "mt_state"):
        assert (getattr(a, k) is None) == (getattr(b, k) is None)
        if getattr(a, k) is not None:
            assert np.array_equal(getattr(a, k), getattr(b, k)), k


def _seg_runs(ctx, rng, seeds, n_iter, output, splits, drop):
    """Chain c: [0, s_c) alone, then all chains in ONE launch from their different iterations for
    n_iter - max(s) iterations, then each alone up to n_iter."""
    nc, hi = len(splits), max(splits)
    first = [_ctx_run(ctx, n_chains=1, n_iter=s, output=output, rng=rng, seeds=seeds[c:c + 1], drop=drop)[0]
             for c, s in enumerate(splits)]
    mid = _ctx_run(ctx, n_chains=nc, n_iter=n_iter - hi, output=output, rng=rng, drop=drop,
                   start=[r.state for r in first])
    last = []
    for c, s in enumerate(splits):
        rest = hi - s
        last.append(None if rest == 0 else
                    _ctx_run(ctx, n_chains=1, n_iter=rest, output=output, rng=rng, drop=drop, start=[mid[c].state])[0])
    return [[first[c], mid[c]] + ([last[c]] if last[c] is not None else []) for c in range(nc)]


SPLITS8 = [1, 2, 5, 777, DROP - 1, DROP + 1, 7777, 3001]


def _seeds(rng, nc):
    if rng == "wh":
        return np.array([(1000 + 7 * c, 2000 + 11 * c, 3000 + 13 * c) for c in range(nc)], np.int32)
    return np.array([[4321 + c] for c in range(nc)], np.int32)


def resume_matrix_case(max_par, rng, output):
    from bayesnetworks_b200 import Context
    z = np.load(os.path.join(ROOT, "tests", "golden", "network_p3sim8.npz"))
    seeds = _seeds(rng, len(SPLITS8))
    with Context.from_data(z["X"], z["source"], z["target"], z["node_type"], max_par=max_par) as ctx:
        full = _ctx_run(ctx, n_chains=len(SPLITS8), n_iter=N_SPLIT, output=output, rng=rng, seeds=seeds, drop=DROP)
        segs = _seg_runs(ctx, rng, seeds, N_SPLIT, output, SPLITS8, DROP)
    for c in range(len(SPLITS8)):
        _gpu_same(full[c], segs[c])


@pytest.mark.gpu
@pytest.mark.parametrize("output", [1, 100])
@pytest.mark.parametrize("rng", ["wh", "rmt"])
@pytest.mark.parametrize("max_par", [8, 50])
def test_gpu_eight_chains_resumed_at_different_iterations(max_par, rng, output):
    resume_matrix_case(max_par, rng, output)


def _synthetic(P, N, max_par, seed):
    from bayesnetworks_b200.synth import make_dag, make_prior, simulate_numpy
    dag = make_dag(P, seed=seed)
    g = make_prior(dag, max_par=max_par, seed=seed + 1)
    return simulate_numpy(dag, N, seed=seed + 2), g, g.node_type_codes()


def _even_segments(ctx, n_iter, k, **kw):
    parts, start = [], None
    for i in range(k):
        n = n_iter // k + (n_iter % k if i == k - 1 else 0)
        r = _ctx_run(ctx, n_iter=n, start=start, **kw)
        parts.append(r)
        start = [x.state for x in r]
    return parts


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["config3_maxpar50", "large_p_global_memory"])
def test_gpu_segments_other_shapes(shape):
    """Config 3 (100 nodes x 10,000 samples) at MaxPar 50: factor cache and the cooperative scorer, four
    segments; the 2,500-node shape whose state partly lives in global memory, three segments."""
    from bayesnetworks_b200 import Context
    if shape == "config3_maxpar50":
        X, g, nt = _synthetic(100, 10000, 50, 42)
        mp, n_iter, k, kw = 50, 8000, 4, dict(output=10, omega=0.3)
    else:
        X, g, nt = _synthetic(2500, 120, 4, 9)
        mp, n_iter, k, kw = 4, 3000, 3, dict(output=50)
    omega = kw.pop("omega", 6.9)
    with Context.from_data(X, g.source, g.target, nt, max_par=mp, omega=omega) as ctx:
        full = _ctx_run(ctx, n_iter=n_iter, rng="wh", **kw)[0]
        parts = _even_segments(ctx, n_iter, k, rng="wh", **kw)
    _gpu_same(full, [p[0] for p in parts])


@pytest.mark.gpu
def test_gpu_reference_parity_through_resumes():
    """The p1000 chains of tests/golden/dense_ref.npz (the compiled reference's trajectories), eight chains per
    launch, as four resumed segments."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from test_dense_parity import CASES, CHAINS, N_ITER, OUTPUT, MAX_PAR, check_against_fixture, inputs_for
    from bayesnetworks_b200 import Context
    dense = np.load(os.path.join(ROOT, "tests", "golden", "dense_ref.npz"))
    X, g, nt = inputs_for(1000, dense)
    seeds = np.array([CASES[n][4] for n in CHAINS], dtype=np.int32)
    with Context.from_data(X, g.source, g.target, nt, max_par=MAX_PAR, phi=0.0, omega=0.0) as ctx:
        parts = _even_segments(ctx, N_ITER, 4, n_chains=8, output=OUTPUT, rng="wh", seeds=seeds)
    for c, name in enumerate(CHAINS):
        j = _gpu_join([p[c] for p in parts])
        st = parts[-1][c].state
        edges = [(int(st.parents[q, e]), q) for q in range(st.P) for e in range(int(st.npar[q]))]
        check_against_fixture(dense, name, j, st.uniforms, j["moves"], edges,
                              sum(p[c].n_nonpd for p in parts), gll_exact=False)


@pytest.mark.gpu
def test_gpu_replay_resume():
    """A replayed stream: the resumed segment gets the rest of the buffer."""
    from bayesnetworks_b200 import Context
    z = np.load(os.path.join(ROOT, "tests", "golden", "network_p3sim8.npz"))
    u = np.random.default_rng(5).random((3, 150000))
    with Context.from_data(z["X"], z["source"], z["target"], z["node_type"], max_par=8) as ctx:
        full = _ctx_run(ctx, n_chains=3, n_iter=10000, output=10, rng="replay", replay=u)
        a = _ctx_run(ctx, n_chains=3, n_iter=4000, output=10, rng="replay", replay=u)
        used = [r.state.uniforms for r in a]
        rest = np.full((3, u.shape[1] - min(used)), 0.5)
        for c in range(3):
            rest[c, :u.shape[1] - used[c]] = u[c, used[c]:]
        b = _ctx_run(ctx, n_chains=3, n_iter=6000, output=10, rng="replay", replay=rest, start=[r.state for r in a])
    for c in range(3):
        _gpu_same(full[c], [a[c], b[c]])


@pytest.mark.gpu
def test_gpu_bad_start_states_are_refused():
    from bayesnetworks_b200 import BnError, ChainState, Context
    from bayesnetworks_b200._lib import BN_ERR_BAD_ARG
    z = np.load(os.path.join(ROOT, "tests", "golden", "network_p3sim8.npz"))
    P = z["X"].shape[1]
    with Context.from_data(z["X"], z["source"], z["target"], z["node_type"], max_par=4) as ctx:
        good = _ctx_run(ctx, n_iter=500, output=10)[0].state
        cases = {
            "cyclic": ChainState.from_edges([(0, 1), (1, 2), (2, 0)], P, 4),
            "duplicate": ChainState.from_edges([(0, 1), (0, 1)], P, 4),
        }
        over = ChainState.from_edges([], P, 4)
        over.npar[3] = 5
        cases["npar > max_par"] = over
        late = ChainState(**{**good.__dict__, "iter": INT_MAX - 100})
        cases["iter overflow"] = late
        cases["other max_par"] = ChainState.from_edges([(0, 1)], P, 5)
        cases["other stream kind"] = good  # resumed WH state, run with rng="rmt"
        for name, st in cases.items():
            rng = "rmt" if name == "other stream kind" else "wh"
            with pytest.raises(BnError) as e:
                ctx.run(n_iter=500, output=10, rng=rng, seeds=[7], start=[st])
            assert e.value.status == BN_ERR_BAD_ARG, name


@pytest.mark.gpu
def test_gpu_two_cta_opt_in_with_start_states():
    """BN_B200_PIPE=1 with start states: bn_run takes the one-CTA kernel for them, and the uninterrupted
    runs (on the two-CTA form) still equal the segments.  In a child process with a time limit."""
    env = dict(os.environ, BN_B200_PIPE="1")
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r); import test_chain_resume as t; "
            "t.resume_matrix_case(8, 'wh', 1); print('OK')") % (ROOT, os.path.join(ROOT, "tests"))
    try:
        res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, env=env)
    except subprocess.TimeoutExpired:
        pytest.xfail("the opt-in two-CTA kernel did not finish in 300 s")
    last = res.stdout.strip().splitlines()[-1] if res.stdout.strip() else ""
    assert res.returncode == 0 and last == "OK", (last, res.stderr[-2000:])
