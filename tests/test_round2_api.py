"""Behaviour added in round 2 (VERDICT r1 / ADVICE r1): iterations of unbounded length, supplied
graphs denser than MaxPar, a defined InitialNetwork = 1, R's stream state in and out, degenerate
(collinear) data.  CPU tests pin the oracle and the host build of the chain core; `gpu` tests go
through the C ABI."""
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
INT_COLS = ("iter", "ChangedNode", "movetype", "additions", "deletions", "FN", "FP")


def _same_trace(r, ref, n_samples):
    for k in INT_COLS:
        assert np.array_equal(r.trace[k], getattr(ref, k)), k
    assert np.allclose(r.trace["globalLL"], ref.globalLL, rtol=1e-9, atol=1e-9 * n_samples / 2)
    assert r.uniforms == ref.uniforms
    assert np.array_equal(r.accepted_moves, ref.accepted_moves())
    assert r.edges() == ref.edges()


def _emu_same(r, ref):
    assert r["rc"] == 0
    for k in INT_COLS:
        assert np.array_equal(r[k], getattr(ref, k)), k
    assert int(r["cnt"][0]) == ref.uniforms
    assert np.array_equal(r["moves"], ref.accepted_moves())


def rare_children_case():
    """1,000 nodes of which 997 are sources: 0.3 % of the child draws of an addition are legal, so
    about one addition in twenty needs more uniforms than the 1,024-entry ring of the CUDA chain
    holds (0.997^1020 = 4.7 %) -- a valid reference run (src/network.h:283-289 just keeps drawing)."""
    rng = np.random.default_rng(23)
    P, N = 1000, 200
    X = np.asfortranarray(rng.standard_normal((N, P)))
    for c, ps in ((997, (0, 1)), (998, (2, 997)), (999, (998, 3, 4))):
        for q in ps:
            X[:, c] += 0.7 * X[:, q]
    nt = np.ones(P, dtype=np.int32)
    nt[997:] = 0
    src = np.array([1, 2, 3, 998], dtype=np.int32)
    tgt = np.array([998, 998, 999, 999], dtype=np.int32)
    return X, src, tgt, nt


def synthetic(P, N, max_par, seed):
    from bayesnetworks_b200.synth import make_dag, make_prior, simulate_numpy
    dag = make_dag(P, seed=seed)
    g = make_prior(dag, max_par=max_par, seed=seed + 1)
    return simulate_numpy(dag, N, seed=seed + 2), g, g.node_type_codes()


# ---------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------
def test_oracle_supplied_graph_denser_than_maxpar_matches_reference(oracle, dataset):
    """InitialNetwork = 2: the supplied graph only feeds simEdge / NsimEdges (src/network.h:138-146,
    164-169), so a node with 8 prior parents and MaxPar = 3 is a legal reference run.  The stored trace
    is tests/golden/denser_maxpar3.npz (tests/golden/make_golden_denser.py; its `source` says what made
    it); where oracle/_ref is built the compiled reference is run as well."""
    from oracle.oracle import RNG_WH, Ref, have_ref
    X, src, tgt, nt = dataset["X"], dataset["source"], dataset["target"], dataset["node_type"]
    o = oracle.mcmc(X, src, tgt, nt, max_par=3, n_iter=3000, output=10, rng_kind=RNG_WH)
    assert o.FN.max() <= 44 and o.additions[-1] > 5
    want = np.load(os.path.join(GOLDEN, "denser_maxpar3.npz"))
    for k in INT_COLS + ("globalLL",):
        assert np.array_equal(getattr(o, k), want[k]), k
    if have_ref():
        r = Ref().main_fun(X, src, tgt, nt, MaxPar=3, N=3000, output=10, rng_kind=RNG_WH, seeds=(10437, 13568, 30524))
        for k in INT_COLS + ("globalLL",):
            assert np.array_equal(getattr(o, k), getattr(r, k)), k
    with pytest.raises(RuntimeError):
        oracle.mcmc(X, src, tgt, nt, max_par=3, n_iter=10, output=10, initial_network=0, rng_kind=RNG_WH)


def test_chain_core_host_build_rare_legal_children(emu_lib, oracle):
    from oracle.oracle import RNG_WH
    from test_host_logic import _emu_run
    X, src, tgt, nt = rare_children_case()
    ref = oracle.mcmc(X, src, tgt, nt, max_par=8, omega=1.0, n_iter=1500, output=5, rng_kind=RNG_WH, seeds=(7, 8, 9))
    r = _emu_run(emu_lib, dict(X=X, source=src, target=tgt, node_type=nt), 8, 1500, 5, 0, (7, 8, 9), omega=1.0)
    _emu_same(r, ref)
    assert ref.uniforms > 150 * 1500   # ~330 child draws per addition


@pytest.mark.parametrize("max_par,P", [(5, 40), (12, 60)])
def test_chain_core_host_build_initial_network_1(emu_lib, oracle, max_par, P):
    """The defined random start (include/bn_b200.h): same stream, same graph, same chain as the
    oracle's statement of it; the start graph is a DAG without duplicate parents."""
    from oracle.oracle import RNG_WH
    from test_host_logic import _emu_run
    X, g, nt = synthetic(P, 300, max_par, 31)
    ref = oracle.mcmc(X, g.source, g.target, nt, max_par=max_par, n_iter=3000, output=7, initial_network=1,
                      rng_kind=RNG_WH, seeds=(5, 6, 7))
    start = oracle.mcmc(X, g.source, g.target, nt, max_par=max_par, n_iter=0, output=7, initial_network=1,
                        rng_kind=RNG_WH, seeds=(5, 6, 7))
    assert start.final_npar.sum() > P and start.uniforms > start.final_npar.sum()
    for c in range(P):
        ps = list(start.final_parents[c, :start.final_npar[c]])
        assert len(set(ps)) == len(ps) and c not in ps
        assert nt[c] != 1 or not ps
    r = _emu_run(emu_lib, dict(X=X, source=g.source, target=g.target, node_type=nt), max_par, 3000, 7, 0,
                 (5, 6, 7), init=1)
    _emu_same(r, ref)


# ---------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_rare_legal_children_vs_oracle(oracle):
    """ADVICE r1: an iteration that needs more uniforms than the ring holds is not an error."""
    from bayesnetworks_b200 import Context
    from oracle.oracle import RNG_WH
    X, src, tgt, nt = rare_children_case()
    ref = oracle.mcmc(X, src, tgt, nt, max_par=8, omega=1.0, n_iter=1500, output=5, rng_kind=RNG_WH, seeds=(7, 8, 9))
    with Context.from_data(X, src, tgt, nt, max_par=8, omega=1.0) as ctx:
        res, _ = ctx.run(n_chains=3, n_iter=1500, output=5, rng="wh", seeds=[(7, 8, 9), (17, 18, 19), (7, 8, 9)],
                         log_moves=True)
    _same_trace(res[0], ref, X.shape[0])
    _same_trace(res[2], ref, X.shape[0])


@pytest.mark.gpu
def test_gpu_supplied_graph_denser_than_maxpar(oracle, dataset):
    from bayesnetworks_b200 import BnError, Context, _lib
    from oracle.oracle import RNG_WH
    X, src, tgt, nt = dataset["X"], dataset["source"], dataset["target"], dataset["node_type"]
    ref = oracle.mcmc(X, src, tgt, nt, max_par=3, n_iter=3000, output=10, rng_kind=RNG_WH)
    with Context.from_data(X, src, tgt, nt, max_par=3) as ctx:
        r = ctx.run(n_iter=3000, output=10, rng="wh", log_moves=True)[0][0]
        _same_trace(r, ref, 2000)
        with pytest.raises(BnError) as ei:     # ... but the chain cannot START from it
            ctx.run(n_iter=10, initial_network=0)
        assert ei.value.status == _lib.BN_ERR_BAD_ARG
        with pytest.raises(BnError):           # any value but 1 / 2 keeps the supplied graph (src/network.h:148-170)
            ctx.run(n_iter=10, initial_network=7)
    ref7 = oracle.mcmc(X, src, tgt, nt, max_par=8, n_iter=500, output=10, initial_network=0, rng_kind=RNG_WH)
    with Context.from_data(X, src, tgt, nt, max_par=8) as ctx:
        _same_trace(ctx.run(n_iter=500, output=10, rng="wh", initial_network=7, log_moves=True)[0][0], ref7, 2000)


@pytest.mark.gpu
@pytest.mark.parametrize("max_par,P", [(5, 40), (12, 60), (8, 1000)])
def test_gpu_initial_network_1_vs_oracle(oracle, max_par, P):
    from bayesnetworks_b200 import Context
    from oracle.oracle import RNG_WH
    X, g, nt = synthetic(P, 300, max_par, 31)
    n_iter = 3000
    ref = oracle.mcmc(X, g.source, g.target, nt, max_par=max_par, n_iter=n_iter, output=7, initial_network=1,
                      rng_kind=RNG_WH, seeds=(5, 6, 7))
    with Context.from_data(X, g.source, g.target, nt, max_par=max_par) as ctx:
        r = ctx.run(n_iter=n_iter, output=7, rng="wh", seeds=(5, 6, 7), initial_network=1, log_moves=True)[0][0]
    _same_trace(r, ref, 300)


@pytest.mark.gpu
def test_gpu_mersenne_twister_state_in_and_out(oracle, dataset, golden):
    """f1: the chain starts from R's stream state (.Random.seed[2:626]) and hands back the state
    after exactly the uniforms it consumed (src/RcppExports.cpp:13: GetRNGstate / PutRNGstate)."""
    from bayesnetworks_b200 import Context
    X, src, tgt, nt = dataset["X"], dataset["source"], dataset["target"], dataset["node_type"]
    with Context.from_data(X, src, tgt, nt, max_par=50) as ctx:
        st0 = oracle.rmt_state_after(1234, 0)                       # the state set.seed(1234) leaves
        r = ctx.run(n_iter=50000, output=100, rng="rmt", mt_state=st0, log_moves=True)[0][0]
        for k in INT_COLS:
            assert np.array_equal(r.trace[k], golden[f"cfg1_{k}"]), k
        assert np.array_equal(r.accepted_moves, golden["cfg1_accepted_moves"])
        assert r.uniforms == 250277
        assert np.array_equal(r.mt_state, oracle.rmt_state_after(1234, 250277))
        # mid-stream state (position inside the 624-word block) and two chains with different states
        st_a, st_b = oracle.rmt_state_after(99, 1000), oracle.rmt_state_after(7, 5)
        assert 0 < st_a[0] < 624
        res, _ = ctx.run(n_chains=2, n_iter=3000, output=10, rng="rmt", mt_state=np.stack([st_a, st_b]))
        u = oracle.uniforms(1000 + 40000, 1, (99,))[1000:]          # R-MT seed 99, from draw 1,000 on
        from oracle.oracle import RNG_REPLAY
        ref = oracle.mcmc(X, src, tgt, nt, max_par=50, n_iter=3000, output=10, rng_kind=RNG_REPLAY, replay=u)
        for k in INT_COLS:
            assert np.array_equal(res[0].trace[k], getattr(ref, k)), k
        assert np.array_equal(res[0].mt_state, oracle.rmt_state_after(0, res[0].uniforms, state=st_a))
        assert np.array_equal(res[1].mt_state, oracle.rmt_state_after(0, res[1].uniforms, state=st_b))
        # same start through seeds (set.seed) and through the state: same chain
        r_seed = ctx.run(n_iter=3000, output=10, rng="rmt", seeds=7, want_mt_state=True)[0][0]
        r_state = ctx.run(n_iter=3000, output=10, rng="rmt", mt_state=oracle.rmt_state_after(7, 0))[0][0]
        assert np.array_equal(r_seed.trace["ChangedNode"], r_state.trace["ChangedNode"])
        assert np.array_equal(r_seed.mt_state, r_state.mt_state)


@pytest.mark.gpu
def test_gpu_replay_buffer_exhausted_is_an_error(dataset):
    from bayesnetworks_b200 import BnError, Context, _lib
    X, src, tgt, nt = dataset["X"], dataset["source"], dataset["target"], dataset["node_type"]
    with Context.from_data(X, src, tgt, nt, max_par=8) as ctx:
        with pytest.raises(BnError) as ei:
            ctx.run(n_iter=1000, output=10, rng="replay", replay=np.random.default_rng(1).random(500))
        assert ei.value.status == _lib.BN_ERR_CAPACITY


@pytest.mark.gpu
def test_gpu_few_samples_with_default_maxpar(oracle):
    """ADVICE r1: MaxPar = 50 with fewer than 52 samples runs (the parent sets that occur are small)."""
    from bayesnetworks_b200 import Context
    from oracle.oracle import RNG_WH
    X, g, nt = synthetic(30, 45, 50, 77)
    ref = oracle.mcmc(X, g.source, g.target, nt, max_par=50, n_iter=2000, output=10, initial_network=2, rng_kind=RNG_WH)
    with Context.from_data(X, g.source, g.target, nt, max_par=50) as ctx:
        r = ctx.run(n_iter=2000, output=10, rng="wh", log_moves=True)[0][0]
    _same_trace(r, ref, 45)


def collinear_case():
    """Column 7 is an exact copy of column 3 and column 11 an exact linear combination of 2 and 5:
    parent sets containing such a pair have a singular Gram, and a node regressed on its own copy
    has RSS = 0."""
    X, g, nt = synthetic(24, 400, 8, 55)
    X = np.array(X)
    X[:, 7] = X[:, 3]
    X[:, 11] = 0.5 * X[:, 2] - 1.5 * X[:, 5]
    nt = np.zeros_like(nt)
    return np.asfortranarray(X), g, nt


def test_chain_core_host_build_collinear_columns(emu_lib):
    """Degenerate data (ADVICE r1): exact fits / singular parent sets are refused and counted, the
    node scores stay finite -- no NaN that would accept everything afterwards."""
    from test_host_logic import _emu_run
    X, g, nt = collinear_case()
    r = _emu_run(emu_lib, dict(X=X, source=g.source, target=g.target, node_type=nt), 8, 20000, 10, 0, (3, 4, 5), omega=0.5)
    assert r["rc"] == 0 and int(r["cnt"][10]) > 0
    assert np.isfinite(r["globalLL"]).all()
    for c in (3, 7):
        ps = set(int(q) for q in r["fpar"][c, :r["fnpar"][c]])
        assert not ({3, 7} - {c}) & ps   # a column is never regressed on its own copy


@pytest.mark.gpu
def test_gpu_collinear_columns_are_flagged():
    from bayesnetworks_b200 import Context
    X, g, nt = collinear_case()
    with Context.from_data(X, g.source, g.target, nt, max_par=8, omega=0.5) as ctx:
        res, _ = ctx.run(n_chains=2, n_iter=20000, output=10, rng="wh", seeds=[(3, 4, 5), (6, 7, 8)])
        for r in res:
            assert r.n_nonpd > 0 and np.isfinite(r.trace["globalLL"]).all()
            for c in (3, 7):
                assert not ({3, 7} - {c}) & set(int(q) for q in r.final_parents[c, :r.final_npar[c]])
        base, score, hr = ctx.score_all_proposals(res[0].final_parents, res[0].final_npar)
        assert np.isfinite(base).all() and score[0, 3, 7] == -np.inf and score[0, 7, 3] == -np.inf


@pytest.mark.gpu
@pytest.mark.parametrize("n_samples", [20000, 20001])
def test_gpu_pageable_matrix_takes_the_staged_copy(n_samples):
    """A pageable host matrix above 32 MB (what R hands over) is staged through pinned buffers by a few
    host threads (gram.cu: StagePool); same statistics as the one-shot paths, ragged sample counts too."""
    import torch
    from bayesnetworks_b200 import Context
    rng = np.random.default_rng(3)
    P = 300
    X = np.asfortranarray(rng.standard_normal((n_samples, P)) + rng.uniform(-2, 2, P))   # 48 MB, pageable
    nt = np.zeros(P, np.int32)
    with Context.from_data(X, [1], [2], nt, max_par=4) as a:
        sa = a.stats()
    Xd = torch.from_numpy(np.ascontiguousarray(X.T)).cuda()
    with Context.from_device(Xd.data_ptr(), n_samples, n_samples, P, [1], [2], nt, max_par=4) as b:
        sb = b.stats()
    for x, y in zip(sa, sb):
        assert np.array_equal(x, y)          # same bits as the device-resident build
    mean = X.mean(axis=0)
    Xc = X - mean
    np.testing.assert_allclose(sa[3], Xc.T @ Xc, rtol=1e-11, atol=1e-7)
