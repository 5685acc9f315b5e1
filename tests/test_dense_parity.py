"""Dense-regime parity at the benchmark's own shape (P = 896, 897, 1000, 1024, 1025; MaxPar 8).

Fixtures (tests/golden/dense_ref.npz) come from the UNMODIFIED reference sources
(oracle/_ref, src/bayesnet_mcmc.cpp:45-70 + src/network.h:281-336,366-432) via
tests/golden/make_golden_dense.py: 20,000 iterations per case, thousands of accepted
additions and deletions, nodes saturating MaxPar, 7-30 % invalid (cyclic / stale) iterations.

CPU tests pin the C restatement (and the host build of the chain core) to those fixtures;
the `gpu` tests run the CUDA chain through the C ABI against the same fixtures: the
8-chunk ancestor path (897..1,024 nodes, all per-chain state in shared memory) is the one
every BENCH/SCALE number runs on.
"""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
from make_golden_dense import (COLS, MAX_PAR, N_ITER, N_ROWS, OUTPUT, dense_cases, dense_inputs,  # noqa: E402
                               moves_digest, x_digest)

INT_COLS = ("iter", "ChangedNode", "movetype", "additions", "deletions", "FN", "FP")
CASES = {c[0]: c for c in dense_cases()}
SINGLE = [n for n in CASES if "chain" not in n]
CHAINS = [f"p1000_chain{c}" for c in range(8)]


@pytest.fixture(scope="module")
def dense():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dense_ref.npz"))


_inputs = {}


def inputs_for(P, dense):
    """Regenerated from the seeds; the stored checksum proves it is the matrix the reference saw."""
    if P not in _inputs:
        X, g, nt = dense_inputs(P)
        assert x_digest(X) == bytes(dense[f"x_sha1_p{P}"]).decode(), "synthetic generator drifted: regenerate the fixture"
        _inputs[P] = (X, g, nt)
    return _inputs[P]


def check_against_fixture(dense, name, cols, uniforms, moves, edges, n_nonpd, gll_exact):
    for k in INT_COLS:
        assert np.array_equal(cols[k], dense[f"{name}_{k}"]), (name, k)
    if gll_exact:
        assert np.array_equal(cols["globalLL"], dense[f"{name}_globalLL"]), name
    else:
        # north_star tolerance: 1e-9 relative (atol for scores that are ~0, as in test_gpu_parity)
        assert np.allclose(cols["globalLL"], dense[f"{name}_globalLL"], rtol=1e-9, atol=1e-9 * N_ROWS / 2), name
    assert int(uniforms) == int(dense[f"{name}_uniforms"]), name
    assert len(moves) == int(dense[f"{name}_n_moves"]), name
    if f"{name}_moves_iter" in dense:
        want = np.stack([dense[f"{name}_moves_iter"], dense[f"{name}_moves_type"], dense[f"{name}_moves_child"],
                         dense[f"{name}_moves_parent"]], 1).astype(np.int64)
        got = np.asarray(moves, dtype=np.int64)
        bad = np.nonzero((got != want).any(axis=1))[0]
        assert bad.size == 0, f"{name}: accepted move {bad[0]} differs: got {got[bad[0]]}, reference {want[bad[0]]}"
    assert moves_digest(moves) == bytes(dense[f"{name}_moves_sha1"]).decode(), name
    assert np.array_equal(np.asarray(edges, dtype=np.int64).reshape(-1, 2),
                          dense[f"{name}_final_edges"].astype(np.int64).reshape(-1, 2)), name
    assert n_nonpd == 0, name


# ---------------------------------------------------------------------------
# CPU: the oracle port and the host build of the chain core against the reference fixture
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("name", SINGLE + CHAINS[:2])
def test_port_pinned_to_reference_dense(oracle, dense, name):
    """bn_oracle.c == oracle/_ref on dense cases, bit for bit (globalLL included)."""
    from oracle.oracle import RNG_WH
    _, P, phi, omega, seeds = CASES[name]
    X, g, nt = inputs_for(P, dense)
    o = oracle.mcmc(X, g.source, g.target, nt, max_par=MAX_PAR, phi=phi, omega=omega, n_iter=N_ITER,
                    output=OUTPUT, rng_kind=RNG_WH, seeds=seeds)
    check_against_fixture(dense, name, {k: getattr(o, k) for k in COLS}, o.uniforms, o.accepted_moves(),
                          o.edges(), o.n_nonpd, gll_exact=True)
    assert list(o.reject) == list(dense[f"{name}_reject"])
    assert list(o.proposed) == list(dense[f"{name}_proposed"])


@pytest.mark.parametrize("name", ["p1000_mid", "p1024_sat", "p1025_sat"])
def test_chain_core_host_build_dense(emu_lib, dense, name):
    """The chain core compiled for the host (one-lane warp) on the same cases: round logic,
    record repair, ancestor updates -- everything but the multi-lane code paths."""
    from test_host_logic import _emu_run
    _, P, phi, omega, seeds = CASES[name]
    X, g, nt = inputs_for(P, dense)
    ds = dict(X=X, source=g.source, target=g.target, node_type=nt)
    r = _emu_run(emu_lib, ds, MAX_PAR, N_ITER, OUTPUT, 0, seeds, phi=phi, omega=omega)
    assert r["rc"] == 0
    edges = [(int(r["fpar"][c, e]), c) for c in range(P) for e in range(int(r["fnpar"][c]))]
    check_against_fixture(dense, name, r, r["cnt"][0], r["moves"], edges, int(r["cnt"][10]), gll_exact=False)


# ---------------------------------------------------------------------------
# GPU: the CUDA chain through the C ABI
# ---------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", SINGLE)
def test_gpu_chain_dense_benchmark_shape(dense, name):
    from bayesnetworks_b200 import Context
    _, P, phi, omega, seeds = CASES[name]
    X, g, nt = inputs_for(P, dense)
    with Context.from_data(X, g.source, g.target, nt, max_par=MAX_PAR, phi=phi, omega=omega) as ctx:
        r = ctx.run(n_iter=N_ITER, output=OUTPUT, rng="wh", seeds=seeds, log_moves=True)[0][0]
    check_against_fixture(dense, name, r.trace, r.uniforms, r.accepted_moves, r.edges(), r.n_nonpd, gll_exact=False)
    assert list(r.reject) == list(dense[f"{name}_reject"])
    assert list(r.proposed) == list(dense[f"{name}_proposed"])


@pytest.mark.gpu
def test_gpu_eight_chains_dense_p1000(dense):
    """Eight chains in one launch (eight CTAs) at the benchmark's node count, each against the
    reference's trajectory for its seeds; chain 0 alone gives the same bits."""
    from bayesnetworks_b200 import Context
    X, g, nt = inputs_for(1000, dense)
    seeds = np.array([CASES[n][4] for n in CHAINS], dtype=np.int32)
    with Context.from_data(X, g.source, g.target, nt, max_par=MAX_PAR, phi=0.0, omega=0.0) as ctx:
        res, _ = ctx.run(n_chains=8, n_iter=N_ITER, output=OUTPUT, rng="wh", seeds=seeds, log_moves=True)
        one = ctx.run(n_chains=1, n_iter=N_ITER, output=OUTPUT, rng="wh", seeds=seeds[:1], log_moves=True)[0][0]
    for name, r in zip(CHAINS, res):
        check_against_fixture(dense, name, r.trace, r.uniforms, r.accepted_moves, r.edges(), r.n_nonpd,
                              gll_exact=False)
    for k in INT_COLS + ("globalLL",):
        assert np.array_equal(one.trace[k], res[0].trace[k]), k
    assert np.array_equal(one.accepted_moves, res[0].accepted_moves)
