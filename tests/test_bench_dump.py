"""bench.py --dump-outputs: the arrays of the last timed step as float64 .npy files, capped in size."""
import os

import numpy as np

import bench
from bayesnetworks_b200.api import ChainResult


def _chain(rows, rng):
    trace = {k: rng.integers(0, 1000, rows).astype(np.int32) for k in bench.TRACE_COLS}
    trace["globalLL"] = rng.standard_normal(rows)
    return ChainResult(trace=trace, uniforms=3 * 10 ** 12, valid_iters=rows, proposed=(1, 2, 3), reject=(0, 1, 2),
                       n_nonpd=0, total_edges=9, windows=1, alg_bytes=0, phase_cycles=(), slots_simulated=0,
                       final_parents=rng.integers(-1, 40, (40, 8)).astype(np.int32),
                       final_npar=rng.integers(0, 9, 40).astype(np.int32))


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def _same_traces(got, res):
    """The trace columns are the chains' rows end to end; n_rows splits them."""
    ends = np.cumsum(got["n_rows"]).astype(int)
    for k in bench.TRACE_COLS:
        parts = np.split(got["trace_" + k], ends[:-1])
        assert len(parts) == len(res)
        for part, r in zip(parts, res):
            assert np.array_equal(part, r.trace[k]), k


def test_dump_outputs_one_gpu(tmp_path, monkeypatch):
    rng = np.random.default_rng(3)
    res = [_chain(6, rng), _chain(4, rng), _chain(5, rng)]   # chains write different numbers of rows
    full = bench.step_outputs({"results": res}, 1)
    bench.dump_outputs(str(tmp_path / "all"), full)
    got = _load(tmp_path / "all")
    assert all(v.dtype == np.float64 and np.isfinite(v).all() for v in got.values())
    assert np.array_equal(got["n_rows"], [6, 4, 5]) and np.array_equal(got["chain_index"], [0, 1, 2])
    _same_traces(got, res)
    assert np.array_equal(got["final_parents"], np.stack([r.final_parents for r in res]))
    assert np.array_equal(got["uniforms"], [3 * 10 ** 12] * 3)
    assert np.array_equal(got["proposed"], [[1, 2, 3]] * 3)
    # above the size limit: a seeded sample of whole chains, the same one every time
    monkeypatch.setattr(bench, "DUMP_LIMIT", 7000)   # any two of the ~3.3 KB chains, not three
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), full)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    idx = a["chain_index"].astype(int)
    assert len(idx) == 2 and all(np.array_equal(a[k], b[k]) for k in a)
    assert sum(v.size for v in a.values()) * 8 <= bench.DUMP_LIMIT
    _same_traces(a, [res[i] for i in idx])
    assert np.array_equal(a["final_parents"], got["final_parents"][idx])


def test_dump_outputs_chain_larger_than_limit(tmp_path, monkeypatch):
    """No whole chain fits: one chain with a seeded sample of its trace rows, still within the limit."""
    rng = np.random.default_rng(4)
    res = [_chain(500, rng) for _ in range(3)]   # ~35 KB each
    full = bench.step_outputs({"results": res}, 1)
    monkeypatch.setattr(bench, "DUMP_LIMIT", 20000)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), full)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert all(np.array_equal(a[k], b[k]) for k in a)
    assert sum(v.size for v in a.values()) * 8 <= bench.DUMP_LIMIT
    (c,) = a["chain_index"].astype(int)
    rows = a["row_index"].astype(int)
    assert 100 < len(rows) < 500 and np.all(np.diff(rows) > 0) and a["n_rows"][0] == 500
    for k in bench.TRACE_COLS:
        assert np.array_equal(a["trace_" + k], res[c].trace[k][rows]), k
    assert np.array_equal(a["final_parents"][0], res[c].final_parents)


def test_dump_outputs_gathered_traces(tmp_path):
    """N > 1: the all-gathered device buffers ([chains, capacity, 7] ints, [chains, capacity] globalLL) past each
    chain's n_rows hold no rows, and none of that is written."""
    import torch
    from bayesnetworks_b200.dist import INT_COLUMNS
    ints = torch.arange(2 * 5 * 7, dtype=torch.int32).reshape(2, 5, 7)
    gll = -torch.arange(10, dtype=torch.float64).reshape(2, 5)
    n_rows = torch.tensor([5, 3], dtype=torch.int32)
    bench.dump_outputs(str(tmp_path), bench.step_outputs({"out": dict(ints=ints, gll=gll, n_rows=n_rows)}, 2))
    got = _load(tmp_path)
    assert all(np.isfinite(v).all() for v in got.values())
    assert np.array_equal(got["trace_globalLL"], [0, -1, -2, -3, -4, -5, -6, -7])
    for i, k in enumerate(INT_COLUMNS):
        assert np.array_equal(got["trace_" + k], np.concatenate([ints[0, :, i], ints[1, :3, i]])), k
