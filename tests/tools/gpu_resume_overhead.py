"""Cost of resuming chains (GPU): one run of n_iter iterations against the same run in ten resumed
segments, with and without the score block, on two shapes:

  bench     the benchmark's shape, 64 chains x 100,000 iterations, 1,000 nodes x 100,000 samples, MaxPar 8
  config3   100 nodes x 10,000 samples, MaxPar 50, 64 chains x 20,000 iterations

Times are host wall clock around bn_run (each call ends in a device synchronise), the best of `--reps`;
the per-segment overhead is (segments - one run) / (segments - 1).  Prints one JSON line per case with the
card's name and power limit.

    python tests/tools/gpu_resume_overhead.py [--reps 2] [--out resume_overhead.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return q
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return time.perf_counter() - t0, out


def case(name, ctx, n_chains, n_iter, output, segments, reps):
    kw = dict(n_chains=n_chains, output=output, rng="wh")
    one = min(timed(lambda: ctx.run(n_iter=n_iter, **kw))[0] for _ in range(reps))
    res = {"case": name, "chains": n_chains, "iters": n_iter, "segments": segments, "one_run_s": one}
    for label, keep_scores in (("with_score_block", True), ("without_score_block", False)):
        best = None
        for _ in range(reps):
            t, start = 0.0, None
            for i in range(segments):
                dt, (out, _) = timed(lambda: ctx.run(n_iter=n_iter // segments, start=start, want_state=True, **kw))
                t += dt
                start = [r.state for r in out]
                if not keep_scores:
                    for s in start:
                        s.score_block = None
            best = t if best is None else min(best, t)
        res[f"{label}_s"] = best
        res[f"{label}_per_segment_overhead_ms"] = 1e3 * (best - one) / (segments - 1)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from bayesnetworks_b200 import Context
    from bayesnetworks_b200.synth import make_dag, make_prior, simulate_numpy
    rows = []
    for name, P, N, mp, n_iter, seed in (("bench", 1000, 100000, 8, 100000, 0), ("config3", 100, 10000, 50, 20000, 42)):
        dag = make_dag(P, seed=seed)
        g = make_prior(dag, max_par=mp, seed=seed + 1)
        X = simulate_numpy(dag, N, seed=seed + 2)
        with Context.from_data(X, g.source, g.target, g.node_type_codes(), max_par=mp) as ctx:
            ctx.run(n_chains=64, n_iter=1000, output=100, rng="wh")  # warm-up: module load, pools
            r = case(name, ctx, 64, n_iter, 100, 10, a.reps)
        r["card"] = card()
        rows.append(r)
        print(json.dumps(r), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(rows, fh, indent=1)


if __name__ == "__main__":
    main()
