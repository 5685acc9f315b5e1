"""Cost of the best-graph tracking (GPU) on the benchmark workload: 1,000 nodes x 100,000 samples, MaxPar 8,
64 chains x 100,000 iterations (bench.py's graph and data seeds), with drop 0 and drop 20,000.

Two arms run in alternating rounds on the same chains, each timed by the device events of bn_run around the
chain kernel:
  state     want_state=True: the kernels the tracking runs on, without it
  best      want_state=True, track_best=True
The tracking's own cost is best - state; per accepted move after drop it divides that by the accepted
additions and deletions of all chains (an exact sum of the node scores and a compare per such move, and a
copy of the changed lists per new best).  Prints one JSON line with the card's name and power limit.

    python tests/tools/gpu_best_overhead.py [--rounds 4] [--out best_overhead.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def card():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from bayesnetworks_b200 import Context
    from bayesnetworks_b200.synth import make_dag, make_prior, simulate_numpy
    P, N, MP, NC, ITERS, OUT = 1000, 100000, 8, 64, 100000, 100
    dag = make_dag(P, seed=42)
    g = make_prior(dag, max_par=MP, seed=43)
    X = simulate_numpy(dag, N, seed=42)
    seeds = np.array([(1 + (7919 * c) % 30000, 1 + (104729 * c + 17) % 30000, 1 + (1299709 * c + 31) % 30000)
                      for c in range(NC)], np.int32)
    arms = {"state": dict(want_state=True), "best": dict(want_state=True, track_best=True)}
    rows = []
    with Context.from_data(X, g.source, g.target, g.node_type_codes(), max_par=MP) as ctx:
        for drop in (0, 20000):
            kw = dict(n_chains=NC, n_iter=ITERS, output=OUT, rng="wh", seeds=seeds, drop=drop)
            for extra in arms.values():  # warm-up of every kernel the rounds use
                ctx.run(**{**kw, "n_iter": 1000}, **extra)
            ms = {k: [] for k in arms}
            res = None
            for _ in range(a.rounds):
                for name, extra in arms.items():
                    r, t = ctx.run(**kw, **extra)
                    ms[name].append(t)
                    if name == "best":
                        res = r
            accepted = sum(r.proposed[t] - r.reject[t] for r in res for t in (1, 2))   # (counted from drop on)
            mean = {k: float(np.mean(v)) for k, v in ms.items()}
            track_ms = mean["best"] - mean["state"]
            rows.append({"drop": drop, "rounds_ms": ms, "mean_ms": mean, "best_over_state": mean["best"] / mean["state"],
                         "tracking_ms": track_ms, "accepted_moves_after_drop_all_chains": accepted,
                         "ns_per_accepted_move_per_chain": 1e6 * track_ms / max(accepted / NC, 1),
                         "best_iter_per_chain_min_max": [min(r.best.iter for r in res), max(r.best.iter for r in res)]})
    out = {"card": card(), "shape": f"{P} nodes x {N} samples, MaxPar {MP}, {NC} chains x {ITERS} iterations",
           "runs": rows}
    print(json.dumps(out), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
