"""Cost of the Markov blanket tabulation (GPU) on the benchmark workload: 1,000 nodes x 100,000 samples, MaxPar 8,
64 chains x 100,000 iterations (bench.py's graph and data seeds), with drop 0 and drop 20,000.

Two arms run in alternating rounds on the same chains, each timed by the device events of bn_run around the
chain kernel:
  state     want_state=True: the kernels the tabulation runs on, without it
  mb        want_state=True, tabulate_markov_blankets=True
The tabulation's own cost is mb - state.  Its per-move work runs on every accepted move, before drop too, so the
cost per accepted move divides it by all accepted additions and deletions of the chains (counted once from a
move log: the trajectory does not depend on drop).  Also reports the memory the tabulation takes: the int32
counts and the 16-bit witness matrix, P * P each per chain.  Prints one JSON line with the card's name and
power limit.

    python tests/tools/gpu_mb_overhead.py [--rounds 4] [--out mb_overhead.json]
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
    arms = {"state": dict(want_state=True), "mb": dict(want_state=True, tabulate_markov_blankets=True)}
    rows = []
    with Context.from_data(X, g.source, g.target, g.node_type_codes(), max_par=MP) as ctx:
        base = dict(n_chains=NC, n_iter=ITERS, output=OUT, rng="wh", seeds=seeds)
        logged = ctx.run(**base, log_moves=True)[0]
        accepted = sum(len(r.accepted_moves) for r in logged)
        final_edges = [int(r.final_npar.sum()) for r in logged]
        for drop in (0, 20000):
            kw = dict(base, drop=drop)
            for extra in arms.values():  # warm-up of every kernel the rounds use
                ctx.run(**{**kw, "n_iter": 1000}, **extra)
            ms = {k: [] for k in arms}
            res = None
            for _ in range(a.rounds):
                for name, extra in arms.items():
                    r, t = ctx.run(**kw, **extra)
                    ms[name].append(t)
                    if name == "mb":
                        res = r
            mean = {k: float(np.mean(v)) for k, v in ms.items()}
            tab_ms = mean["mb"] - mean["state"]
            off = ~np.eye(P, dtype=bool)
            rows.append({"drop": drop, "rounds_ms": ms, "mean_ms": mean, "mb_over_state": mean["mb"] / mean["state"],
                         "tabulation_ms": tab_ms, "accepted_moves_all_chains": accepted,
                         "ns_per_accepted_move_per_chain": 1e6 * tab_ms / max(accepted / NC, 1),
                         "tabulated_iterations": int(res[0].mb_freq[0, 0]),
                         "blanket_pairs_ever_per_chain_mean": float(np.mean([(r.mb_freq[off] > 0).sum() / 2
                                                                              for r in res]))})
    out = {"card": card(), "shape": f"{P} nodes x {N} samples, MaxPar {MP}, {NC} chains x {ITERS} iterations",
           "memory_bytes": {"counts_int32": NC * P * P * 4, "witnesses_uint16": NC * P * P * 2},
           "final_edges_per_chain_min_max": [min(final_edges), max(final_edges)], "runs": rows}
    print(json.dumps(out), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
