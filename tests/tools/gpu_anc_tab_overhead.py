"""Cost of the posterior ancestor tabulation (GPU) on the benchmark workload: 1,000 nodes x 100,000 samples,
MaxPar 8, 64 chains x 100,000 iterations (bench.py's graph and data seeds).

Three arms run in alternating rounds, each timed by the device events of bn_run around the chain kernel:
  default   the benchmark's own call
  state     want_state=True: the kernels the tabulation runs on, without it
  anc       tabulate_ancestors=True
The tabulation's own cost is anc - state; the switch to those kernels is state - default.  The cost per
accepted move divides anc - state by the accepted additions and deletions of all chains (the three arms run
the same chains); the cost per ancestor-changing move divides it by those moves that change the closure,
counted by the from-scratch replay of tests/emu/anc_replay.cpp on the first `--replay-chains` chains and
scaled to all chains; the same replay counts the ancestor bits those moves flip, each one counter
update.  Prints one JSON line with the card's name and power limit.

    python tests/tools/gpu_anc_tab_overhead.py [--rounds 4] [--out anc_tab_overhead.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

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
    ap.add_argument("--replay-chains", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from bayesnetworks_b200 import Context
    from bayesnetworks_b200.synth import make_dag, make_prior, simulate_numpy
    from test_ancestor_tab import empty_start, replay
    P, N, MP, NC, ITERS, OUT = 1000, 100000, 8, 64, 100000, 100
    dag = make_dag(P, seed=42)
    g = make_prior(dag, max_par=MP, seed=43)
    X = simulate_numpy(dag, N, seed=42)
    seeds = np.array([(1 + (7919 * c) % 30000, 1 + (104729 * c + 17) % 30000, 1 + (1299709 * c + 31) % 30000)
                      for c in range(NC)], np.int32)
    arms = {"default": {}, "state": dict(want_state=True), "anc": dict(tabulate_ancestors=True)}
    ms = {k: [] for k in arms}
    with Context.from_data(X, g.source, g.target, g.node_type_codes(), max_par=MP) as ctx:
        kw = dict(n_chains=NC, n_iter=ITERS, output=OUT, rng="wh", seeds=seeds)
        for extra in arms.values():  # warm-up of every kernel the rounds use
            ctx.run(**{**kw, "n_iter": 1000}, **extra)
        res = None
        for _ in range(a.rounds):
            for name, extra in arms.items():
                r, t = ctx.run(**kw, **extra)
                ms[name].append(t)
                if name == "anc":
                    res = r
        accepted = sum(r.proposed[t] - r.reject[t] for r in res for t in (1, 2))
        # closure-changing moves of the first chains, from a logged run of the same chains
        k = a.replay_chains
        logged = ctx.run(**{**kw, "n_chains": k, "seeds": seeds[:k]}, log_moves=True)[0]
    stats = np.zeros(2, np.int64)
    n_changed, n_flips, n_moves = 0, 0, 0
    for r in logged:
        par, npar = empty_start(P, MP)
        replay(par, npar, r.accepted_moves, 0, ITERS, 0, stats=stats)
        n_changed += int(stats[0])
        n_flips += int(stats[1])
        n_moves += len(r.accepted_moves)
    frac = n_changed / n_moves
    mean = {k: float(np.mean(v)) for k, v in ms.items()}
    tab_ms = mean["anc"] - mean["state"]
    row = {"card": card(), "shape": f"{P} nodes x {N} samples, MaxPar {MP}, {NC} chains x {ITERS} iterations",
           "rounds_ms": ms, "mean_ms": mean, "anc_over_default": mean["anc"] / mean["default"],
           "state_over_default": mean["state"] / mean["default"], "tabulation_ms": tab_ms,
           "accepted_moves_all_chains": accepted, "ancestor_changing_fraction": frac,
           "replayed_chains": k, "ns_per_accepted_move_per_chain": 1e6 * tab_ms / (accepted / NC),
           "ns_per_ancestor_changing_move_per_chain": 1e6 * tab_ms / (frac * accepted / NC),
           "bits_flipped_per_ancestor_changing_move": n_flips / n_changed,
           "ns_per_flipped_bit_per_chain": 1e6 * tab_ms / (n_flips / n_moves * accepted / NC)}
    print(json.dumps(row), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            json.dump(row, fh, indent=1)


if __name__ == "__main__":
    main()
