"""Golden trace of a supplied graph denser than MaxPar (tests/test_round2_api.py).

    python tests/golden/make_golden_denser.py

The shipped `network` dataset with its prior DAG as the start graph (InitialNetwork = 2; one node has
8 prior parents) and MaxPar 3: 3,000 Wichmann-Hill iterations from the reference seeds, a row every 10.
Where oracle/_ref is built (``make -C oracle ref``) the trace comes from the UNMODIFIED reference
sources and the C restatement (oracle/bn_oracle.c) is asserted identical to it; elsewhere it comes
from the restatement.  The file's `source` entry says which.

Writes tests/golden/denser_maxpar3.npz (committed).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle.oracle import RNG_WH, Oracle, Ref, have_ref  # noqa: E402

COLS = ("iter", "ChangedNode", "movetype", "globalLL", "additions", "deletions", "FN", "FP")
MAX_PAR, N_ITER, OUTPUT = 3, 3000, 10
SEEDS = (10437, 13568, 30524)


def main():
    z = np.load(os.path.join(HERE, "network_p3sim8.npz"))
    X, src, tgt, nt = z["X"], z["source"], z["target"], z["node_type"]
    o = Oracle().mcmc(X, src, tgt, nt, max_par=MAX_PAR, n_iter=N_ITER, output=OUTPUT, rng_kind=RNG_WH, seeds=SEEDS)
    out, source = {k: getattr(o, k) for k in COLS}, "oracle/bn_oracle.c"
    if have_ref():
        r = Ref().main_fun(X, src, tgt, nt, MaxPar=MAX_PAR, N=N_ITER, output=OUTPUT, rng_kind=RNG_WH, seeds=SEEDS)
        for k in COLS:
            assert np.array_equal(getattr(r, k), out[k]), k
        out, source = {k: getattr(r, k) for k in COLS}, "oracle/_ref (reference sources)"
    np.savez_compressed(os.path.join(HERE, "denser_maxpar3.npz"), source=np.array(source), **out)
    print(f"denser_maxpar3.npz written from {source}")


if __name__ == "__main__":
    main()
