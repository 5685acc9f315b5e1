import os, sys, time
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from bayesnetworks_b200 import Context
from bayesnetworks_b200.synth import chain_seeds, make_dag, make_prior, simulate_torch
P, N, MP, chains, iters = 1000, 100000, 8, 64, 100000
dag = make_dag(P, seed=42); g = make_prior(dag, max_par=MP, seed=43); nt = g.node_type_codes()
X = simulate_torch(dag, N, seed=42, device="cuda"); torch.cuda.synchronize()
Xh = torch.empty((P, N), dtype=torch.float64, pin_memory=True); Xh.copy_(X); Xn = Xh.numpy().T
seeds = chain_seeds(chains)
for rep in range(4):
    if rep == 3: os.environ["BN_B200_TIMING"] = "1"
    t0 = time.perf_counter()
    ctx = Context.from_data(Xn, g.source, g.target, nt, max_par=MP)
    t1 = time.perf_counter()
    res, ms = ctx.run(n_chains=chains, n_iter=iters, output=100, rng="wh", seeds=seeds)
    t2 = time.perf_counter()
    ctx.close()
    t3 = time.perf_counter()
    print(f"rep {rep}: create {1e3*(t1-t0):.2f} ms, run {1e3*(t2-t1):.2f} ms (kernel {ms:.2f}), close {1e3*(t3-t2):.2f} ms, total {1e3*(t3-t0):.2f}", flush=True)
