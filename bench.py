#!/usr/bin/env python
"""bench.py -- edge proposals scored/sec and MCMC iters/sec of the structure-MCMC hot path.

    python bench.py --gpus N --steps K --warmup W            (ours; torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K --warmup W

Workload (BASELINE.json configs[3], the configuration the metric is quoted on): synthetic
linear-Gaussian DAG, 1,000 nodes x 100,000 samples, MaxPar 8, 64 chains per GPU (weak
scaling: chains are independent and sharded by global index), 100,000 iterations per chain,
a trace row every 100 iterations.

A "step" is one whole job on that input: sufficient statistics (Gram) + all chains.
  value : job throughput with X already resident in HBM (bn_create_from_device + bn_run),
          timed with CUDA events on the launching stream, max over ranks.
  e2e   : the same job through the host-pointer API (bn_create + bn_run): X starts in pinned
          host memory, H2D inside the timed region, traces copied back to the host.
For N > 1 both timed regions contain the NCCL all-gather of the device-resident traces
(`gather`); e2e then also shards the sample axis of X over the ranks (fixed-order exchange of
partial statistics).  The line also carries `configs` (BASELINE configs 1, 2(i), 3 on one GPU and
config 5 on eight, with parity flags), `strong_64_chains` (N > 1), `e2e.pageable_host` (N = 1)
and `roofline.sm_cycles_per_iteration_per_chain`.
One proposal scored = one iteration that reached checker() (src/network.h:330-336), i.e. one
evaluation of a proposed parent set -- the definition under which the reference's
iterations/s equals its proposals/s (BASELINE.md section 2).

--impl reference times the reference's own CPU implementation (oracle/_ref, the unmodified
sources compiled by oracle/Makefile; else the oracle port) on all host cores, one chain per
core, on a bounded row-subsample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "edge_proposals_scored_per_sec"
UNIT = "proposals/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nodes", type=int, default=1000)
    ap.add_argument("--samples", type=int, default=100000)
    ap.add_argument("--max-par", type=int, default=8)
    ap.add_argument("--chains-per-gpu", type=int, default=64)
    ap.add_argument("--iters", type=int, default=100000)
    ap.add_argument("--output", type=int, default=100)
    ap.add_argument("--ref-rows", type=int, default=1000, help="row subsample of the reference arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernels", action="store_true", help="skip the K1/K2 side measurements")
    ap.add_argument("--no-configs", action="store_true", help="skip the other BASELINE configurations")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling sub-record (N > 1)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned (traces, final graphs, counters) as DIR/<name>.npy")
    return ap.parse_args()


def workload_name(a):
    return (f"synthetic Gaussian DAG {a.nodes} nodes x {a.samples} samples, MaxPar {a.max_par}, "
            f"{a.chains_per_gpu} chains/GPU x {a.iters} iters, output every {a.output}")


# ---------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------
# reference arm (CPU)
# ---------------------------------------------------------------------------
def _ref_worker(job):
    (use_ref, X, src, tgt, nt, max_par, n_iter, output, seeds) = job
    from oracle.oracle import RNG_WH, Oracle, Ref
    t0 = time.perf_counter()
    if use_ref:
        r = Ref().main_fun(X, src, tgt, nt, MaxPar=max_par, N=n_iter, output=output, rng_kind=RNG_WH, seeds=seeds)
        rows = len(r.iter)
    else:
        r = Oracle().mcmc(X, src, tgt, nt, max_par=max_par, n_iter=n_iter, output=output, rng_kind=RNG_WH,
                          seeds=seeds, log_moves=False)
        rows = len(r.iter)
    return time.perf_counter() - t0, rows


def reference_sample(a, cores=None):
    """One step of the reference arm: `cores` independent chains (one process each) on a row
    subsample.  Returns (proposals/s, iters/s, seconds, description dict)."""
    import multiprocessing as mp
    from bayesnetworks_b200.synth import chain_seeds, make_dag, make_prior, simulate_numpy
    from oracle.oracle import have_ref
    cores = cores or os.cpu_count() or 1
    dag = make_dag(a.nodes, seed=42)
    g = make_prior(dag, max_par=a.max_par, seed=43)
    rows = min(a.ref_rows, a.samples)
    X = simulate_numpy(dag, rows, seed=42)
    nt = g.node_type_codes()
    use_ref = have_ref()
    seeds = chain_seeds(cores)
    jobs = [(use_ref, X, g.source, g.target, nt, a.max_par, a.iters, a.output, tuple(int(v) for v in seeds[c]))
            for c in range(cores)]
    t0 = time.perf_counter()
    with mp.get_context("spawn").Pool(cores) as pool:
        res = pool.map(_ref_worker, jobs)
    wall = time.perf_counter() - t0
    # every iteration of the reference that reaches checker() scores one proposal; invalid
    # (cyclic) proposals are <0.2% of iterations, so iterations are counted as proposals here
    total_iters = cores * a.iters
    desc = {"kind": "reference" if use_ref else "port", "cores": cores,
            "sample": (f"{cores} chains (one per core) x {a.iters} iters on {a.nodes} nodes x {rows} of "
                       f"{a.samples} rows (row subsample; the reference's per-proposal cost grows with the "
                       f"row count, so this overstates its full-size throughput), Gram/ctor included")}
    return total_iters / wall, total_iters / wall, wall, desc


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals, secs = [], []
    desc = None
    for i in range(a.warmup + a.steps):
        v, _, wall, desc = reference_sample(a)
        if i >= a.warmup:
            vals.append(v); secs.append(wall)
    value = float(np.mean(vals)) if vals else 0.0
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * float(np.mean(secs)) if secs else None,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": {"workload": workload_name(a), "l2": "n/a (CPU)"},
            "iters_per_sec": value, "gpu_launches": 0,
            "cpu_baseline": dict(desc, value=value, unit=UNIT),
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------
# our arm (GPU)
# ---------------------------------------------------------------------------
def run_ours(a):
    import torch
    import torch.distributed as dist
    from bayesnetworks_b200 import Context, set_default_stream
    from bayesnetworks_b200.dist import (blocks_of_rank, context_row_sharded, row_blocks, run_sharded_device,
                                         shard_chains)
    from bayesnetworks_b200.synth import chain_seeds, make_dag, make_prior, simulate_torch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product has no CPU path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    sharded_stats = world > 1 and 8 % world == 0   # the sample axis has 8 logical row blocks (dist.py)

    n_chains_total = a.chains_per_gpu * world  # weak scaling: fixed work per GPU
    first, count = shard_chains(n_chains_total, world, rank)
    seeds = chain_seeds(count, first_chain=first)
    cap = max(1, (a.iters + a.output - 1) // a.output)

    dag = make_dag(a.nodes, seed=42)
    g = make_prior(dag, max_par=a.max_par, seed=43)
    nt = g.node_type_codes()
    X = simulate_torch(dag, a.samples, seed=42, device=dev)  # (P, N): column-major N x P
    torch.cuda.synchronize()
    x_bytes = X.numel() * 8
    stream = torch.cuda.current_stream().cuda_stream
    set_default_stream(stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    state = {}

    # ---- X resident in HBM ----------------------------------------------------------------
    def step_resident(n_total=n_chains_total, key="res"):
        with Context.from_device(X.data_ptr(), a.samples, a.samples, a.nodes, g.source, g.target, nt,
                                 max_par=a.max_par, device=local_rank) as ctx:
            if world == 1:
                res, ms = ctx.run(n_chains=n_total, n_iter=a.iters, output=a.output, rng="wh",
                                  seeds=chain_seeds(n_total))
                state[key] = dict(valid=sum(r.valid_iters for r in res), alg_bytes=sum(r.alg_bytes for r in res),
                                  rows=sum(len(r.trace["iter"]) for r in res), nonpd=sum(r.n_nonpd for r in res),
                                  changed=[r.trace["ChangedNode"] for r in res], results=res,
                                  cycles=max(r.kernel_cycles for r in res))
            else:
                # chains sharded by global index, traces left in HBM and all-gathered over NCCL (north_star 4)
                out = run_sharded_device(ctx, n_total, a.iters, a.output, rank, world, dev)
                st = out["stats"]
                state[key] = dict(valid=int(st["valid_iters"].sum()) if st is not None else 0,
                                  alg_bytes=int(st["alg_bytes"].sum()) if st is not None else 0,
                                  rows=int(out["n_rows"][out["first"]:out["first"] + out["count"]].sum().item()),
                                  nonpd=int(st["n_nonpd"].sum()) if st is not None else 0, out=out,
                                  cycles=int(st["kernel_cycles"].max()) if st is not None else 0,
                                  gather_ms=out["gather_ms"], gather_ok=out["gather_ok"])
                ms = out["kernel_ms"]
            state[key].update(chain_ms=ms, gram_ms=ctx.gram_ms, launches=ctx.launch_count)

    # ---- end to end: X in pinned host memory, results read back to the host ---------------
    if world == 1 or not sharded_stats:
        Xh = torch.empty((a.nodes, a.samples), dtype=torch.float64, pin_memory=True)
        Xh.copy_(X)
        Xh_np = Xh.numpy().T  # (N, P) Fortran-ordered view of the pinned buffer
        h2d_bytes = x_bytes
    else:
        # every rank holds its share of the 8 logical row blocks of X (column-major rows_b x P each)
        rb = row_blocks(a.samples)
        my_blocks = blocks_of_rank(rank, world)
        Xh_blocks = []
        for b_ in my_blocks:
            lo, cnt = rb[b_]
            hb = torch.empty((a.nodes, cnt), dtype=torch.float64, pin_memory=True)
            hb.copy_(X[:, lo:lo + cnt])
            Xh_blocks.append(hb)
        h2d_bytes = sum(hb.numel() * 8 for hb in Xh_blocks)
    host_out = {}

    def step_e2e():
        if world == 1:
            with Context.from_data(Xh_np, g.source, g.target, nt, max_par=a.max_par, device=local_rank) as ctx:
                res, ms = ctx.run(n_chains=count, n_iter=a.iters, output=a.output, rng="wh", seeds=seeds)
                state["e2e"] = dict(changed=[r.trace["ChangedNode"] for r in res])
            return
        if sharded_stats:
            # H2D of this rank's rows, partial statistics, fixed-order NCCL exchange (bit-identical for any
            # GPU count), context from the device-resident statistics
            blocks = [hb.to(dev, non_blocking=True) for hb in Xh_blocks]
            ctx, _, _, gms = context_row_sharded(blocks, a.samples, a.nodes, g.source, g.target, nt, rank, world, dev,
                                                 max_par=a.max_par)
        else:
            ctx = Context.from_data(Xh_np, g.source, g.target, nt, max_par=a.max_par, device=local_rank)
        with ctx:
            out = run_sharded_device(ctx, n_chains_total, a.iters, a.output, rank, world, dev)
        # the step's result on the host: every chain's trace, on every rank
        for k in ("ints", "gll", "n_rows"):
            if k not in host_out:
                host_out[k] = torch.empty(out[k].shape, dtype=out[k].dtype, pin_memory=True)
            host_out[k].copy_(out[k], non_blocking=True)
        torch.cuda.synchronize()
        state["e2e"] = dict(out=out, gather_ok=out["gather_ok"], gather_ms=out["gather_ms"])

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            t0 = time.perf_counter()
            fn()
            if os.environ.get("BN_BENCH_VERBOSE"):
                print(f"[bench] {fn.__name__}: {1e3 * (time.perf_counter() - t0):.1f} ms", file=sys.stderr)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def reduce_sum_max(sums, maxs):
        t1 = torch.tensor(sums, dtype=torch.float64, device=dev)
        t2 = torch.tensor(maxs, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t1, op=dist.ReduceOp.SUM)
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        return [float(v) for v in t1.tolist()], [float(v) for v in t2.tolist()]

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    total_ms = timed(step_resident, a.steps, a.warmup)
    clocks = sampler.stop() if rank == 0 else None
    e2e_ms = timed(step_e2e, a.steps, max(1, a.warmup // 3))

    # the same end-to-end step from PAGEABLE host memory (what R hands over): the driver stages the copy
    pageable = None
    if world == 1 and not a.no_configs:
        Xp = np.array(Xh_np, order="F", copy=True)   # ordinary (pageable) allocation

        def step_pageable():
            with Context.from_data(Xp, g.source, g.target, nt, max_par=a.max_par, device=local_rank) as ctx:
                ctx.run(n_chains=count, n_iter=a.iters, output=a.output, rng="wh", seeds=seeds)
        pageable = timed(step_pageable, 2, 1) / 2
        del Xp

    # per-step work (identical every step: same seeds)
    r0 = state["res"]
    (proposals, iters, alg_bytes, rows, nonpd), (chain_ms, gram_ms, cycles) = reduce_sum_max(
        [r0["valid"], count * a.iters, r0["alg_bytes"], r0["rows"], r0["nonpd"]],
        [r0["chain_ms"], r0["gram_ms"], r0["cycles"]])
    ms_per_step = total_ms / a.steps
    e2e_ms_per_step = e2e_ms / a.steps
    # parity guard inside the bench: the end-to-end path must give the same trajectories
    if world == 1:
        same = all(np.array_equal(x, y) for x, y in zip(r0["changed"], state["e2e"]["changed"]))
        gather = None
    else:
        o1, o2 = r0["out"], state["e2e"]["out"]
        same = bool(torch.equal(o1["ints"][:, :, 1], o2["ints"][:, :, 1]))   # ChangedNode of every chain
        (_, ), (g1, g2, bad) = reduce_sum_max([0.0], [r0["gather_ms"], state["e2e"]["gather_ms"],
                                                      0.0 if (r0["gather_ok"] and state["e2e"]["gather_ok"] and same) else 1.0])
        gather = {"collective": "ncclAllGather of device-resident trace blocks (7 int32 columns, globalLL, row counts), "
                                "no host staging; every rank ends with every chain's trace",
                  "gather_ok": bad == 0.0, "gather_ms": g1, "gather_ms_e2e": g2,
                  "bytes_per_rank": int(count * cap * 36 + 4 * count)}
        same = bad == 0.0

    # strong scaling as BASELINE config 4 is written: 64 chains IN TOTAL on N GPUs
    strong = None
    if world > 1 and not a.no_strong:
        n_strong = a.chains_per_gpu
        s_ms = timed(lambda: step_resident(n_strong, "strong"), a.steps, max(1, a.warmup // 3)) / a.steps
        (s_prop, ), (s_chain_ms, ) = reduce_sum_max([state["strong"]["valid"]], [state["strong"]["chain_ms"]])
        strong = {"chains_total": n_strong, "chains_per_gpu": n_strong / world, "ms_per_step": s_ms,
                  "value": s_prop / (s_ms * 1e-3), "unit": UNIT, "chain_kernel_ms": s_chain_ms,
                  "note": "a chain is a dependent instruction stream: fewer chains per GPU do not make a chain faster"}

    cfg5 = None
    if world == 8 and not a.no_configs:
        cfg5 = config5(a, dev, rank, world)

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, step_outputs(r0, world))

    peaks = {}
    pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk_path):
        peaks = json.load(open(pk_path))
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    # dominant kernel of the step = the persistent chain kernel (one launch per step per GPU)
    per_gpu_bytes = alg_bytes / world
    achieved = per_gpu_bytes / (chain_ms * 1e-3) / 1e9
    # DRAM bytes of one launch from the committed ncu --set full capture (null if absent)
    traffic = None
    for name in ("r02_chain_traffic.json", "r01_chain_traffic.json"):
        tr_path = os.path.join(ROOT, "profiles", name)
        if os.path.exists(tr_path):
            tr = json.load(open(tr_path))
            traffic = float(tr["dram_bytes_read"]) + float(tr["dram_bytes_write"])
            break
    roofline = {"bound": "hbm", "kernel": "chain_kernel", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                "frac": achieved / hbm_peak, "traffic": traffic, "peak_source": peak_src,
                "kernel_ms": chain_ms, "share_of_step": chain_ms / ms_per_step,
                "sm_cycles_per_iteration_per_chain": cycles / a.iters,
                "note": "latency-bound sequential chains (dependent instruction stream, see "
                        "profiles/r02_chain_kernel.md): algorithmic gather bytes = sum over scored proposals of "
                        "8*(k'+1)(k'+2)/2+8 (SURVEY.md 8d); the Gram (8 MB) is L2 resident, so DRAM traffic "
                        "(`traffic`, bytes per launch, ncu) is far BELOW the algorithmic bytes; the figure that is "
                        "optimised is SM cycles per iteration per chain; the HBM-bound scoring kernel of this "
                        "path is kernels.sweep"}

    line = {"metric": METRIC, "value": proposals / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(a), "chains_total": n_chains_total,
                       "l2": "inputs larger than L2 (X = %.0f MB per GPU, re-read every step)" % (x_bytes / 1e6),
                       "parallelism": (f"chains sharded over {world} GPU(s); " +
                                       ("no collective at N=1" if world == 1 else
                                        "traces all-gathered over NCCL from HBM inside the timed region; e2e also "
                                        "shards the sample axis of X (8 logical row blocks, fixed-order exchange of "
                                        "the partial Gram matrices)"))},
            "iters_per_sec": iters / (ms_per_step * 1e-3),
            "clocks": clocks,
            "e2e": {"value": proposals / (e2e_ms_per_step * 1e-3), "unit": UNIT,
                    "iters_per_sec": iters / (e2e_ms_per_step * 1e-3), "ms_per_step": e2e_ms_per_step,
                    "h2d_bytes_per_step": int(h2d_bytes + 4 * (2 * len(g.source) + a.nodes) + 12 * count),
                    "d2h_bytes_per_step": int((n_chains_total if world > 1 else count) * cap * 36 + 64 * count),
                    "same_trajectories_as_resident_path": bool(same),
                    "pageable_host": (None if pageable is None else
                                      {"ms_per_step": pageable, "value": proposals / (pageable * 1e-3), "unit": UNIT,
                                       "note": "X in ordinary (pageable) host memory, as R owns it"})},
            "gpu_launches": int(r0["launches"]) * a.steps,
            "roofline": roofline,
            "step_breakdown_ms": {"gram_build": gram_ms, "chain_kernel": chain_ms},
            "trace_rows_per_step": rows, "n_nonpd": nonpd}
    if gather is not None:
        line["gather"] = gather
    if strong is not None:
        line["strong_64_chains"] = strong

    if world == 1 and not a.no_configs:
        # every SM busy: the workload's 64 chains light 64 of the 148 SMs (one CTA per chain, the chain is a
        # latency-bound dependent instruction stream); the same run with one chain per SM shows what the GPU
        # sustains on this path.  Reported beside the headline, which stays at BASELINE's 64 chains.
        try:
            n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
            with Context.from_device(X.data_ptr(), a.samples, a.samples, a.nodes, g.source, g.target, nt,
                                     max_par=a.max_par, device=local_rank) as ctx:
                res3, ms3 = ctx.run(n_chains=n_sm, n_iter=a.iters, output=a.output, rng="wh", seeds=chain_seeds(n_sm))
            roofline["one_chain_per_sm"] = {
                "chains": n_sm, "chain_kernel_ms": ms3,
                "proposals_per_sec": sum(r.valid_iters for r in res3) / (ms3 * 1e-3),
                "iters_per_sec": n_sm * a.iters / (ms3 * 1e-3),
                "sm_cycles_per_iteration_per_chain": max(r.kernel_cycles for r in res3) / a.iters,
                "first_64_chains_same_as_headline_run": bool(all(
                    np.array_equal(r.trace["ChangedNode"], c) for r, c in zip(res3[:n_chains_total], state["res"]["changed"])))}
        except Exception as exc:
            roofline["one_chain_per_sm"] = f"failed: {type(exc).__name__}: {exc}"

    if world == 1 and not a.no_configs:
        # the opt-in two-CTA form of the chain kernel (BN_B200_PIPE=1, profiles/r02_two_cta_chain.md) on the same
        # workload, measured in a CHILD process with a time limit (an experimental kernel must not be able to
        # take the headline run with it) and outside every timed region: a reported comparison
        try:
            env = dict(os.environ, BN_B200_PIPE="1", H2D="0", REPS="3", P=str(a.nodes), N=str(a.samples), MP=str(a.max_par),
                       CHAINS=str(n_chains_total), ITERS=str(a.iters), CUDA_VISIBLE_DEVICES=str(local_rank))
            res2 = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "tools", "gpu_perf.py")], capture_output=True,
                                  text=True, timeout=150, env=env)
            import re
            m_ms = re.search(r"kernel ([0-9.]+) ms", res2.stdout)
            m_cy = re.search(r"kernel cycles/iter/chain ([0-9.]+) \(max chain ([0-9.]+)\)", res2.stdout)
            roofline["two_cta_form"] = {
                "chain_kernel_ms": float(m_ms.group(1)), "sm_cycles_per_iteration_per_chain": float(m_cy.group(2)),
                "one_cta_chain_kernel_ms": chain_ms,
                "note": "a cluster of two CTAs per chain (128 SMs busy): rank 1 builds the next window's records while "
                        "rank 0 walks; bit-identical (tests/test_gpu_pipeline.py), opt-in because it is not faster "
                        "(instruction-fetch bound, profiles/r02_two_cta_chain.md)"}
        except Exception as exc:
            roofline["two_cta_form"] = f"not measured: {type(exc).__name__}: {exc}"

    if not a.no_kernels and world == 1:   # (the sweep is timed on the chains' final graphs)
        line["kernels"] = side_kernels(a, X, g, nt, r0.get("results"), local_rank, hbm_peak)
    if not a.no_configs:
        cfgs = {}
        if world == 1:
            try:
                cfgs.update(baseline_configs(local_rank))
            except Exception as exc:  # reported numbers, never a dependency of the headline
                cfgs["error"] = f"{type(exc).__name__}: {exc}"
        if cfg5 is not None:
            cfgs["config5"] = cfg5
        if cfgs:
            line["configs"] = cfgs
    if world == 1 and not a.no_cpu_baseline:
        try:
            v, _, wall, desc = reference_sample(a)
            line["cpu_baseline"] = dict(desc, value=v, unit=UNIT, seconds=wall)
        except Exception as exc:  # the baseline is a reported number, never a dependency
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port",
                                    "sample": f"failed: {exc}"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


TRACE_COLS = ("iter", "ChangedNode", "movetype", "globalLL", "additions", "deletions", "FN", "FP")
COUNTERS = ("uniforms", "valid_iters", "proposed", "reject", "n_nonpd", "total_edges")
DUMP_LIMIT = 64 << 20   # bytes


def step_outputs(r0, world):
    """What one resident step hands its caller, one entry per chain: the trace columns (a list of the chains'
    rows; chains write different numbers of rows) and, on one GPU, the final graphs and chain counters (chains
    on axis 0).  With N > 1 the traces of all chains, which every rank holds after the all-gather."""
    if world > 1:
        from bayesnetworks_b200.dist import INT_COLUMNS
        o = r0["out"]
        n_rows = o["n_rows"].cpu().numpy()
        ints = o["ints"].cpu().numpy()   # [chains, capacity, 7]
        gll = o["gll"].cpu().numpy()
        out = {"n_rows": n_rows, "trace_globalLL": [gll[c, :r] for c, r in enumerate(n_rows)]}
        for i, k in enumerate(INT_COLUMNS):
            out["trace_" + k] = [ints[c, :r, i] for c, r in enumerate(n_rows)]
        return out
    res = r0["results"]
    out = {"n_rows": np.array([len(r.trace["iter"]) for r in res])}
    for k in TRACE_COLS:
        out["trace_" + k] = [r.trace[k] for r in res]
    out["final_parents"] = np.stack([r.final_parents for r in res])
    out["final_npar"] = np.stack([r.final_npar for r in res])
    for k in COUNTERS:
        out[k] = np.array([getattr(r, k) for r in res])
    return out


def dump_outputs(path, arrays):
    """Write `arrays` as path/<name>.npy in float64.  Each value has one entry per chain: an array with chains on
    axis 0, or a list of per-chain rows (trace columns), written end to end in chain order (n_rows.npy splits
    them).  Above DUMP_LIMIT bytes in all, a fixed seeded sample of whole chains is written; chain_index.npy
    says which.  When no single chain fits, the first chain of that sample is written with a seeded sample of
    its trace rows; row_index.npy says which (n_rows.npy keeps the chain's full row count)."""
    n = len(arrays["n_rows"])
    arrays = dict(arrays, chain_index=np.arange(n))
    size = np.zeros(n)
    for v in arrays.values():
        size += [8 * np.size(x) for x in v]
    order = np.random.default_rng(0).permutation(n) if size.sum() > DUMP_LIMIT else np.arange(n)
    idx = np.sort(order[np.cumsum(size[order]) <= DUMP_LIMIT])
    if n and not len(idx):
        c = int(order[0])
        cols = [k for k, v in arrays.items() if isinstance(v, list)]
        n_r = len(arrays[cols[0]][c])
        fixed = size[c] - 8 * len(cols) * n_r   # bytes of the chain outside its trace rows
        keep = min(n_r, max(0, int(DUMP_LIMIT - fixed) // (8 * (len(cols) + 1))))   # (+ row_index)
        rows = np.sort(np.random.default_rng(0).choice(n_r, keep, replace=False))
        arrays.update({k: {c: np.asarray(arrays[k][c])[rows]} for k in cols}, row_index={c: rows})
        idx = np.array([c])
    os.makedirs(path, exist_ok=True)
    for name, v in arrays.items():
        if isinstance(v, (list, dict)):   # per-chain rows (a dict: only the sampled chain's)
            out = np.concatenate([np.zeros(0)] + [np.ravel(v[i]) for i in idx])
        else:
            out = np.asarray(v)[idx]
        np.save(os.path.join(path, name + ".npy"), out.astype(np.float64))


def config5(a, dev, rank, world):
    """BASELINE config 5 (Gram-build stress, 8 GPUs): 5,000 nodes x 1,000,000 samples (X = 40 GB FP64), the
    sample axis sharded over the GPUs in 8 logical row blocks (generated on the device that owns them),
    512 chains x 20,000 iterations sharded over the GPUs."""
    import torch
    import torch.distributed as dist
    from bayesnetworks_b200.dist import blocks_of_rank, context_row_sharded, row_blocks, run_sharded_device
    from bayesnetworks_b200.synth import make_dag, make_prior, simulate_torch
    P, N, chains, iters, MP = 5000, 1000000, 512, 20000, 8
    try:
        dag = make_dag(P, seed=42)
        g = make_prior(dag, max_par=MP, seed=43)
        nt = g.node_type_codes()
        rb = row_blocks(N)
        mine = [simulate_torch(dag, rb[b][1], seed=42 + b, device=dev) for b in blocks_of_rank(rank, world)]
        times = []
        ctx = None
        for rep in range(3):
            dist.barrier(); torch.cuda.synchronize(); t0 = time.perf_counter()
            ctx, mean, gram, kms = context_row_sharded(mine, N, P, g.source, g.target, nt, rank, world, dev, max_par=MP)
            dist.barrier(); torch.cuda.synchronize()
            times.append((time.perf_counter() - t0, kms))
            if rep < 2:
                ctx.close()
        wall, kms = min(times)
        dist.barrier(); torch.cuda.synchronize(); t0 = time.perf_counter()
        out = run_sharded_device(ctx, chains, iters, 100, rank, world, dev)
        dist.barrier(); torch.cuda.synchronize()
        cwall = time.perf_counter() - t0
        ctx.close()
        v = torch.tensor([float(out["stats"]["valid_iters"].sum()), 1.0 if out["gather_ok"] else 0.0],
                         dtype=torch.float64, device=dev)
        dist.all_reduce(v[:1], op=dist.ReduceOp.SUM)
        ok = v[1:].clone(); dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        del mine
        torch.cuda.empty_cache()
        return {"workload": f"{P} nodes x {N} samples (X = 40 GB FP64), {chains} chains x {iters} iters, 8 GPUs",
                "gram_wall_ms_incl_exchange": 1e3 * wall, "gram_kernel_ms_per_gpu": kms,
                "gram_tflops_full_count_boxwide": 2.0 * N * P * P / wall / 1e12,
                "chains_wall_ms_incl_gather": 1e3 * cwall, "gather_ms": out["gather_ms"], "gather_ok": bool(ok.item() == 1.0),
                "proposals_per_sec": float(v[0].item()) / cwall, "iters_per_sec": chains * iters / cwall}
    except Exception as exc:
        return {"error": f"{type(exc).__name__}: {exc}"}


def baseline_configs(local_rank):
    """The other BASELINE.json configurations on one GPU, each with its parity flag against the golden
    fixture (tests/golden, generated from the compiled reference) where one exists."""
    from bayesnetworks_b200 import Context, main_fun
    from bayesnetworks_b200.synth import make_dag, make_prior, simulate_numpy
    out = {}
    gold_dir = os.path.join(ROOT, "tests", "golden")
    z = np.load(os.path.join(gold_dir, "network_p3sim8.npz"))
    gold = np.load(os.path.join(gold_dir, "golden_ref.npz"))
    X, src, tgt, nt = z["X"], z["source"], z["target"], z["node_type"]
    labels = np.arange(X.shape[1], dtype=np.int32)
    int_cols = ("iter", "ChangedNode", "movetype", "additions", "deletions", "FN", "FP")

    def shipped(max_par, rng, seed, name):
        best, r = 1e30, None
        for _ in range(3):   # one call = bn_main_fun: context + Gram + chain + copies (the R drop-in call)
            t0 = time.perf_counter()
            r = main_fun(X, src, tgt, labels, nt, MaxPar=max_par, N=50000, output=100, rng=rng, seed=seed)
            best = min(best, time.perf_counter() - t0)
        ok = all(np.array_equal(r[k], gold[f"{name}_{k}"]) for k in int_cols)
        ok = ok and bool(np.allclose(r["globalLL"], gold[f"{name}_globalLL"], rtol=1e-9, atol=1e-9 * 1000))
        return {"call_ms": 1e3 * best, "iters_per_sec": 50000 / best, "rows": int(len(r["iter"])),
                "bit_identical_trace_vs_reference": bool(ok)}

    out["config1"] = {"workload": "shipped `network` dataset (81 nodes x 2,000 samples), bn_mcmc(N=50000), "
                                  "set.seed(1234), 1 chain, one bn_main_fun call (context + Gram + chain + copies)",
                      "maxpar50": shipped(50, "rmt", 1234, "cfg1"), "maxpar8": shipped(8, "rmt", 1234, "cfg1")}
    out["config2_wichmann_hill"] = {"workload": "same data, Wichmann-Hill reference seeds (Bayes-networks/random4f.h)",
                                    "maxpar50": shipped(50, "wh", None, "cfg2")}
    # first call of a cold process (CUDA context, module load)
    try:
        code = ("import time,sys,json,numpy as np;sys.path.insert(0,%r);"
                "z=np.load(%r);from bayesnetworks_b200 import main_fun;t0=time.perf_counter();"
                "r=main_fun(z['X'],z['source'],z['target'],np.arange(81,dtype=np.int32),z['node_type'],MaxPar=50,N=50000,"
                "output=100,rng='rmt',seed=1234);t1=time.perf_counter();"
                "r=main_fun(z['X'],z['source'],z['target'],np.arange(81,dtype=np.int32),z['node_type'],MaxPar=50,N=50000,"
                "output=100,rng='rmt',seed=1234);t2=time.perf_counter();print(json.dumps([t1-t0,t2-t1]))"
                % (ROOT, os.path.join(gold_dir, "network_p3sim8.npz")))
        env = dict(os.environ, CUDA_VISIBLE_DEVICES=str(local_rank))
        res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120, env=env)
        first, second = json.loads(res.stdout.strip().splitlines()[-1])
        out["config1"]["cold_process_first_call_ms"] = 1e3 * first
        out["config1"]["cold_process_second_call_ms"] = 1e3 * second
    except Exception as exc:
        out["config1"]["cold_process_first_call_ms"] = f"failed: {exc}"
    # config 3: synthetic 100 nodes x 10,000 samples, one chain, 1e6 iterations
    dag = make_dag(100, seed=42)
    X3 = simulate_numpy(dag, 10000, seed=42)
    c3 = {"workload": "synthetic Gaussian DAG 100 nodes x 10,000 samples, 1 chain x 1,000,000 iterations"}
    for mp in (8, 50):
        g3 = make_prior(dag, max_par=mp, seed=43)
        with Context.from_data(X3, g3.source, g3.target, g3.node_type_codes(), max_par=mp, device=local_rank) as ctx:
            ctx.run(n_chains=1, n_iter=1000, output=100)
            res, ms = ctx.run(n_chains=1, n_iter=1000000, output=100, rng="wh")
            r = res[0]
            c3[f"maxpar{mp}"] = {"chain_kernel_ms": ms, "iters_per_sec": 1e6 / (ms * 1e-3),
                                 "proposals_per_sec": r.valid_iters / (ms * 1e-3), "n_nonpd": r.n_nonpd,
                                 "largest_parent_set": int(r.final_npar.max()),
                                 "sm_cycles_per_iteration": r.kernel_cycles / 1e6}
    c3["maxpar50_over_maxpar8"] = c3["maxpar50"]["chain_kernel_ms"] / c3["maxpar8"]["chain_kernel_ms"]
    out["config3"] = c3
    return out


def side_kernels(a, X, g, nt, res, local_rank, hbm_peak):
    """K1 (Gram, FP64 tensor pipe) and K2 (all-proposal sweep) timed alone, plus the in-run
    cuBLAS DGEMM figure that stands in for the FP64 peak (MEASURED_PEAKS.json has none)."""
    import torch
    from bayesnetworks_b200 import Context
    out = {}
    P, N = a.nodes, a.samples
    # cuBLAS DGEMM (library call: denominator only, not on the product path)
    n = 8192
    A = torch.randn((n, n), dtype=torch.float64, device=X.device)
    B = torch.randn((n, n), dtype=torch.float64, device=X.device)
    for _ in range(2):
        torch.matmul(A, B)
    torch.cuda.synchronize()
    best = 1e30
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(A, B); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    dgemm_tf = 2.0 * n ** 3 / (best * 1e-3) / 1e12
    del A, B
    gram_ms = []
    with Context.from_device(X.data_ptr(), N, N, P, g.source, g.target, nt, max_par=a.max_par,
                             device=local_rank) as ctx:
        gram_ms.append(ctx.gram_ms)
        # K2: sweep over the chains' final graphs
        G = len(res)
        par = np.stack([r.final_parents for r in res]).astype(np.int32)
        npar = np.stack([r.final_npar for r in res]).astype(np.int32)
        d_par = torch.from_numpy(par).to(X.device)
        d_np = torch.from_numpy(npar).to(X.device)
        d_base = torch.empty((G, P), dtype=torch.float64, device=X.device)
        d_score = torch.empty((G, P, P), dtype=torch.float64, device=X.device)
        d_hr = torch.empty((G, P, P), dtype=torch.float64, device=X.device)
        ms = [ctx.score_all_proposals_device(G, d_par.data_ptr(), d_np.data_ptr(), d_base.data_ptr(),
                                             d_score.data_ptr(), d_hr.data_ptr()) for _ in range(6)][1:]
        sweep_ms = float(np.mean(ms))
        score = d_score.cpu().numpy()
        scored = int(np.isfinite(score).sum())
        kk = npar.astype(np.int64)
        # algorithmic bytes: adds score k+1 parents, deletes k-1 (8*(k'+1)(k'+2)/2 + 8 each)
        is_par = np.zeros((G, P, P), bool)
        for gi in range(G):
            for c in range(P):
                is_par[gi, c, par[gi, c, :npar[gi, c]]] = True
        kprime = np.where(is_par, kk[:, :, None] - 1, kk[:, :, None] + 1)
        alg = float(np.where(np.isfinite(score), 4 * (kprime + 1) * (kprime + 2) + 8, 0).sum())
        out["sweep"] = {"ms": sweep_ms, "graphs": G, "proposals_scored": scored,
                        "proposals_per_sec": scored / (sweep_ms * 1e-3),
                        "roofline": {"bound": "hbm", "achieved": alg / (sweep_ms * 1e-3) / 1e9, "peak": hbm_peak,
                                     "unit": "GB/s", "frac": alg / (sweep_ms * 1e-3) / 1e9 / hbm_peak,
                                     "min_traffic_GBps": (scored * 8.0 * 2 + G * P * 8.0) / (sweep_ms * 1e-3) / 1e9,
                                     "note": "achieved = algorithmic per-proposal gather bytes (SURVEY.md 8d); the "
                                             "kernel shares one factorisation per child, so its real traffic is the "
                                             "two output tables (min_traffic_GBps)"}}
    for _ in range(3):
        with Context.from_device(X.data_ptr(), N, N, P, g.source, g.target, nt, max_par=a.max_par,
                                 device=local_rank) as ctx:
            gram_ms.append(ctx.gram_ms)
    gm = float(np.min(gram_ms[1:]))
    tiles = (P + 127) // 128
    executed = tiles * (tiles + 1) / 2 * 128 * 128 * 2.0 * N
    out["gram"] = {"ms": gm, "tflops_full_count": 2.0 * N * P * P / (gm * 1e-3) / 1e12,
                   "tflops_executed": executed / (gm * 1e-3) / 1e12, "dgemm_cublas_tflops": dgemm_tf,
                   "roofline": {"bound": "tensor", "achieved": executed / (gm * 1e-3) / 1e12, "peak": dgemm_tf,
                                "unit": "TFLOP/s", "frac": executed / (gm * 1e-3) / 1e12 / dgemm_tf,
                                "note": "FP64 DMMA; peak = cuBLAS DGEMM 8192^3 measured in this run (no FP64 figure "
                                        "in MEASURED_PEAKS.json); ms covers means+centring+DMMA+reduce"}}
    return out


def main():
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
