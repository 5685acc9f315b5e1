"""Posterior summary of a run: the legacy program's ``Summarize()`` (Bayes-networks/main.cpp:299-339).

The tallies come from the device (``bn_run_args.edge_freq`` / ``npar_freq`` = ``freqEdge`` /
``freqNpar`` of ``Tabulate()``, main.cpp:289-297; ``bn_chain_stats.proposed`` / ``reject`` =
``ProposedMoves`` / ``reject``); this module only turns them into the reference's report --
the two text blocks it writes to ``networks-summary.txt`` and ``networks-edges.txt``, byte for
byte in the reference's layout -- and into posterior probabilities.
"""
from __future__ import annotations

import numpy as np


def _ratio(num: int, den: int) -> str:
    """printf("%6.3f", double(num) / den) as glibc prints it (0 / 0 is "-nan" on x86-64)."""
    if den == 0:
        return "  -nan" if num == 0 else ("   inf" if num > 0 else "  -inf")
    return "%6.3f" % (num / den)


def summarize(proposed, reject, npar_freq, edge_freq, prior_source, prior_target, final_parents, final_npar,
              max_par: int, n_counted: int | None = None) -> dict:
    """``proposed`` / ``reject``: 3 counters each (invalid, addition, deletion); ``npar_freq``
    [P, >= max_par] and ``edge_freq`` [child, parent] as ``ChainResult`` holds them;
    ``prior_source`` / ``prior_target``: the supplied graph, 1-based (simEdge, Nsimpar);
    ``final_parents`` / ``final_npar``: the last graph (for the reversal list).
    Returns ``summary_text`` and ``edges_text`` (main.cpp:300-338), and -- when ``n_counted``
    (iterations tabulated, i.e. N - drop) is given -- ``edge_posterior`` [child, parent] and
    ``npar_posterior`` [P, k]."""
    npar_freq = np.asarray(npar_freq)
    edge_freq = np.asarray(edge_freq)
    P = edge_freq.shape[0]
    sim = np.zeros((P, P), dtype=np.int64)      # [child, parent]
    nsim = np.zeros(P, dtype=np.int64)
    for s_, t_ in zip(prior_source, prior_target):
        sim[t_ - 1, s_ - 1] = 1
        nsim[t_ - 1] += 1
    out = ["\n\nNumber of proposals accepted \n"]
    for typ, name in ((0, "invalid  "), (1, "addition "), (2, "deletion ")):
        acc = int(proposed[typ]) - int(reject[typ])
        out.append(name + "%5d / %5d %s\n" % (acc, int(proposed[typ]), _ratio(acc, int(proposed[typ]))))
    out.append("\n\nFrequency distribution of number of parents fo each node")
    out.append("\n  Npar:" + "".join("%4d  " % e for e in range(max_par)))
    for p in range(P):
        out.append("\n%4d  " % p)
        for e in range(max_par):
            out.append(" %4d" % int(npar_freq[p, e]) + ("*" if e == nsim[p] else " "))
    out.append("\n\nReversals of direction")
    fp, fn = np.asarray(final_parents), np.asarray(final_npar)
    for p1 in range(P):
        for e1 in range(int(fn[p1])):
            for p2 in range(p1 + 1, P):
                for e2 in range(int(fn[p2])):
                    if fp[p1, e1] == p2 and fp[p2, e2] == p1:
                        out.append("\n%2d -> %2d  %d %4d  <===>   %2d -> %2d  %d %4d" % (
                            p2, p1, sim[p1, p2], int(edge_freq[p1, p2]), p1, p2, sim[p2, p1], int(edge_freq[p2, p1])))
    edges = ["\n\nFrequency distribution of edges\n p    par   freq simulated?"]
    for p in range(P):
        for e in range(P):
            if edge_freq[p, e] or sim[p, e]:
                edges.append("\n%2d -> %2d  %6d    %d" % (e, p, int(edge_freq[p, e]), int(sim[p, e])))
    res = {"summary_text": "".join(out), "edges_text": "".join(edges)}
    if n_counted:
        res["edge_posterior"] = edge_freq / float(n_counted)
        res["npar_posterior"] = npar_freq / float(n_counted)
    return res


def summarize_result(result, graph, max_par: int, n_iter: int, drop: int = 0) -> dict:
    """``summarize`` for a :class:`~bayesnetworks_b200.api.ChainResult` run with ``tabulate=True``."""
    return summarize(result.proposed, result.reject, result.npar_freq, result.edge_freq, graph.source, graph.target,
                     result.final_parents, result.final_npar, max_par, n_counted=max(n_iter - drop, 0))


def ancestor_posterior(results) -> np.ndarray:
    """Posterior probability of a directed path, [descendant, ancestor], pooled over chains.

    ``results``: :class:`~bayesnetworks_b200.api.ChainResult` objects run with ``tabulate_ancestors=True``,
    or their ``anc_freq`` arrays (segments of resumed runs may be listed alongside: counts add up).  The
    counts are summed in int64 and each row is divided by the pooled diagonal, the number of tabulated
    iterations; entry [d, a] is the share of them in which a is an ancestor of d (the diagonal is 1).
    Rows without tabulated iterations are NaN."""
    arrs = [np.asarray(getattr(r, "anc_freq", r)) for r in results]
    if not arrs or any(a is None or a.ndim != 2 or a.shape[0] != a.shape[1] for a in arrs):
        raise ValueError("ancestor_posterior needs [P, P] anc_freq arrays (run with tabulate_ancestors=True)")
    total = np.zeros(arrs[0].shape, dtype=np.int64)
    for a in arrs:
        total += a
    n = np.diagonal(total).astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        return total / n[:, None]


def best_graph(results):
    """The best graph over chains of one run, or over the segments of a resumed chain listed in order.

    ``results``: :class:`~bayesnetworks_b200.api.ChainResult` objects run with ``track_best=True``, or their
    :class:`~bayesnetworks_b200.api.BestGraph`.  Returns the first of the highest ``log_post``, skipping those
    with ``found`` False; None when none was found.  Over the segments of a resumed run this is the
    uninterrupted run's best: a graph held across a boundary is a candidate in both segments, and the earlier
    one wins the tie."""
    best = None
    for r in results:
        b = getattr(r, "best", r)
        if b is None or not hasattr(b, "log_post"):
            raise ValueError("best_graph needs BestGraph objects (run with track_best=True)")
        if b.found and (best is None or b.log_post > best.log_post):
            best = b
    return best
