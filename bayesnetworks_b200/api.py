"""Host-side mirror of the reference's operator interface for the hot path.

* :func:`bn_mcmc`  -- ``R/bn_mcmc.R:8-25``  (same arguments and defaults)
* :func:`main_fun` -- ``src/bayesnet_mcmc.cpp:27-38`` (same arguments and defaults;
  result columns ``iter, ChangedNode, movetype, globalLL, additions, deletions, FN, FP``
  as in ``network::result``, ``src/network.h:353-364``)
* :class:`Context` -- the C ABI of ``include/bn_b200.h`` one level up: sufficient
  statistics once per dataset, then scoring / chains on the device.

Every compute call goes through ``libbn_b200.so``; there is no CPU path here.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np

from . import _lib
from ._lib import BN_RNG_REPLAY, BN_RNG_RMT, BN_RNG_WH, BnError, as_i32, check, ptr
from .network import Network

TRACE_COLUMNS = ("iter", "ChangedNode", "movetype", "globalLL", "additions", "deletions", "FN", "FP")
_RNG_KINDS = {"wh": BN_RNG_WH, "rmt": BN_RNG_RMT, "replay": BN_RNG_REPLAY,
              BN_RNG_WH: BN_RNG_WH, BN_RNG_RMT: BN_RNG_RMT, BN_RNG_REPLAY: BN_RNG_REPLAY}


@dataclass
class ChainResult:
    """One chain: the eight trace columns plus counters and the final graph."""
    trace: dict
    uniforms: int
    valid_iters: int
    proposed: tuple
    reject: tuple
    n_nonpd: int
    total_edges: int
    windows: int
    alg_bytes: int
    phase_cycles: tuple
    slots_simulated: int
    final_parents: np.ndarray   # [P, max_par], -1 padded, per-child list order
    final_npar: np.ndarray
    accepted_moves: Optional[np.ndarray] = None  # rows (iter, movetype, child, parent)
    edge_freq: Optional[np.ndarray] = None       # [child, parent] counts (posterior tabulation)
    npar_freq: Optional[np.ndarray] = None       # [node, k] iterations spent with k parents
    kernel_cycles: int = 0                       # SM cycles of the chain, first to last iteration
    mt_state: Optional[np.ndarray] = None        # R-MT stream state after the run (.Random.seed[2:626])
    state: Optional["ChainState"] = None         # run(want_state=True): where the chain continues from
    anc_freq: Optional[np.ndarray] = None        # [descendant, ancestor] counts of directed paths (tabulate_ancestors)
    best: Optional["BestGraph"] = None           # run(track_best=True): the best graph the chain visited
    mb_freq: Optional[np.ndarray] = None         # [P, P] symmetric counts of Markov blanket pairs (tabulate_markov_blankets)

    def edges(self):
        """(parent, child) pairs, 0-based, per-child list order."""
        return [(int(self.final_parents[c, e]), c)
                for c in range(len(self.final_npar)) for e in range(int(self.final_npar[c]))]


@dataclass
class BestGraph:
    """The graph with the highest log posterior ``log_lik + log_prior`` among the graphs a chain held in
    the iterations ``edge_freq`` counts (``Context.run(track_best=True)``; bn_best_graph of the C ABI).
    ``log_lik`` is its globalLL, ``log_prior`` the chain's LogPrior of it; ``iter`` the first tabulated
    iteration after which the chain held it.  ``found`` is False when the call tabulated no iteration:
    the lists are then -1 / 0, the scores -inf and ``iter`` -1."""
    parents: np.ndarray   # [P, max_par] int32, -1 padded, list order
    npar: np.ndarray      # [P] int32
    log_post: float
    log_lik: float
    log_prior: float
    iter: int
    found: bool

    def edges(self):
        """(parent, child) pairs, 0-based, per-child list order."""
        return [(int(self.parents[c, e]), c) for c in range(len(self.npar)) for e in range(int(self.npar[c]))]

    def as_start(self) -> "ChainState":
        """A fresh chain from this graph (``Context.run(start=[...])``)."""
        return ChainState.from_graph(self.parents, self.npar)


_STATE_SCALARS = ("iter", "valid", "total_edges_member", "additions", "deletions", "uniforms")


@dataclass
class ChainState:
    """Where a chain continues from: its ordered parent lists, the scalars of ``bn_chain_state``, its
    uniform stream and, optionally, its score block (per-node scores, and for max_par > 8 the per-node
    Cholesky factors).  ``Context.run(start=[...])`` continues each chain with ``n_iter`` more iterations;
    a run split into segments this way computes the same bits as the uninterrupted run.

    A state made by :meth:`from_graph` / :meth:`from_edges` is a fresh chain from that graph (iteration 0,
    the stream from the run's seeds); ``rng`` and ``n_samples`` are then None.  A state returned by a run
    (``ChainResult.state``) is a resume and only fits a run with the same node count, max_par, sample
    count and stream kind."""
    parents: np.ndarray                      # [P, max_par] int32, -1 padded, list order
    npar: np.ndarray                         # [P] int32
    n_samples: Optional[int] = None
    rng: Optional[int] = None                # BN_RNG_* of the stream to continue; None = fresh start
    iter: int = 0                            # next iteration index
    valid: int = 1                           # the stale `valid` flag
    total_edges_member: int = 0              # TotalEdges as the last LogPrior() left it
    additions: int = 0                       # accepted moves since `drop` (trace columns)
    deletions: int = 0
    uniforms: int = 0                        # uniforms consumed since iteration 0
    wh_state: Optional[np.ndarray] = None    # rng WH: the stream state (a seed triple)
    mt_state: Optional[np.ndarray] = None    # rng RMT: .Random.seed[2:626] after the consumed uniforms
    score_block: Optional[np.ndarray] = None  # float64 [Context.score_state_len]

    @property
    def P(self) -> int:
        return int(self.npar.shape[0])

    @property
    def max_par(self) -> int:
        return int(self.parents.shape[1])

    @property
    def resumed(self) -> bool:
        return self.rng is not None

    @classmethod
    def from_graph(cls, parents, npar) -> "ChainState":
        """A fresh chain from ordered parent lists ([P, max_par], -1 padded) and their lengths."""
        parents, npar = as_i32(parents), as_i32(npar)
        if parents.ndim != 2 or npar.shape != (parents.shape[0],):
            raise ValueError("parents must be (P, max_par) and npar (P,)")
        return cls(parents=parents.copy(), npar=npar.copy())

    @classmethod
    def from_edges(cls, edges, n_nodes: int, max_par: int) -> "ChainState":
        """A fresh chain from 0-based (parent, child) pairs; each child's parents keep the pairs' order."""
        parents = np.full((n_nodes, max_par), -1, dtype=np.int32)
        npar = np.zeros(n_nodes, dtype=np.int32)
        for j, c in edges:
            if npar[c] >= max_par:
                raise ValueError(f"node {c} has more than max_par = {max_par} parents")
            parents[c, npar[c]] = j
            npar[c] += 1
        return cls(parents=parents, npar=npar)

    def save(self, path) -> None:
        """Write the state as .npz (a checkpoint that outlives the process)."""
        d = {"parents": self.parents, "npar": self.npar}
        for k in _STATE_SCALARS:
            d[k] = np.int64(getattr(self, k))
        for k in ("n_samples", "rng"):
            if getattr(self, k) is not None:
                d[k] = np.int64(getattr(self, k))
        for k in ("wh_state", "mt_state", "score_block"):
            if getattr(self, k) is not None:
                d[k] = getattr(self, k)
        np.savez(path, **d)

    @classmethod
    def load(cls, path) -> "ChainState":
        with np.load(path) as z:
            kw = {k: int(z[k]) for k in _STATE_SCALARS}
            for k in ("n_samples", "rng"):
                kw[k] = int(z[k]) if k in z else None
            for k in ("wh_state", "mt_state", "score_block"):
                kw[k] = z[k].copy() if k in z else None
            return cls(parents=z["parents"].copy(), npar=z["npar"].copy(), **kw)


def _bad_arg(msg):
    return BnError(_lib.BN_ERR_BAD_ARG, msg)


def _i32_bits(a) -> np.ndarray:
    """Integers as 32-bit patterns (R stores the Mersenne-Twister words as signed ints)."""
    return np.ascontiguousarray((np.asarray(a).astype(np.int64) & 0xFFFFFFFF).astype(np.uint32).view(np.int32))


def set_default_stream(cuda_stream: Optional[int]) -> None:
    """Contexts created afterwards by this thread launch on ``cuda_stream`` (a raw
    ``cudaStream_t`` value, e.g. ``torch.cuda.current_stream().cuda_stream``); None resets."""
    check(_lib.lib().bn_set_default_stream(C.c_void_p(cuda_stream or 0)))


class Context:
    """Device-resident sufficient statistics + prior graph (``bn_ctx``)."""

    def __init__(self, handle, n_samples, n_nodes, max_par):
        self._h = handle
        self.n_samples, self.n_nodes, self.max_par = n_samples, n_nodes, max_par

    # -- constructors --------------------------------------------------------
    @staticmethod
    def _graph_args(graph_source, graph_target, graph_node_type, n_nodes):
        src, tgt = as_i32(graph_source), as_i32(graph_target)
        if src.shape != tgt.shape:
            raise ValueError("graph_source and graph_target must have the same length")
        nt = as_i32(graph_node_type)
        if nt.shape != (n_nodes,):
            raise ValueError("graph_node_type must have one entry per column of X")
        return src, tgt, nt

    @classmethod
    def from_data(cls, X, graph_source, graph_target, graph_node_type, max_par=50, phi=1.0,
                  omega=6.9, device=0):
        """``X``: (n_samples, n_nodes) float64; stored column-major like R's matrix."""
        Xf = np.asfortranarray(np.asarray(X, dtype=np.float64))
        n, p = Xf.shape
        src, tgt, nt = cls._graph_args(graph_source, graph_target, graph_node_type, p)
        h = C.c_void_p()
        check(_lib.lib().bn_create(ptr(Xf), n, p, ptr(src), ptr(tgt), len(src), ptr(nt), int(max_par),
                                   float(phi), float(omega), int(device), C.byref(h)))
        return cls(h, n, p, int(max_par))

    @classmethod
    def from_device(cls, data_ptr, ld, n_samples, n_nodes, graph_source, graph_target,
                    graph_node_type, max_par=50, phi=1.0, omega=6.9, device=0):
        """X already in HBM (column-major, leading dimension ``ld``), e.g. ``tensor.data_ptr()``."""
        src, tgt, nt = cls._graph_args(graph_source, graph_target, graph_node_type, n_nodes)
        h = C.c_void_p()
        check(_lib.lib().bn_create_from_device(C.c_void_p(int(data_ptr)), int(ld), int(n_samples),
                                               int(n_nodes), ptr(src), ptr(tgt), len(src), ptr(nt),
                                               int(max_par), float(phi), float(omega), int(device),
                                               C.byref(h)))
        return cls(h, int(n_samples), int(n_nodes), int(max_par))

    @classmethod
    def from_stats(cls, n_samples, mean, centered_gram, graph_source, graph_target,
                   graph_node_type, max_par=50, phi=1.0, omega=6.9, device=0):
        mean = np.ascontiguousarray(mean, dtype=np.float64)
        cg = np.ascontiguousarray(centered_gram, dtype=np.float64)
        p = mean.shape[0]
        if cg.shape != (p, p):
            raise ValueError("centered_gram must be (n_nodes, n_nodes)")
        src, tgt, nt = cls._graph_args(graph_source, graph_target, graph_node_type, p)
        h = C.c_void_p()
        check(_lib.lib().bn_create_from_stats(int(n_samples), p, ptr(mean), ptr(cg), ptr(src), ptr(tgt),
                                              len(src), ptr(nt), int(max_par), float(phi),
                                              float(omega), int(device), C.byref(h)))
        return cls(h, int(n_samples), p, int(max_par))

    @classmethod
    def from_stats_device(cls, n_samples, n_nodes, d_mean, d_centered_gram, graph_source, graph_target,
                          graph_node_type, max_par=50, phi=1.0, omega=6.9, device=0):
        """Sufficient statistics already in HBM (device pointers): the row-sharded Gram path."""
        src, tgt, nt = cls._graph_args(graph_source, graph_target, graph_node_type, n_nodes)
        h = C.c_void_p()
        check(_lib.lib().bn_create_from_stats_device(int(n_samples), int(n_nodes), C.c_void_p(int(d_mean)),
                                                     C.c_void_p(int(d_centered_gram)), ptr(src), ptr(tgt),
                                                     len(src), ptr(nt), int(max_par), float(phi), float(omega),
                                                     int(device), C.byref(h)))
        return cls(h, int(n_samples), int(n_nodes), int(max_par))

    def close(self):
        if self._h is not None and self._h.value:
            _lib.lib().bn_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- introspection -------------------------------------------------------
    def set_stream(self, cuda_stream: Optional[int]):
        check(_lib.lib().bn_set_stream(self._h, C.c_void_p(cuda_stream or 0)))

    @property
    def gram_ms(self) -> float:
        ms = C.c_float(0)
        check(_lib.lib().bn_get_gram_ms(self._h, C.byref(ms)))
        return float(ms.value)

    @property
    def launch_count(self) -> int:
        return int(_lib.lib().bn_get_launch_count(self._h))

    def stats(self):
        """(sumX, sumXX, mean, centered): ``src/network.h:124-136`` + the centred form used here."""
        p = self.n_nodes
        sum_x, mean = np.empty(p), np.empty(p)
        sum_xx = np.empty((p, p), order="F")
        centered = np.empty((p, p))
        check(_lib.lib().bn_get_stats(self._h, ptr(sum_x), ptr(sum_xx), ptr(mean), ptr(centered)))
        return sum_x, np.ascontiguousarray(sum_xx), mean, centered

    # -- scoring -------------------------------------------------------------
    def score_nodes(self, child, parents, n_par):
        """``network::score`` for explicit (child, ordered parent list) items."""
        child, n_par = as_i32(child), as_i32(n_par)
        parents = as_i32(parents)
        n = child.shape[0]
        if parents.shape != (n, self.max_par):
            raise ValueError(f"parents must be ({n}, {self.max_par})")
        out = np.empty(n)
        check(_lib.lib().bn_score_nodes(self._h, n, ptr(child), ptr(parents), ptr(n_par), ptr(out)))
        return out

    def score_all_proposals(self, parents, n_par, want_score=True, want_log_hr=True):
        """Every add/delete proposal of each DAG; returns (base, score, log_hr)."""
        parents, n_par = as_i32(parents), as_i32(n_par)
        if parents.ndim == 2:
            parents, n_par = parents[None], n_par[None]
        g, p = n_par.shape
        if parents.shape != (g, p, self.max_par) or p != self.n_nodes:
            raise ValueError("parents must be (n_graphs, n_nodes, max_par)")
        base = np.empty((g, p))
        score = np.empty((g, p, p)) if want_score else None
        hr = np.empty((g, p, p)) if want_log_hr else None
        check(_lib.lib().bn_score_all_proposals(self._h, g, ptr(parents), ptr(n_par), ptr(base),
                                                ptr(score), ptr(hr)))
        return base, score, hr

    def score_all_proposals_device(self, n_graphs, d_parents, d_npar, d_base, d_score, d_log_hr):
        """Device-pointer variant; returns the device time of the launch in ms."""
        ms = C.c_float(0)
        check(_lib.lib().bn_score_all_proposals_device(
            self._h, int(n_graphs), C.c_void_p(d_parents), C.c_void_p(d_npar), C.c_void_p(d_base or 0),
            C.c_void_p(d_score or 0), C.c_void_p(d_log_hr or 0), C.byref(ms)))
        return float(ms.value)

    # -- chains --------------------------------------------------------------
    @property
    def score_state_len(self) -> int:
        """Per-chain length (doubles) of ``ChainState.score_block``."""
        n = C.c_int64(0)
        check(_lib.lib().bn_score_state_len(self._h, C.byref(n)))
        return int(n.value)

    def _start_args(self, start, n_chains, kind, args, keep):
        """bn_run_args.start_parents / state_in / score_state_in / mt_state_in from ChainStates."""
        p, mp = self.n_nodes, self.max_par
        if len(start) != n_chains:
            raise _bad_arg(f"start holds {len(start)} states for {n_chains} chains")
        for c, st in enumerate(start):
            if st.P != p or st.max_par != mp:
                raise _bad_arg(f"start state of chain {c} is for P={st.P}, max_par={st.max_par}; "
                               f"the context has P={p}, max_par={mp}")
            if st.resumed and (st.rng != kind or st.n_samples != self.n_samples):
                raise _bad_arg(f"start state of chain {c} continues a stream of kind {st.rng} over "
                               f"{st.n_samples} samples; this run is kind {kind} over {self.n_samples}")
        resumed = {st.resumed for st in start}
        if len(resumed) > 1:
            raise _bad_arg("start mixes fresh and resumed chains")
        par = np.ascontiguousarray(np.stack([as_i32(st.parents) for st in start]))
        npar = np.ascontiguousarray(np.stack([as_i32(st.npar) for st in start]))
        keep += [par, npar]
        args.start_parents, args.start_n_par = par.ctypes.data_as(_lib._ip), npar.ctypes.data_as(_lib._ip)
        if resumed.pop():
            sts = (_lib.ChainStateC * n_chains)()
            for c, st in enumerate(start):
                o = sts[c]
                for k in _STATE_SCALARS:
                    setattr(o, k, int(getattr(st, k)))
                if kind == BN_RNG_WH:
                    o.wh_state[:] = [int(v) for v in st.wh_state]
            keep.append(sts)
            args.state_in = C.cast(sts, C.c_void_p)
            if kind == BN_RNG_RMT:
                mt_in = np.ascontiguousarray(np.stack([_i32_bits(st.mt_state) for st in start]))
                keep.append(mt_in)
                args.mt_state_in = mt_in.ctypes.data_as(_lib._ip)
        blocks = [st.score_block is not None for st in start]
        if any(blocks):
            if not all(blocks):
                raise _bad_arg("start gives a score block for some chains only")
            sb = np.ascontiguousarray(np.stack([np.asarray(st.score_block, dtype=np.float64) for st in start]))
            if sb.shape[1] != self.score_state_len:
                raise _bad_arg(f"score block of {sb.shape[1]} doubles; this context needs {self.score_state_len}")
            keep.append(sb)
            args.score_state_in = sb.ctypes.data_as(_lib._dp)

    def run(self, n_chains=1, n_iter=1000, output=100, initial_network=2, drop=0, rng="wh",
            seeds=None, replay=None, log_moves=False, moves_capacity=None, tabulate=False,
            mt_state=None, want_mt_state=False, start=None, want_state=False, tabulate_ancestors=False,
            track_best=False, tabulate_markov_blankets=False):
        """Run ``n_chains`` independent chains; returns (list[ChainResult], kernel_ms).

        ``mt_state`` (rng="rmt"): R's stream state per chain, ``.Random.seed[2:626]`` (625 ints:
        position + 624 words), instead of ``set.seed(seeds)``; ``want_mt_state`` returns the
        state after the run in ``ChainResult.mt_state``.

        ``start``: one :class:`ChainState` per chain.  Fresh states start the chains from their graphs
        (``initial_network`` is not read); resumed states continue each chain for ``n_iter`` more
        iterations with its own stream (rng="replay": ``replay`` holds the remaining uniforms, the
        original buffer from ``state.uniforms`` on).  ``want_state`` returns the state to continue
        from in ``ChainResult.state``, score block included.  Trace, move log and tabulation cover
        the iterations of this call.

        ``tabulate_ancestors``: ``ChainResult.anc_freq`` [descendant, ancestor] counts the tabulated
        iterations (those ``tabulate`` counts) after which the graph has a directed path ancestor -> ... ->
        descendant; its diagonal is the number of tabulated iterations.  Every other output is the same as
        without it.  ``summary.ancestor_posterior`` pools chains into probabilities.

        ``track_best``: ``ChainResult.best`` is the :class:`BestGraph` of the chain, the highest log posterior
        among the graphs held in the tabulated iterations of this call.  Every other output is the same as
        without it.  ``summary.best_graph`` picks the best over chains, or over the segments of a resumed
        run (the uninterrupted run's best).

        ``tabulate_markov_blankets``: ``ChainResult.mb_freq`` [P, P] (symmetric) counts the tabulated iterations
        after which j is in the Markov blanket of i: i -> j, j -> i, or a common child.  Its diagonal is the
        number of tabulated iterations.  Every other output is the same as without it.
        ``summary.markov_blanket_posterior`` pools chains into probabilities."""
        L = _lib.lib()
        kind = _RNG_KINDS[rng]
        p, mp = self.n_nodes, self.max_par
        cap = max(1, (n_iter + output - 1) // output)
        # (np.empty: bn_run overwrites every row up to n_rows, and only those are handed out)
        ints = {k: np.empty((n_chains, cap), dtype=np.int32) for k in
                ("iter", "ChangedNode", "movetype", "additions", "deletions", "FN", "FP")}
        gll = np.empty((n_chains, cap))
        n_rows = np.zeros(n_chains, dtype=np.int32)
        tr = _lib.Trace(cap, n_rows.ctypes.data_as(_lib._ip), ints["iter"].ctypes.data_as(_lib._ip),
                        ints["ChangedNode"].ctypes.data_as(_lib._ip),
                        ints["movetype"].ctypes.data_as(_lib._ip), gll.ctypes.data_as(_lib._dp),
                        ints["additions"].ctypes.data_as(_lib._ip),
                        ints["deletions"].ctypes.data_as(_lib._ip), ints["FN"].ctypes.data_as(_lib._ip),
                        ints["FP"].ctypes.data_as(_lib._ip))
        args = _lib.RunArgs()
        args.n_chains, args.rng_kind = int(n_chains), int(kind)
        sd = None
        if seeds is not None:
            sd = np.zeros((n_chains, 3), dtype=np.int32)
            s_in = np.asarray(seeds, dtype=np.int64)
            if s_in.ndim == 0:
                s_in = s_in.reshape(1, 1)
            if s_in.ndim == 1:
                s_in = s_in.reshape(n_chains, -1) if n_chains > 1 else s_in.reshape(1, -1)
            sd[:, :s_in.shape[1]] = s_in
            args.seeds = sd.ctypes.data_as(_lib._ip)
        rp = None
        if kind == BN_RNG_REPLAY:
            rp = np.ascontiguousarray(replay, dtype=np.float64)
            if rp.ndim == 1:
                rp = rp[None]
            if rp.shape[0] != n_chains:
                raise ValueError("replay must be (n_chains, replay_len)")
            args.replay = rp.ctypes.data_as(_lib._dp)
            args.replay_len = rp.shape[1]
        mt_in = mt_out = None
        if mt_state is not None:
            mt_in = _i32_bits(mt_state).reshape(n_chains, 625)
            args.mt_state_in = mt_in.ctypes.data_as(_lib._ip)
        if want_mt_state or mt_state is not None:
            mt_out = np.zeros((n_chains, 625), dtype=np.int32)
            args.mt_state_out = mt_out.ctypes.data_as(_lib._ip)
        args.initial_network, args.drop = int(initial_network), int(drop)
        args.n_iter, args.output_every, args.device_outputs = int(n_iter), int(output), 0
        moves = n_moves = None
        if log_moves:
            mc = int(moves_capacity if moves_capacity is not None else n_iter)
            moves = np.zeros((n_chains, max(mc, 1), 4), dtype=np.int32)
            n_moves = np.zeros(n_chains, dtype=np.int32)
            args.moves_capacity = moves.shape[1]
            args.moves = moves.ctypes.data_as(_lib._ip)
            args.n_moves = n_moves.ctypes.data_as(_lib._ip)
        freq = nfreq = None
        if tabulate:
            freq = np.zeros((n_chains, p, p), dtype=np.int32)
            args.edge_freq = freq.ctypes.data_as(_lib._ip)
            nfreq = np.zeros((n_chains, p, mp + 1), dtype=np.int32)
            args.npar_freq = nfreq.ctypes.data_as(_lib._ip)
        afreq = None
        if tabulate_ancestors:
            afreq = np.zeros((n_chains, p, p), dtype=np.int32)
            args.anc_freq = afreq.ctypes.data_as(_lib._ip)
        mbfreq = None
        if tabulate_markov_blankets:
            mbfreq = np.zeros((n_chains, p, p), dtype=np.int32)
            args.mb_freq = mbfreq.ctypes.data_as(_lib._ip)
        bpar = bnpar = bst = None
        if track_best:
            bpar = np.empty((n_chains, p, mp), dtype=np.int32)   # the library fills every entry
            bnpar = np.empty((n_chains, p), dtype=np.int32)
            bst = (_lib.BestGraphC * n_chains)()
            args.best_parents, args.best_n_par = bpar.ctypes.data_as(_lib._ip), bnpar.ctypes.data_as(_lib._ip)
            args.best = C.cast(bst, C.c_void_p)
        keep = []
        if start is not None:
            self._start_args(start, n_chains, kind, args, keep)
            if kind == BN_RNG_RMT and start[0].resumed and mt_out is None:
                mt_out = np.zeros((n_chains, 625), dtype=np.int32)
                args.mt_state_out = mt_out.ctypes.data_as(_lib._ip)
        st_out = sb_out = None
        if want_state:
            st_out = (_lib.ChainStateC * n_chains)()
            args.state_out = C.cast(st_out, C.c_void_p)
            sb_out = np.empty((n_chains, self.score_state_len))
            args.score_state_out = sb_out.ctypes.data_as(_lib._dp)
            if kind == BN_RNG_RMT and mt_out is None:
                mt_out = np.zeros((n_chains, 625), dtype=np.int32)
                args.mt_state_out = mt_out.ctypes.data_as(_lib._ip)
        fpar = np.empty((n_chains, p, mp), dtype=np.int32)   # the library pads unused slots with -1
        fnpar = np.empty((n_chains, p), dtype=np.int32)
        stats = (_lib.ChainStats * n_chains)()
        ms = C.c_float(0)
        status = L.bn_run(self._h, C.byref(args), C.byref(tr), ptr(fpar), ptr(fnpar),
                          C.cast(stats, C.c_void_p), C.byref(ms))
        check(status)
        # everything below is views (the per-chain Python work is part of every end-to-end step)
        st = np.frombuffer(stats, dtype=_lib.CHAIN_STATS_DTYPE, count=n_chains)
        out = []
        for ch in range(n_chains):
            r = int(n_rows[ch])
            trace = {k: ints[k][ch, :r] for k in ("iter", "ChangedNode", "movetype")}
            trace["globalLL"] = gll[ch, :r]
            for k in ("additions", "deletions", "FN", "FP"):
                trace[k] = ints[k][ch, :r]
            s = st[ch]
            out.append(ChainResult(
                trace=trace, uniforms=int(s["uniforms"]), valid_iters=int(s["valid_iters"]),
                proposed=tuple(s["proposed"].tolist()), reject=tuple(s["reject"].tolist()), n_nonpd=int(s["n_nonpd"]),
                total_edges=int(s["total_edges"]), windows=int(s["windows"]), alg_bytes=int(s["alg_bytes"]),
                phase_cycles=tuple(s["phase_cycles"].tolist()),
                slots_simulated=int(s["slots_simulated"]), kernel_cycles=int(s["kernel_cycles"]),
                mt_state=None if mt_out is None else mt_out[ch],
                final_parents=fpar[ch],
                final_npar=fnpar[ch],
                accepted_moves=None if moves is None else moves[ch, :int(n_moves[ch])],
                edge_freq=None if freq is None else freq[ch],
                npar_freq=None if nfreq is None else nfreq[ch],
                anc_freq=None if afreq is None else afreq[ch],
                mb_freq=None if mbfreq is None else mbfreq[ch]))
            if bst is not None:
                b = bst[ch]
                out[-1].best = BestGraph(parents=bpar[ch], npar=bnpar[ch], log_post=float(b.log_post),
                                         log_lik=float(b.log_lik), log_prior=float(b.log_prior), iter=int(b.iter),
                                         found=bool(b.found))
            if st_out is not None:
                o = st_out[ch]
                out[-1].state = ChainState(
                    parents=fpar[ch].copy(), npar=fnpar[ch].copy(), n_samples=self.n_samples, rng=kind,
                    wh_state=np.array(o.wh_state[:], dtype=np.int32) if kind == BN_RNG_WH else None,
                    mt_state=mt_out[ch].copy() if kind == BN_RNG_RMT else None, score_block=sb_out[ch],
                    **{k: int(getattr(o, k)) for k in _STATE_SCALARS})
        return out, float(ms.value)


    def run_device(self, n_chains, n_iter, output, d_ints, d_gll, d_n_rows, initial_network=2, drop=0,
                   rng="wh", seeds=None):
        """The same chains with the trace left in HBM (``bn_run_args.device_outputs = 1``): no
        device-to-host copy of the columns, so that they can be exchanged between GPUs directly
        (``dist.run_sharded_device``).  ``d_ints``: device pointer of an int32 buffer
        [7][n_chains][capacity] (columns iter, ChangedNode, movetype, additions, deletions, FN, FP),
        ``d_gll``: float64 [n_chains][capacity], ``d_n_rows``: int32 [n_chains]; capacity =
        ceil(n_iter / output).  Returns (stats array, kernel_ms)."""
        L = _lib.lib()
        cap = max(1, (n_iter + output - 1) // output)
        col = lambda k: C.cast(C.c_void_p(int(d_ints) + 4 * k * n_chains * cap), _lib._ip)
        tr = _lib.Trace(cap, C.cast(C.c_void_p(int(d_n_rows)), _lib._ip), col(0), col(1), col(2),
                        C.cast(C.c_void_p(int(d_gll)), _lib._dp), col(3), col(4), col(5), col(6))
        args = _lib.RunArgs()
        args.n_chains, args.rng_kind = int(n_chains), int(_RNG_KINDS[rng])
        sd = None
        if seeds is not None:
            sd = np.zeros((n_chains, 3), dtype=np.int32)
            s_in = np.asarray(seeds, dtype=np.int64).reshape(n_chains, -1)
            sd[:, :s_in.shape[1]] = s_in
            args.seeds = sd.ctypes.data_as(_lib._ip)
        args.initial_network, args.drop = int(initial_network), int(drop)
        args.n_iter, args.output_every, args.device_outputs = int(n_iter), int(output), 1
        stats = (_lib.ChainStats * n_chains)()
        ms = C.c_float(0)
        check(L.bn_run(self._h, C.byref(args), C.byref(tr), None, None, C.cast(stats, C.c_void_p), C.byref(ms)))
        return np.frombuffer(stats, dtype=_lib.CHAIN_STATS_DTYPE, count=n_chains).copy(), float(ms.value)


def block_colsum_device(data_ptr, ld, n_rows, n_nodes, out_ptr, device=0, stream=0):
    """Column sums of one row block of X (device pointers); see ``bn_block_colsum_device``."""
    check(_lib.lib().bn_block_colsum_device(C.c_void_p(int(data_ptr)), int(ld), int(n_rows), int(n_nodes),
                                            C.c_void_p(int(out_ptr)), int(device), C.c_void_p(int(stream))))


def block_gram_device(data_ptr, ld, n_rows, n_nodes, mean_ptr, out_ptr, device=0, stream=0):
    """One row block's part of the centred cross-product matrix (device pointers); returns kernel ms."""
    ms = C.c_float(0)
    check(_lib.lib().bn_block_gram_device(C.c_void_p(int(data_ptr)), int(ld), int(n_rows), int(n_nodes),
                                          C.c_void_p(int(mean_ptr)), C.c_void_p(int(out_ptr)), int(device),
                                          C.c_void_p(int(stream)), C.byref(ms)))
    return float(ms.value)


# ---------------------------------------------------------------------------
# the reference's two entry points
# ---------------------------------------------------------------------------
def main_fun(X, graph_source: Sequence[int], graph_target: Sequence[int],
             graph_node_labels: Sequence[int], graph_node_type: Sequence[int], MaxPar: int = 50,
             phi: float = 1, omega: float = 6.9, InitialNetwork: int = 2, drop: int = 0,
             N: int = 1000, output: int = 10, *, rng="wh", seed=None, random_seed=None) -> dict:
    """``main_fun`` of ``src/bayesnet_mcmc.cpp:27-38`` through the C ABI (``bn_main_fun``).

    ``rng``/``seed`` choose the uniform stream that stands in for ``R::runif``:
    ``"wh"`` (Wichmann-Hill, ``seed`` = (ix, iy, iz) or None for the reference's
    10437/13568/30524) or ``"rmt"`` (R's Mersenne-Twister, ``seed`` as in ``set.seed``).
    ``random_seed``: R's ``.Random.seed`` (626 ints, Mersenne-Twister kind 10403) as the reference
    finds it on entry (``Rcpp::RNGScope``, ``src/RcppExports.cpp:13``); the state it would leave
    behind is returned under the key ``".Random.seed"``.
    Returns the eight result columns as arrays, in the reference's order.
    """
    Xf = np.asfortranarray(np.asarray(X, dtype=np.float64))
    n, p = Xf.shape
    src, tgt = as_i32(graph_source), as_i32(graph_target)
    labels, nt = as_i32(graph_node_labels), as_i32(graph_node_type)
    if src.shape != tgt.shape:
        raise ValueError("graph_source and graph_target must have the same length")
    kind = _RNG_KINDS[rng]
    sd = None
    if seed is not None:
        sd = np.zeros(3, dtype=np.int32)
        s_in = np.atleast_1d(np.asarray(seed, dtype=np.int64))
        sd[:len(s_in)] = s_in
    st_in = st_out = None
    if random_seed is not None:
        rs = np.asarray(random_seed, dtype=np.int64)
        if rs.shape != (626,) or rs[0] % 100 != 3:
            raise ValueError("random_seed must be R's .Random.seed of the Mersenne-Twister (626 ints, kind %%100 == 3)")
        kind = BN_RNG_RMT
        st_in = _i32_bits(rs[1:])
        st_out = np.zeros(625, dtype=np.int32)
    elif kind == BN_RNG_RMT and seed is None:
        raise ValueError("rng='rmt' needs seed= (the value given to set.seed) or random_seed=")
    cap = max(1, (int(N) + int(output) - 1) // int(output)) if output > 0 else 1
    cols = {k: np.zeros(cap, dtype=np.float64 if k == "globalLL" else np.int32) for k in TRACE_COLUMNS}
    rows = _lib.lib().bn_main_fun(ptr(Xf), n, p, ptr(src), ptr(tgt), len(src), ptr(labels), ptr(nt),
                                  int(MaxPar), float(phi), float(omega), int(InitialNetwork),
                                  int(drop), int(N), int(output), int(kind), ptr(sd), cap,
                                  *[ptr(cols[k]) for k in TRACE_COLUMNS], ptr(st_in), ptr(st_out))
    if rows < 0:
        raise BnError(-rows, _lib.lib().bn_last_error().decode("utf-8", "replace"))
    out = {k: cols[k][:rows].copy() for k in TRACE_COLUMNS}
    if st_out is not None:
        out[".Random.seed"] = np.concatenate([[int(np.asarray(random_seed)[0])], st_out]).astype(np.int32)
    return out


def bn_mcmc(X, graph: Network, MaxPar: int = 50, phi: float = 1, omega: float = 6.9,
            InitialNetwork: int = 2, drop: int = 0, N: int = 1000, output: int = 100, *,
            rng="wh", seed=None, random_seed=None) -> dict:
    """``bn_mcmc`` of ``R/bn_mcmc.R:8-25``: unpack the network object and forward to main_fun."""
    return main_fun(X=X, graph_target=graph.target, graph_source=graph.source,
                    graph_node_labels=np.arange(graph.n_nodes, dtype=np.int32),
                    graph_node_type=graph.node_type_codes(), MaxPar=MaxPar, phi=phi, omega=omega,
                    InitialNetwork=InitialNetwork, drop=drop, N=N, output=output, rng=rng, seed=seed,
                    random_seed=random_seed)
