/* bn_b200.h -- C ABI of libbn_b200.so: the B200 (sm_100a) implementation of the
 * structure-MCMC scoring hot path of USCbiostats/bayesnetworks.
 *
 * This is the drop-in boundary: the host `main_fun` (same signature as the
 * reference's src/bayesnet_mcmc.cpp:27-38) calls these entry points instead of
 * running the CPU loop of src/bayesnet_mcmc.cpp:40-71.  Plain pointers and
 * sizes only; nothing throws across the boundary; every function returns a
 * status (0 = ok) and bn_last_error() describes the last failure of the
 * calling thread.  All host pointers are borrowed for the duration of the call
 * (caller-owned, like R's memory behind NumericMatrix); results are written
 * into caller-allocated buffers.
 *
 * There is no CPU fallback: without a CUDA device every compute entry point
 * fails with BN_ERR_NO_DEVICE.
 */
#ifndef BN_B200_H
#define BN_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BN_B200_ABI_VERSION 3

/* ---- status codes -------------------------------------------------------- */
enum {
  BN_OK = 0,
  BN_ERR_BAD_ARG = 1,            /* NULL pointer, size <= 0, edge index out of range, ... */
  BN_ERR_CUDA = 2,               /* a CUDA runtime/driver call failed */
  BN_ERR_OOM = 3,                /* device or host allocation failed */
  BN_ERR_NO_LEGAL_PROPOSAL = 4,  /* no legal child / parent exists at all (every candidate child is
                                    a source or at max_par, every candidate parent a sink or
                                    already a parent): the reference would spin forever in
                                    src/network.h:283-299.  Rare-but-legal proposals never fail:
                                    an iteration may consume any number of uniforms */
  BN_ERR_NO_DEVICE = 5,          /* no CUDA device / device index out of range */
  BN_ERR_CAPACITY = 6,           /* caller buffer too small */
  BN_ERR_UNSUPPORTED = 7         /* e.g. max_par > 64 */
};

/* ---- uniform streams (replaces R::runif, call sites src/bayesnet_mcmc.cpp:48,
 *      src/network.h:284,292,309,318,319,335) ------------------------------ */
enum {
  BN_RNG_WH = 0,      /* Wichmann-Hill, Bayes-networks/random4f.h:17-49; 3 seeds per chain */
  BN_RNG_RMT = 1,     /* R's Mersenne-Twister: set.seed(seeds[3c]) scrambling, or the stream state
                         itself (bn_run_args.mt_state_in = .Random.seed[2:626]) */
  BN_RNG_REPLAY = 2   /* caller-supplied uniforms (replay_len per chain) */
};

typedef struct bn_ctx bn_ctx; /* opaque: one per device / per calling thread */

const char* bn_last_error(void);
int bn_abi_version(void);
int bn_device_count(void);

/* ---- context: dataset -> sufficient statistics on the device ---------------
 * Replaces network::network (src/network.h:101-171): the constructor's
 * sumX / sumXX triple loop (:124-136) becomes the FP64 tensor-core Gram kernel,
 * the prior adjacency simEdge / NsimEdges (:138-146) and node types are
 * uploaded once.  X is column-major n_samples x n_nodes (R layout, X(n,p) =
 * X[n + p*n_samples]).  Edges are 1-based (source -> target), as in
 * graph$source / graph$target.  node_type: 0 neither, 1 source, 2 sink.
 * A node of the supplied graph may have more than max_par parents: with
 * InitialNetwork = 2 the graph only feeds simEdge / NsimEdges (:138-146,164-169);
 * bn_run refuses InitialNetwork = 0 in that case. */
int bn_create(const double* X_colmajor, int n_samples, int n_nodes,
              const int* edge_src_1b, const int* edge_tgt_1b, int n_edges,
              const int* node_type, int max_par, double phi, double omega,
              int device, bn_ctx** out);

/* Same, X already resident in device memory on `device` (not modified);
 * ld = leading dimension in elements (>= n_samples). */
int bn_create_from_device(const double* dX_colmajor, int64_t ld, int n_samples, int n_nodes,
                          const int* edge_src_1b, const int* edge_tgt_1b, int n_edges,
                          const int* node_type, int max_par, double phi, double omega,
                          int device, bn_ctx** out);

/* Same, from sufficient statistics computed elsewhere: column means and the
 * centred cross-product matrix S(i,j) = sum_n (x_ni - mean_i)(x_nj - mean_j)
 * (n_nodes x n_nodes, symmetric, either major). */
int bn_create_from_stats(int n_samples, int n_nodes, const double* mean,
                         const double* centered_gram,
                         const int* edge_src_1b, const int* edge_tgt_1b, int n_edges,
                         const int* node_type, int max_par, double phi, double omega,
                         int device, bn_ctx** out);

/* Row-sharded sufficient statistics (the N axis of a matrix too large or too slow for one
 * GPU, e.g. 5,000 x 1,000,000): a row block dX (n_rows x n_nodes, column-major, device
 * memory) contributes its column sums, and -- once the caller has formed the GLOBAL means
 * from the sums of all blocks -- its part of the centred cross-product matrix
 *   out_gram[p1 + p2*P] = sum over the block's rows of (x_np1 - mean_p1)(x_np2 - mean_p2).
 * The caller adds the parts of all blocks in a fixed block order (bit-identical for any
 * number of GPUs; bayesnetworks_b200/dist.py does it with an NCCL all-gather) and hands the
 * result to bn_create_from_stats_device.  All pointers are device pointers on `device`;
 * stream NULL = the thread's default stream (bn_set_default_stream).  Replaces the same
 * loop as bn_create: network::network, src/network.h:124-136. */
int bn_block_colsum_device(const double* dX_colmajor, int64_t ld, int n_rows, int n_nodes,
                           double* d_out_sum, int device, void* cuda_stream);
int bn_block_gram_device(const double* dX_colmajor, int64_t ld, int n_rows, int n_nodes,
                         const double* d_mean, double* d_out_gram, int device, void* cuda_stream,
                         float* kernel_ms);
int bn_create_from_stats_device(int n_samples, int n_nodes, const double* d_mean,
                                const double* d_centered_gram,
                                const int* edge_src_1b, const int* edge_tgt_1b, int n_edges,
                                const int* node_type, int max_par, double phi, double omega,
                                int device, bn_ctx** out);

void bn_destroy(bn_ctx* ctx);

/* Scratch device buffers are pooled per device between calls (cudaMalloc/cudaFree cost more
 * than the kernels); this returns the idle ones to the driver.  BN_B200_POOL=0 disables. */
int bn_trim_pool(void);

/* Launch all subsequent work of this context on the given cudaStream_t
 * (passed as void*); NULL restores the context's own stream. */
int bn_set_stream(bn_ctx* ctx, void* cuda_stream);

/* Stream that contexts created afterwards BY THIS THREAD start on (so that the
 * Gram build of bn_create* can be bracketed by the caller's CUDA events); NULL =
 * each context creates its own non-blocking stream (the default). */
int bn_set_default_stream(void* cuda_stream);

/* Read back the sufficient statistics.  Any pointer may be NULL.
 *   sum_x[p]            = sum_n X(n,p)                       (src/network.h:129)
 *   sum_xx[p1 + p2*P]   = sum_n X(n,p1) X(n,p2)              (src/network.h:131)
 *   mean[p], centered[p1 + p2*P] as in bn_create_from_stats. */
int bn_get_stats(bn_ctx* ctx, double* sum_x, double* sum_xx, double* mean, double* centered);

/* Device time of the last Gram build in milliseconds (CUDA events), and the
 * number of kernels this context has launched so far. */
int bn_get_gram_ms(bn_ctx* ctx, float* ms);
int64_t bn_get_launch_count(bn_ctx* ctx);

/* ---- scoring -------------------------------------------------------------- */
/* score(child | ordered parent list): network::score, src/network.h:183-237.
 * parents is [n_items][max_par] (row stride = the context's max_par).
 * A non-positive-definite parent Gram yields -inf (and is counted). */
int bn_score_nodes(bn_ctx* ctx, int n_items, const int* child, const int* parents,
                   const int* n_par, double* out_ll);

/* Batched proposal scoring: for each of n_graphs DAGs (parents [g][P][max_par],
 * n_par [g][P]) score EVERY single-edge add/delete proposal in one launch.
 *   out_base[g][c]       score of node c with its current parents
 *   out_score[g][c][j]   score of node c after toggling parent j (add if absent,
 *                        delete if present); NaN where the move is masked:
 *                        j == c, child is a source (node_type 1), parent is a sink
 *                        (node_type 2), or the child already has max_par parents;
 *                        -inf where the new parent set is degenerate: its parent Gram
 *                        is not positive definite, it fits the child exactly, or an
 *                        addition leaves no residual degrees of freedom
 *                        (n_samples - k - 2 <= 0 for k current parents)
 *   out_log_hr[g][c][j]  (new - old) + (NewLogPrior - OldLogPrior): the log Hastings
 *                        ratio of src/network.h:334 with the Potts prior of
 *                        src/network.h:254-279 applied in-kernel; NaN where masked,
 *                        and where both the current and the new score are -inf.
 * Acyclicity is not checked here (src/network.h:415-432 runs per proposal in
 * the chain).  Any output pointer may be NULL.  Host pointers. */
int bn_score_all_proposals(bn_ctx* ctx, int n_graphs, const int* parents, const int* n_par,
                           double* out_base, double* out_score, double* out_log_hr);

/* Device-pointer variant of the same launch (for timing without copies);
 * *kernel_ms receives the device time of the launch. */
int bn_score_all_proposals_device(bn_ctx* ctx, int n_graphs, const int* d_parents,
                                  const int* d_n_par, double* d_out_base, double* d_out_score,
                                  double* d_out_log_hr, float* kernel_ms);

/* ---- the chains ------------------------------------------------------------
 * Replaces the loop of src/bayesnet_mcmc.cpp:45-70 with network::propose_*,
 * CheckValidity, checker, logger (src/network.h:281-364), for n_chains
 * independent chains on this context's device. */
typedef struct bn_trace {
  int capacity;        /* rows allocated per chain; needs >= ceil(n_iter/output_every) */
  int* n_rows;         /* [n_chains]            rows written (invalid iterations log nothing) */
  int* iter;           /* [n_chains*capacity]   columns of network::result(), src/network.h:353-364 */
  int* changed_node;
  int* movetype;
  double* global_ll;
  int* additions;
  int* deletions;
  int* fn;
  int* fp;
} bn_trace;

typedef struct bn_chain_stats {
  int64_t uniforms;        /* uniforms consumed */
  int64_t valid_iters;     /* iterations that reached checker() = proposals scored */
  int proposed[3];         /* ProposedMoves[], src/network.h:331 */
  int reject[3];           /* reject[],        src/network.h:87-89,434-437 */
  int n_nonpd;             /* proposals whose parent Gram was not positive definite */
  int total_edges;         /* edges of the final graph */
  int status;              /* BN_OK or BN_ERR_NO_LEGAL_PROPOSAL */
  int windows;             /* rounds (position-parallel) + sequential windows executed */
  int64_t alg_bytes;       /* sum over scored proposals of 8*(k'+1)(k'+2)/2 + 8: the algorithmic
                              gather bytes of the roofline (k' = parents in the scored set) */
  int64_t phase_cycles[12];/* SM cycles of the chain's warp per phase: uniform refill, position records
                              (draw replay + scoring), walk + repair, commit, accepted additions,
                              accepted deletions; [6..11] split the last two (list update, ancestor
                              update, -) */
  int64_t slots_simulated; /* iterations emitted by the record walk */
  int64_t kernel_cycles;   /* SM cycles of the chain from its first to its last iteration (ABI >= 3);
                              phase_cycles are filled by diagnostics builds only (-DBN_PHASE_CYCLES) */
} bn_chain_stats;

/* What a chain carries across a segment boundary besides its graph, its scores and its stream. */
typedef struct bn_chain_state {
  int64_t iter;              /* next iteration index */
  int valid;                 /* the stale `valid` flag, src/bayesnet_mcmc.cpp:40 (0 or 1) */
  int total_edges_member;    /* TotalEdges as the last LogPrior() left it, src/network.h:262-267 */
  int additions, deletions;  /* accepted moves since `drop` (trace columns) */
  int wh_state[3];           /* BN_RNG_WH: the stream state, a seed triple (state_out: after the uniforms
                                consumed); 0 for the other streams */
  int64_t uniforms;          /* uniforms consumed since iteration 0 (random start graph included) */
} bn_chain_state;

/* The best graph a chain visited in one call (bn_run_args.best). */
typedef struct bn_best_graph {
  double log_post, log_lik, log_prior;
  int64_t iter;        /* first tabulated iteration after which the chain held it; -1 if none */
  int total_edges;
  int found;           /* 0: this call tabulated no iteration */
} bn_best_graph;

typedef struct bn_run_args {
  int n_chains;
  int rng_kind;            /* BN_RNG_* */
  const int* seeds;        /* [3*n_chains] (WH: ix,iy,iz; RMT: seed,-,-); NULL = chain 0 uses
                              the reference seeds 10437/13568/30524, chain c > 0 a SplitMix64
                              derived triple (see DESIGN.md) */
  const double* replay;    /* BN_RNG_REPLAY: [n_chains*replay_len] */
  int64_t replay_len;
  int initial_network;     /* 2 = empty graph; 1 = random graph drawn from the chain's own stream before
                              iteration 0 (the defined variant of src/network.h:148-163, which is
                              undefined behaviour in the reference: same draw order, but duplicate
                              parents and cycle-closing parents are re-drawn, at most 100 draws per
                              slot); any other value = start from the supplied graph (:148-170) */
  int drop;
  int n_iter;
  int output_every;
  int device_outputs;      /* 0: trace/final_* pointers are host memory; 1: device memory */
  /* accepted-move log (optional, may be NULL): up to moves_capacity rows per chain of
     (iter, movetype, child, parent) */
  int moves_capacity;
  int* n_moves;            /* [n_chains] */
  int* moves;              /* [n_chains*moves_capacity*4] */
  /* posterior tabulation (optional, may be NULL), Bayes-networks/main.cpp:289-297:
     edge_freq[chain][parent + child*P] += 1 for every edge of the kept graph after each
     iteration i with i+1 > drop (anc_freq and mb_freq, at the end of this struct, tabulate directed paths and
     Markov blankets the same way) */
  int* edge_freq;
  /* freqNpar of the same Tabulate(), main.cpp:291 (optional, may be NULL; ABI version >= 2):
     npar_freq[chain][node*(max_par+1) + k] = counted iterations the node spent with k parents */
  int* npar_freq;
  /* R's Mersenne-Twister stream state (ABI >= 3; BN_RNG_RMT only; HOST memory whatever
     device_outputs says; may be NULL).  625 ints per chain in the layout of R's
     .Random.seed[2:626]: the position (dummy[0], 624 = regenerate first) and the 624 state
     words.  mt_state_in: the chains start from this state instead of set.seed(seeds[3c]);
     mt_state_out: the state after exactly the uniforms the chain consumed, i.e. what
     GetRNGstate / R::runif x n / PutRNGstate of the reference leaves behind
     (src/RcppExports.cpp:13, src/bayesnet_mcmc.cpp:48, src/network.h:284,292,309,318,319,335). */
  const int* mt_state_in;
  int* mt_state_out;
  /* ---- resumable chains (all NULL = the chains start as above; bn_score_state_len marks a library that has them) ----
     A run of N iterations split into segments, each started from what the previous one returned
     (state_out, final_parents/final_n_par, score_state_out, and the stream: wh_state, mt_state_out, or the
     rest of the replay buffer), computes the same bits as one run of N iterations: trace, move log,
     summed tabulations, final graph, stream state.
     start_parents / start_n_par: [n_chains][P][max_par] (-1 padded, list order) and [n_chains][P]; HOST
       memory.  The chains start from these graphs instead of the one initial_network names.  Each graph
       must be acyclic, without self-loops or duplicate parents, with n_par <= max_par.
       Without state_in this is a fresh chain from that graph: iteration 0, valid = 1, member TotalEdges 0,
       streams from seeds / mt_state_in as above.
     state_in: [n_chains], HOST memory, needs start_parents: a resume.  Each chain runs n_iter more
       iterations, from state_in[c].iter up to state_in[c].iter + n_iter (<= INT_MAX).  Its stream:
       BN_RNG_WH from wh_state (seeds are not read), BN_RNG_RMT from mt_state_in (required), BN_RNG_REPLAY
       from `replay`, which then holds the remaining uniforms (the run's buffer from state_in[c].uniforms on).
     state_out: [n_chains], HOST memory: the state to continue from (the graph is final_parents/final_n_par).
     score_state_in / score_state_out: [n_chains][bn_score_state_len] doubles, host or device memory as
       device_outputs says (score_state_in needs start_parents).  The per-node scores, followed for
       max_par > 8 by the per-node Cholesky factors.  Without score_state_in the chains recompute them
       from the start graphs: exactly the same bits for max_par <= 8; for max_par > 8 a factor that
       followed accepted deletions (Givens downdates) is refactorised, which agrees to rounding only, so
       globalLL may differ in the last bits and, very rarely, a decision with it.
     The edge and parent-count tabulations count the iterations of this call only (from
     max(drop, iter)); the segments' tabulations add up to the whole run's.  The opt-in two-CTA form
     (BN_B200_PIPE) is not used when any of these fields is set: the one-CTA kernel runs instead. */
  const int* start_parents;
  const int* start_n_par;
  const bn_chain_state* state_in;
  bn_chain_state* state_out;
  const double* score_state_in;
  double* score_state_out;
  /* ---- posterior ancestor tabulation (optional, may be NULL; host or device memory as device_outputs says) ----
     anc_freq[chain][a + d*P] counts the iterations i with i+1 > drop after which the kept graph has a
     directed path a -> ... -> d (a is an ancestor of d): the iterations and graphs edge_freq counts, from
     max(drop, iter) on, with the same index orientation, edge_freq[parent + child*P].  So
       - the diagonal holds the number of tabulated iterations (a node is its own ancestor): the
         denominator of the posterior probability of a path;
       - anc_freq >= edge_freq elementwise.
     Like edge_freq it covers the iterations of this call only; the segments of a resumed run add up to
     the uninterrupted run's counts, and bn_chain_state carries nothing for it.  The chains run the
     kernels of the resumable-chain fields (the two-CTA form is not used); every other output is the
     same as without it.  P*P ints per chain, as edge_freq. */
  int* anc_freq;
  /* ---- best graph visited (optional: all three set, or none; host or device memory as device_outputs says) ----
     For each chain, the graph with the highest log posterior log_lik + log_prior among the graphs edge_freq
     counts: those kept after the iterations i with i+1 > drop, from max(drop, iter) up to the end of the
     call.  With D = max(drop, iter), a graph created by the move at iteration t and replaced at iteration t'
     (or held to the end) is a candidate iff t' > D (end > D); so the start graph is not one when the move at
     iteration D is accepted, and it is the best when no move is accepted after D.
       - log_lik is the chain's globalLL of that graph (the sum of its node scores in the chain's fixed order):
         exactly the value a trace row logged while the graph was held shows.
       - log_prior = -phi*(FP + FN) - omega*TotalEdges of that graph, FP = TotalEdges - Nagree and
         FN = NsimEdges - Nagree (the chain's LogPrior, evaluated without contraction).
       - Ties: a later graph replaces the best only if its log_post is strictly greater (the first graph to
         reach the maximum wins).
       - iter: the first tabulated iteration after which the chain held it, max(creation iteration, D).
     When the call tabulates no iteration (end <= D): found = 0, the lists are -1 / 0, log_post, log_lik and
     log_prior are -inf, iter = -1 and total_edges = 0.
     Like edge_freq it covers the iterations of this call only and bn_chain_state carries nothing for it.
     Segments of a resumed run combine on the host: the first of the highest log_post over the segments in
     order, skipping found = 0, is the uninterrupted run's best (a graph held across a boundary is a candidate
     in both segments and the earlier wins the tie); bit for bit when resumed with score_state_in.  The chains
     run the kernels of the resumable-chain fields (the two-CTA form is not used); every other output is the
     same as without it. */
  int* best_parents;         /* [n_chains][P][max_par], -1 padded, list order */
  int* best_n_par;           /* [n_chains][P] */
  bn_best_graph* best;       /* [n_chains] */
  /* ---- posterior Markov blanket tabulation (optional, may be NULL; host or device memory as device_outputs says) ----
     mb_freq[chain][i + j*P] counts the iterations i' with i'+1 > drop after which j is in the Markov blanket of i
     in the kept graph: i -> j, j -> i, or some node has both i and j as parents.  These are the iterations and
     graphs edge_freq counts, from max(drop, iter) on.  So
       - the matrix is symmetric, and its diagonal holds the number of tabulated iterations: the denominator
         of the posterior probability of blanket membership;
       - off the diagonal, mb_freq >= edge_freq + its transpose, with equality at max_par = 1.
     Like edge_freq it covers the iterations of this call only; the segments of a resumed run add up to
     the uninterrupted run's counts, and bn_chain_state carries nothing for it.  The chains run the
     kernels of the resumable-chain fields (the two-CTA form is not used); every other output is the
     same as without it.  P*P ints per chain, as edge_freq, and a P*P matrix of 16-bit witness counts per
     chain in scratch memory. */
  int* mb_freq;
} bn_run_args;

/* Per-chain length (doubles) of score_state_in / score_state_out. */
int bn_score_state_len(bn_ctx* ctx, int64_t* n_doubles);

/* final_parents: [n_chains][P][max_par] (-1 padded), final_n_par: [n_chains][P]; may be NULL.
 * stats: [n_chains]; may be NULL.  *kernel_ms (may be NULL) = device time of the run. */
int bn_run(bn_ctx* ctx, const bn_run_args* args, bn_trace* trace, int* final_parents,
           int* final_n_par, bn_chain_stats* stats, float* kernel_ms);

/* ---- host twin of the reference's main_fun (src/bayesnet_mcmc.cpp:27-38) ----
 * Plain-type signature of
 *   DataFrame main_fun(NumericMatrix X, vector<int> graph_source, graph_target,
 *                      graph_node_labels, graph_node_type, int MaxPar, double phi,
 *                      double omega, int InitialNetwork, int drop, int N, int output)
 * One chain, one device (device 0).  graph_node_labels is accepted and unused, as
 * in the reference (src/bayesnet_mcmc.cpp:30).  The eight result columns are
 * written to caller arrays of `capacity` rows; returns the number of rows
 * (>= 0) or -(status) on error.  rng_kind/seeds select the uniform stream; with
 * BN_RNG_RMT, mt_state_in / mt_state_out carry R's stream state in and out (see
 * bn_run_args), which is how the Rcpp glue keeps R's `bn_mcmc` after `set.seed` on the
 * reference's trajectory and R's .Random.seed advanced as the reference leaves it. */
int bn_main_fun(const double* X_colmajor, int n_samples, int n_nodes,
                const int* graph_source, const int* graph_target, int n_edges,
                const int* graph_node_labels, const int* graph_node_type,
                int MaxPar, double phi, double omega, int InitialNetwork, int drop, int N,
                int output, int rng_kind, const int* seeds,
                int capacity, int* iter, int* ChangedNode, int* movetype, double* globalLL,
                int* additions, int* deletions, int* FN, int* FP,
                const int* mt_state_in /* [625] or NULL */, int* mt_state_out /* [625] or NULL */);

#ifdef __cplusplus
}
#endif
#endif /* BN_B200_H */
