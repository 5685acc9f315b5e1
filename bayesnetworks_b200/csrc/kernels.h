// Host-side interface of kernels.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "chain_core.cuh"

namespace bn {

// (a kernel parameter: 16-byte aligned, so that a new field shifts the parameters behind it by whole 16-byte
// steps and the default kernels keep their code)
struct alignas(16) ChainWorkspace {  // arrays over all chains of a run (device memory)
  int* par; int* npar; int* born; double* base;
  int* hp_list;
  uint32_t* anc; uint32_t* haspar;   // anc rows are anc_stride(W) words apart in global memory
  int* scratch; int scratch_n;        // scratch_words(P, ...) ints per chain
  int* t_iter; int* t_changed; int* t_movetype; double* t_gll;
  int* t_add; int* t_del; int* t_fn; int* t_fp;
  int* moves; int* edge_freq; int* npar_freq; int* npar_since;
  double* dscore;                      // [nc][P][max_par] deletion-score cache (all-ones = unknown)
  double* fac;                         // [nc][P][fac_stride(max_par)] per-node Cholesky factors
  double* rowbuf;                      // [nc][REPLAY_POS][row_stride(max_par)] candidate rows of a round
  int pipeline;                        // 1: two CTAs per chain (chain_pipe_kernel): dscore holds (score, tag) pairs,
                                       // the R-MT states are [2][nc][624] (one copy per CTA)
  // supplied starts (one-CTA kernel only; null = the start graph of initial_network)
  const int* start_par; const int* start_npar;  // [nc][P][max_par], [nc][P]
  const ChainStart* start;             // [nc] resumed chains: each runs n_iter iterations from its start->iter
  int scores_in;                       // base (and fac) already hold the chains' scores and factors
  int scores_out;                      // write the final scores back to base when they lived in shared memory
  int with_state;                      // any of the above, the chains' end state wanted, anc_freq or best: the
                                       // WITH_STATE kernels
  int* anc_freq;                       // [nc][P][P] posterior ancestor tabulation, or null (last: the fields the
                                       // default kernels read keep their offsets)
  BestTrack* best;                     // [nc] best graph visited (its arrays and constants set up by the caller), or null
};

// Which per-chain arrays live in dynamic shared memory (byte offset, -1 = global memory).
// One chain = one CTA, so the hot state (parent lists, scores, ancestor bitsets) sits
// ~30 cycles away instead of an L2 round trip; arrays that do not fit stay in global.
struct ChainSmemPlan {
  int off_types, off_npar, off_base, off_haspar, off_hplist, off_par, off_scratch, off_anc, off_nver;
  int off_ubuf, off_ws, off_helper, off_dof, off_link;  // two-CTA form only
  int total_bytes;
};

// row stride (words) of the ancestor bitsets: a multiple of 4 (128-bit chunks)
inline int anc_stride(int W) { return (W + 3) / 4 * 4; }

struct ChainRngArgs {
  int kind;
  const int* seeds;          // [3*n_chains]
  uint32_t* mt_states;       // [624*n_chains] (R-MT)
  const int* mt_pos;         // [n_chains] position within the state (624 = regenerate first)
  const double* replay;      // [replay_len*n_chains]
  int64_t replay_len;
};

struct ChainResult {
  int64_t uniforms, valid_iters, alg_bytes;
  int proposed[3], reject[3];
  int n_nonpd, total_edges, status, windows, n_rows, n_moves;
  long long cyc[12], slots_sim, cyc_total;
  long long pipe_cyc[6];
  int pipe[4];  // two-CTA form: windows requested, waits for the builder, windows discarded, in-place rebuilds
  ChainStart end;  // (one-CTA kernel) the scalars to resume from
};

struct SweepParams {
  int P, max_par, n_graphs, n_samples, n_sim_edges;
  const double* C; int64_t ldc; const double* diag;
  const uint8_t* node_type; const uint8_t* sim_edge;
  double phi, omega;
  const int* parents; const int* n_par;   // [g][P][max_par], [g][P]
  int* te; int* agree;                     // [g] scratch
  int* order;                              // [g*P] scratch: items by falling parent count (null: natural order)
  double* out_base; double* out_score; double* out_log_hr;
};

// true when launch_chains can run the two-CTA form for this shape (MaxPar <= 8, state fits in shared memory)
bool chains_can_pipeline(ChainParams p, int scratch_n);
const char* launch_chains(ChainParams p, const ChainWorkspace& w, const ChainRngArgs& ra,
                          ChainResult* d_results, int n_chains, cudaStream_t stream);
const char* launch_score_nodes(const double* C, int64_t ldc, int n_samples, int max_par, int n_items,
                               const int* d_child, const int* d_parents, const int* d_npar, double* d_out,
                               int* d_nonpd, cudaStream_t stream);
void launch_diag(const double* C, int64_t ldc, int P, double* d_diag, cudaStream_t stream);
const char* launch_sweep(const SweepParams& sp, cudaStream_t stream);

}  // namespace bn
