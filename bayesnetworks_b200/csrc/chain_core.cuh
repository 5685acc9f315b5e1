// One MCMC chain = one CTA of eight warps, persistent for the whole run.  Replaces the loop of
// src/bayesnet_mcmc.cpp:45-70 and network::{propose_addition, propose_deletion, CheckValidity,
// checker, LogPrior, logger} (src/network.h:254-364,415-437).
//
// The reference's chain is strictly sequential, but the only dependences between iterations are
// the uniform-stream position (an iteration consumes a data-dependent number of uniforms), the
// stale `valid` flag, and the graph, which changes on the few percent of iterations that are
// accepted.  So the chain works in ROUNDS of 256 stream positions (run_round):
//   records   one thread per stream position q builds the record of the iteration that WOULD
//             start at q: the reference's draw order (move type, rejection-sampled child and
//             parent, the deletion draws), the acyclicity bit, the score of the proposed parent
//             set and the accept decision (build_record);
//   walk      warp 0 chases the records from the committed position (each record says how many
//             uniforms it consumes for either value of the incoming `valid` flag), one lane per
//             iteration, up to the first accepted one; statistics stay lane-private
//             (round_epoch);
//   apply     the accepted move is applied (parent list, ancestor bitsets by all eight warps) and
//             the remaining records are REPAIRED instead of discarded: records of the changed
//             child go stale, cycle bits are re-tested, deletion records are redone when the set
//             of nodes with parents changed (repair_record, build_record with redo_from).
// The committed result is exactly the sequential one (bit-identical trajectories).  Iterations
// the records cannot represent -- `TotalEdges < 3` (src/bayesnet_mcmc.cpp:48), more than 254
// uniforms -- take sequential windows (phase_a / phase_bc / commit); an iteration that needs more
// uniforms than the ring holds slides the ring along (phase_a, unbounded).
//
// Acyclicity (pathExists, src/network.h:366-413, a BFS per proposal) is an O(1) bit test against
// per-node ancestor bitsets, maintained on accepted moves.
//
// An experimental second form (chain_pipe_kernel, opt-in) spreads a chain over a cluster of two CTAs: one walks,
// commits and applies, the other keeps a replica of the graph and builds the records of the next window
// ("Two-CTA pipeline" below; bit-identical, not faster: profiles/r02_two_cta_chain.md).
//
// The same source compiles for the host with a one-lane warp (tests/emu): the sequential logic is
// checked against the oracle without a GPU.
#pragma once

#include "bn_common.cuh"
#include "rng_core.cuh"
#include "score_core.cuh"

namespace bn {

constexpr int WIN = 32;  // iterations committed per epoch, one lane each
constexpr int REPLAY_POS = 256;  // stream positions replayed and scored per round (8 warps x 32 lanes)

// t_rec layout of a position record
constexpr int REC_LEN_MASK = 0xff;      // uniforms consumed before the acceptance draw
constexpr int REC_TYPE = 1 << 8;        // 0 = addition, 1 = deletion
constexpr int REC_CYC = 1 << 9;         // addition that closes a cycle (invalid)
constexpr int REC_OVF = 1 << 10;        // ran out of the uniform ring
constexpr int REC_AG = 1 << 11;         // edge is in the prior graph
constexpr int REC_ACC = 1 << 12;        // checker() accepts (given the iteration is valid)
constexpr int REC_NPD = 1 << 13;        // non-positive-definite parent Gram
constexpr int REC_FULLMANY = 1 << 14;   // more than two children were skipped for being at MaxPar
constexpr int REC_STALE = 1 << 15;      // an accepted move of this round changed what the record depends on
constexpr int REC_KK_SHIFT = 16;        // size of the scored parent set (7 bits)
constexpr int REC_NOSCORE = 1 << 23;    // cyclic when built: never scored (stale if the cycle bit clears)
constexpr int REC_CLOSE = 1 << 24;      // log u within 1e-6 of the log Hastings ratio: decided by the
                                        // reference's own expression, stale after any accepted move
// t_walk: bits 0-7 / 8-15 uniforms consumed when the incoming `valid` flag is 0 / 1 (with the
// acceptance draw), bits 16 / 17 outgoing `valid`, bits 18 / 19 "this iteration is accepted",
// bits 20 and 21 record overflow (so that w >> (16 + v) has valid, accept, overflow at bits 0, 2, 4)
constexpr int WALK_STOP = 3 << 20;            // the walk cannot consume this record, because ...
constexpr int WALK_OVF = WALK_STOP | (1 << 24);    // ... it ran out of the uniform ring
constexpr int WALK_STALE = WALK_STOP | (1 << 25);  // ... an accepted move changed what it depends on
constexpr int WALK_END = WALK_STOP | (1 << 26);    // ... it lies behind the positions of this round

struct ChainParams {  // read-only, shared by all chains of a run
  int P, max_par, W, Ws, n_samples;  // W = words per bitset, Ws = row stride of anc (odd when in smem)
  const double* C;      // centred Gram [P][ldc]
  int64_t ldc;
  const double* diag;   // [P] its diagonal
  ScoreConsts sc;       // N / 2 and the (N - 1) / (N - k - 1) table of the score
  const uint8_t* node_type;  // [P] 0 neither / 1 source / 2 sink
  const uint8_t* sim_edge;   // [parent + child*P] prior adjacency, src/network.h:138-146
  int n_sim_edges;
  double phi, omega;
  int initial_network, drop, n_iter, output_every;
  int trace_capacity, moves_capacity;
  // prior graph (InitialNetwork == 0 start), [P][prior_stride] + [P]
  const int* prior_par;
  const int* prior_npar;
  int prior_stride;
  // row geometry of the ancestor bitsets for this warp width (set_row_geom)
  int g_chunks, g_lpr, g_rpp;
};

struct PipeLink;

// What a resumed chain carries over from the run that stopped it, besides its graph and its stream
struct ChainStart {
  int64_t iter;          // next iteration index
  int valid;             // stale `valid` flag, src/bayesnet_mcmc.cpp:40
  int te_m;              // member TotalEdges as left by the last LogPrior()
  int acc_add, acc_del;  // accepted moves since `drop`
};

// Best graph visited (ChainMem.best; see best_visit), one per chain in global memory.  The first six fields
// are bn_best_graph of include/bn_b200.h, which bn_run copies out; then the tracking state; then what the
// caller sets up (so that the chain itself carries one pointer for it).
struct BestTrack {
  double log_post, log_lik, log_prior;
  int64_t iter;          // first tabulated iteration after which the chain held the best graph (-1: none)
  int total_edges;
  int found;             // 0: no graph was a candidate yet
  int64_t from;          // D = max(drop, start iteration): a graph left at an iteration > D is a candidate
  int64_t born;          // iteration of the move that created the current graph (the start iteration at first)
  int n_dirty;           // length of list
  // set by the caller
  int n_sim;             // NsimEdges
  double phi, omega;
  int* par;              // [P][max_par] the best graph's lists: valid for every node outside the dirty set
  int* npar;             // [P]
  uint32_t* dirty;       // [W] nodes whose list changed since par / npar were last synchronised
  int* list;             // [P] the same set as a list, in marking order
};

// Posterior Markov blanket tabulation (ChainMem.mb; see mb_pairs), one per chain in global memory, set up by
// the caller (so that the chain itself carries one pointer for it).  Both matrices are symmetric.
struct MbTrack {
  int* freq;             // [i + j*P] iterations with (i, j) in the blanket (bn_run_args.mb_freq)
  uint16_t* wit;         // [i + j*P] witnesses of the pair: the edge between i and j, and each common child
};

struct ChainMem {  // per-chain global memory
  int* par;            // [P][max_par] ordered parent lists (edges[child])
  int* npar;           // [P]
  int* born;           // [P][max_par] first counted iteration of the edge (tabulation)
  double* base;        // [P] score of each node under the current graph
  double* fac;         // [P][fac_stride(fac_mp(max_par))] Cholesky factor of each node's parent set (score_core.cuh)
  double* rowbuf;      // [REPLAY_POS][row_stride(fac_mp(max_par))] candidate factor rows of the addition records
  uint32_t* anc;       // [P][Ws] ancestor bitsets
  uint32_t* haspar;    // [W] nodes with >= 1 parent (bitset)
  int* hp_list;        // [P] the same set as an ascending list (CurrOutputs, src/network.h:311-316)
  int* scratch;        // [scratch_words(P, ...)] row lists / dirty bitsets of the ancestor updates
  volatile int* helper;  // device only: command block of the CTA's helper warps (null = none)
  // outputs
  int* t_iter; int* t_changed; int* t_movetype; double* t_gll;
  int* t_add; int* t_del; int* t_fn; int* t_fp;
  int* moves;          // [moves_capacity][4]
  int* edge_freq;      // [parent + child*P] or null
  double* dscore;      // [P][max_par] cache of score(c | parents without slot e), NaN = unknown; or null
  int* npar_freq;      // [P][max_par + 1] iterations node p spent with k parents, or null
  int* npar_since;     // [P] first counted iteration of the node's current parent count
  // two-CTA pipeline (chain_pipe_kernel; device only, null otherwise)
  uint32_t* nver = nullptr;   // [P] accepted moves per node: the tag of the node's dscore entries -- with it
                              // dscore is [P][max_par] PAIRS (score, tag) and nothing is ever invalidated
  PipeLink* pipe = nullptr;        // mailbox shared with the peer CTA of the cluster
  int pipe_rank = 0;          // 0 = the chain's CTA, 1 = the record builder
  int pipe_debug = 0;         // (developer switch BN_B200_PIPE=3) 1: every window is rebuilt by the chain's own CTA
  // supplied start (chain_init; all null: the start graph of initial_network, scores computed)
  const int* start_par = nullptr;     // [P][max_par] ordered parent lists, -1 padded
  const int* start_npar = nullptr;    // [P]
  const ChainStart* start = nullptr;  // a resumed chain's scalars (null: iteration 0 of a fresh chain)
  const double* base_in = nullptr;    // [P] scores to start from; with it fac already holds the factors (MaxPar > 8)
  // posterior ancestor tabulation (anc_tab_*; null: off)
  int* anc_freq = nullptr;            // [ancestor + descendant*P] iterations with a directed path ancestor -> descendant
  // best graph visited (best_*; null: off)
  BestTrack* best = nullptr;
  // posterior Markov blanket tabulation (mb_*; null: off)
  MbTrack* mb = nullptr;
};

struct ChainScalars {  // lives in registers (warp-uniform)
  int64_t iter;        // next iteration index
  int64_t read_pos;    // committed uniform stream position
  int valid;           // stale `valid` flag, src/bayesnet_mcmc.cpp:40
  int te_m;            // member TotalEdges as left by the last LogPrior(), src/network.h:262-267
  int te_true, agree_true, n_haspar;
  // statistics: warp-uniform parts (sequential path) + lane-private parts (rounds: lane q adds
  // what the iteration in its slot contributes; summed over the lanes when the chain ends)
  int proposed[3], reject[3];
  int n_rows, n_moves, n_nonpd;
  int64_t valid_iters;
  int lane_prop[3], lane_rej[3], lane_nonpd, lane_valid;
  int64_t lane_bytes;
  int acc_add, acc_del;  // accepted moves since `drop`: the additions / deletions columns (src/network.h:340-341)
  int gll_ok; double gll;
  int64_t alg_bytes;   // sum over scored proposals of 8*(k'+1)(k'+2)/2 + 8 (SURVEY.md 8d)
  long long cyc[12];   // cycles per phase: refill, replay (A), score (B/C), commit, accepted add, accepted delete;
                       // [6..11] split the accepted moves: list update, ancestor test, ancestor team op (add 6-8, delete 9-11)
  long long slots_sim; // iterations replayed speculatively (committed + discarded)
  int win;             // current window size
  int windows;
  int need_full;       // the last round could not start: top the ring up completely before retrying
  int anc_changed;     // the last accepted move changed ancestor rows (else no cycle bit can differ)
  int next_log;        // smallest multiple of output_every >= s.iter (rounds; n_iter is an int)
  int status;
  // two-CTA pipeline (chain's CTA): first stream position of the window in ws (-1: none), the
  // outstanding request (number, position, in flight?), counters
  int64_t pw_cur, pw_out_pos;
  int pw_out_seq, pw_out;
  int pw_seen;         // accepted moves the records in ws have been repaired for
  int pw_waits, pw_discards, pw_rebuilds;
  long long pw_cyc[6];  // (diagnostics build) wait for the builder, copy, batch repair, redo after it, stale rebuilds, publish
};

struct WindowSlots {  // shared memory on the device
  int child[WIN], parent[WIN], pos[WIN], kk[WIN];
  int te_m[WIN], fp_m[WIN], fn_m[WIN];
  int64_t pos_after[WIN];
  double u_acc[WIN], new_score[WIN];
  signed char type[WIN], valid[WIN], do_check[WIN], accept[WIN], nonpd[WIN];
  // lane-parallel draw replay: outcome of a slot that would start at stream position pos + lane
  int t_c[REPLAY_POS], t_j[REPLAY_POS], t_e[REPLAY_POS];
  int t_rec[REPLAY_POS];   // REC_* bits
  double t_score[REPLAY_POS];  // score of the proposed parent set
  uint32_t t_full[REPLAY_POS]; // the (up to two) children the draw skipped for being at MaxPar, +1, 16 bits each
  double t_lu[REPLAY_POS];     // log of the acceptance uniform (accept test in log space)
  int t_walk[2 * REPLAY_POS];  // what the walk needs of the record, per incoming `valid` v (WALK_* bits);
                               // entries REPLAY_POS.. are WALK_END (a step is at most 255 positions)
  int s_k[WIN];     // walk result: record index of slot n (relative to the round start)
};

// Per-phase SM cycle counters (bn_chain_stats.phase_cycles) are a diagnostics build
// (-DBN_PHASE_CYCLES, BN_B200_DIAG=1 of build.py): reading the clock a dozen times per epoch costs
// the chain's warp a few percent, so the product build folds them to zero.
BN_HD long long cycle_now() {
#if defined(__CUDA_ARCH__) && defined(BN_PHASE_CYCLES)
  return clock64();
#else
  return 0;
#endif
}

// counters of the ancestor updates: host emulation builds with -DBN_EMU_STATS only (tests/tools)
#if defined(BN_EMU_STATS) && !defined(__CUDA_ARCH__)
struct EmuStats { long del_total, del_trivial, del_desc, del_rounds, del_rows_eval, del_lost_bits, add_total, add_trivial, add_desc; };
inline EmuStats& emu_stats() { static EmuStats s = {}; return s; }
#define BN_STAT(x) x
#else
#define BN_STAT(x)
#endif

BN_HD bool test_bit(const uint32_t* row, int b) { return (row[b >> 5] >> (b & 31)) & 1u; }

// LogPrior value from the integer counts, evaluated like src/network.h:277:
//   - phi * dist - omega * TotalEdges
BN_HD double prior_value(double phi, double omega, int dist, int total_edges) {
  return sub_rn(mul_rn(-phi, (double)dist), mul_rn(omega, (double)total_edges));
}

// number of set bits of a bitset strictly below position c, by the whole warp
BN_HD int rank_below(const uint32_t* bits, int c) {
  const int l = Warp::lane(), cw = c >> 5;
  int cnt = 0;
  for (int w = l; w <= cw; w += Warp::NL) {
    uint32_t word = bits[w];
    if (w == cw) word &= (1u << (c & 31)) - 1u;
    cnt += popc32(word);
  }
  return Warp::sum(cnt);
}

// keep hp_list (ascending nodes with >= 1 parent) in step with the haspar bitset
BN_HD void hp_insert(ChainMem& m, int n_before, int c) {
  const int l = Warp::lane();
  const int idx = rank_below(m.haspar, c);
  for (int hi = n_before; hi > idx; hi -= Warp::NL) {
    const int i = hi - 1 - l;
    const int v = (i >= idx) ? m.hp_list[i] : 0;
    Warp::sync();
    if (i >= idx) m.hp_list[i + 1] = v;
    Warp::sync();
  }
  if (l == 0) m.hp_list[idx] = c;
  Warp::sync();
}
BN_HD void hp_remove(ChainMem& m, int n_before, int c) {
  const int l = Warp::lane();
  const int idx = rank_below(m.haspar, c);
  for (int lo = idx; lo < n_before - 1; lo += Warp::NL) {
    const int i = lo + l;
    const int v = (i < n_before - 1) ? m.hp_list[i + 1] : 0;
    Warp::sync();
    if (i < n_before - 1) m.hp_list[i] = v;
    Warp::sync();
  }
}

// ---------------------------------------------------------------------------
// Ancestor bitsets.  Row d = ancestors of node d AND d itself (the reflexive closure: the
// equations become row[d] = {d} u U_q row[q] over the parents q, one plain OR per parent),
// Ws words apart (Ws % 4 == 0, 16 B aligned), processed in 128-bit chunks: `lpr` lanes share one row, so a warp updates
// `rpp` = 32/lpr rows per pass (4 rows for 1,000 nodes).
// ---------------------------------------------------------------------------
struct alignas(16) U4 { uint32_t x, y, z, w; };
BN_HD U4 or4(U4 a, U4 b) { U4 r; r.x = a.x | b.x; r.y = a.y | b.y; r.z = a.z | b.z; r.w = a.w | b.w; return r; }
BN_HD U4 andn4(U4 a, U4 b) { U4 r; r.x = a.x & ~b.x; r.y = a.y & ~b.y; r.z = a.z & ~b.z; r.w = a.w & ~b.w; return r; }
BN_HD U4 and4(U4 a, U4 b) { U4 r; r.x = a.x & b.x; r.y = a.y & b.y; r.z = a.z & b.z; r.w = a.w & b.w; return r; }
BN_HD bool nz4(U4 a) { return (a.x | a.y | a.z | a.w) != 0u; }
BN_HD bool ne4(U4 a, U4 b) { return ((a.x ^ b.x) | (a.y ^ b.y) | (a.z ^ b.z) | (a.w ^ b.w)) != 0u; }
BN_HD int popc4(U4 a) { return popc32(a.x) + popc32(a.y) + popc32(a.z) + popc32(a.w); }
BN_HD U4 with_bit(U4 v, int b) {  // set bit b (0..127) of the chunk
  const uint32_t m = 1u << (b & 31);
  const int w = b >> 5;
  v.x |= (w == 0) ? m : 0u; v.y |= (w == 1) ? m : 0u; v.z |= (w == 2) ? m : 0u; v.w |= (w == 3) ? m : 0u;
  return v;
}

struct RowGeom { int chunks, lpr, rpp; };
// computed once per chain (the device and the one-lane host build differ in Warp::NL)
BN_HD void set_row_geom(ChainParams& p) {
  p.g_chunks = (p.W + 3) / 4;
  p.g_lpr = 1;
  while (p.g_lpr < p.g_chunks && p.g_lpr < Warp::NL) p.g_lpr <<= 1;
  p.g_rpp = Warp::NL / p.g_lpr;
}
BN_HD RowGeom row_geom(const ChainParams& p) {
  RowGeom g;
  g.chunks = p.g_chunks; g.lpr = p.g_lpr; g.rpp = p.g_rpp;
  return g;
}

BN_HD int group_sum(int v, int lpr) {  // sum over the lpr lanes that share a row
#if defined(__CUDA_ARCH__)
  for (int o = 1; o < lpr; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
#else
  (void)lpr;
#endif
  return v;
}

BN_HD int atomic_fetch_inc(int* p) {
#if defined(__CUDA_ARCH__)
  return atomicAdd(p, 1);
#else
  return (*p)++;
#endif
}

BN_HD uint32_t atomic_or_u32(uint32_t* p, uint32_t v) {
#if defined(__CUDA_ARCH__)
  return atomicOr(p, v);
#else
  const uint32_t o = *p; *p = o | v; return o;
#endif
}

// most rows one warp can own under the block-cyclic partition (blocks of nl rows)
BN_HD int rows_per_part(int P, int nparts, int nl) {
  const int nblk = (P + nl - 1) / nl;
  return (nblk + nparts - 1) / nparts * nl;
}
// per-chain scratch (ints) of the ancestor updates.  anc_add_part: one row list per warp.
// anc_del_team: two row lists per warp, the lost-ancestor bitset, three dirty bitsets and four
// round flags (del_layout).
BN_HD int scratch_words(int P, int nparts, int nl) {
  const int W = (P + 31) / 32;
  const int n = 2 * rows_per_part(P, nparts, nl) * nparts + 4 + (W + 3) / 4 * 4 + 3 * W + 4 + 1 + (W + 3) / 4 + 28;
  return (n + 3) / 4 * 4;  // keeps every chain's block 16-byte aligned
}

// nodes that have c as an ancestor (ascending), optionally c itself as well: the share of
// `part` under a block-cyclic partition of the rows (blocks of Warp::NL rows; descendants
// cluster in index ranges, contiguous ranges would leave most of the work to one warp)
BN_HD int collect_desc_part(const ChainParams& p, const ChainMem& m, int c, int include_self, int* list,
                            int part, int nparts) {
  const int l = Warp::lane();
  const uint32_t Ws = (uint32_t)p.Ws, cb = (uint32_t)c & 31u;
  const uint32_t* col = m.anc + (c >> 5);  // word (c >> 5) of every row
  const uint32_t lt = (1u << l) - 1u;
  int n = 0;
  const int step = nparts * Warp::NL;
  for (int d0 = part * Warp::NL; d0 < p.P; d0 += 4 * step) {  // four independent column loads in flight
    int d[4], flag[4];
#pragma unroll
    for (int t = 0; t < 4; t++) {
      d[t] = d0 + t * step + l;
      flag[t] = 0;
      if (d[t] < p.P) flag[t] = ((col[(uint32_t)d[t] * Ws] >> cb) & 1u) & ((include_self || d[t] != c) ? 1u : 0u);
    }
#pragma unroll
    for (int t = 0; t < 4; t++) {
      const uint32_t mask = Warp::ballot(flag[t]);
      if (flag[t]) list[n + popc32(mask & lt)] = d[t];
      n += popc32(mask);
    }
  }
  Warp::sync();
  return n;
}

// after adding parent j to child c: every node in {c} u desc(c) gains anc[j] u {j}
// (one warp's share of the rows; everything on the host)
BN_HD void anc_add_part(const ChainParams& p, const ChainMem& m, int j, int c, int* list, int part, int nparts) {
  const RowGeom g = row_geom(p);
  const int l = Warp::lane(), sub = l / g.lpr, li = l % g.lpr;
  const int n = collect_desc_part(p, m, c, 1, list, part, nparts);
  BN_STAT(emu_stats().add_desc += n;)
  const U4* aj = (const U4*)(m.anc + (uint32_t)j * (uint32_t)p.Ws);
  if (g.chunks == 8 && Warp::NL == 32) {
    // 897..1,024 nodes: 8 lanes per row, 4 rows per pass, four passes in flight.  A pass index
    // behind the list repeats the lane group's first row (the OR is idempotent), so the loop
    // body carries no predicates.
    const int sub8 = l >> 3, li8 = l & 7;
    const U4 a = aj[li8];  // row j holds j itself
    for (int r0 = sub8; r0 < n; r0 += 16) {
      U4* ad[4];
      U4 v[4];
#pragma unroll
      for (int t = 0; t < 4; t++) {
        const int r = (r0 + 4 * t < n) ? r0 + 4 * t : r0;
        ad[t] = (U4*)(m.anc + (uint32_t)list[r] * (uint32_t)p.Ws) + li8;
      }
#pragma unroll
      for (int t = 0; t < 4; t++) v[t] = *ad[t];
#pragma unroll
      for (int t = 0; t < 4; t++) *ad[t] = or4(v[t], a);
    }
  } else if (g.chunks <= g.lpr) {
    // one 128-bit chunk per lane (up to 4,096 nodes): the source chunk stays in registers
    U4 a = {0u, 0u, 0u, 0u};
    if (li < g.chunks) {
      a = aj[li];  // row j holds j itself
    }
    for (int r0 = 0; r0 < n; r0 += 4 * g.rpp) {  // four rows in flight per lane group
      U4* ad[4];
      U4 v[4];
#pragma unroll
      for (int t = 0; t < 4; t++) {
        const int r = r0 + t * g.rpp + sub;
        ad[t] = (r < n && li < g.chunks) ? (U4*)(m.anc + (uint32_t)list[r] * (uint32_t)p.Ws) + li : nullptr;
      }
#pragma unroll
      for (int t = 0; t < 4; t++) if (ad[t]) v[t] = *ad[t];
#pragma unroll
      for (int t = 0; t < 4; t++) if (ad[t]) *ad[t] = or4(v[t], a);
    }
  } else {
    for (int r0 = 0; r0 < n; r0 += g.rpp) {
      const int r = r0 + sub;
      if (r < n) {
        U4* ad = (U4*)(m.anc + (int64_t)list[r] * p.Ws);
        for (int ch = li; ch < g.chunks; ch += g.lpr) {
          ad[ch] = or4(ad[ch], aj[ch]);
        }
      }
    }
  }
  Warp::sync();
}

// The CTA of a chain has HELPER_WARPS extra warps parked on a named barrier; they take an
// equal share of the rows of an ancestor update (the scan and the ORs are independent per row).
constexpr int HELPER_WARPS = 7;
enum { HELPER_EXIT = 0, HELPER_ANC_ADD = 1, HELPER_RECORDS = 2, HELPER_REPAIR = 3, HELPER_ANC_DEL = 4,
       HELPER_FILL_WH = 5, HELPER_PIPE_COPY = 6, HELPER_REPAIR_BATCH = 7 };
// command block (ints): [0] op, [1..2] stream position, [3..4] ring limit, [5] n_haspar,
// [6] TotalEdges, [7] Nagree, [8] node / parent, [9] child, [10] span limit (atomicMin target),
// [11] child dropped below MaxPar
constexpr int HELPER_WORDS = 12;
#if defined(__CUDACC__)
__device__ __forceinline__ void cta_bar(int id) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"((HELPER_WARPS + 1) * 32) : "memory");
}
#endif
// ---------------------------------------------------------------------------
// Two-CTA pipeline (chain_pipe_kernel in kernels.cu; MaxPar <= 8 with the whole state in shared
// memory).  A chain is a thread-block CLUSTER of two CTAs on two SMs:
//   rank 0  the chain: walks the records, commits, applies the accepted moves -- everything the
//           single-CTA kernel does except building the records of a window;
//   rank 1  the record builder: keeps a REPLICA of the graph state (parent lists, ancestor
//           bitsets, scores, its own copy of the uniform stream) by applying the accepted moves
//           the chain publishes, and builds the 256 position records of the NEXT window while the
//           chain is busy with the current one.
// A window is picked up by copying its records over distributed shared memory; it was built when
// the replica had applied a known number of moves, so the chain repairs it for the moves accepted since
// (repair_record_batch: the same rules as the in-round repair, applied for a list of moves), and
// from there on everything is the single-CTA round.  Windows sit on a 256-position grid; a stale
// record under the walk is rebuilt in place by the chain's own CTA.
// Mailboxes: each CTA polls its OWN shared memory; the peer writes into it with remote stores
// (mapa + st.shared::cluster).
// ---------------------------------------------------------------------------
constexpr int PIPE_WIN = HELPER_WARPS * 32;  // stream positions per window: one record per HELPER thread.  In this
                               // form the chain warps only direct (walk, commit, mailbox): every team operation is
                               // executed by the seven helper warps alone, so each SM runs ONE copy of its code
                               // (the one-CTA kernel keeps a second, inlined copy for warp 0 -- the instruction
                               // cache is what limits these kernels)
constexpr int PIPE_MQ = 64;    // accepted moves in flight between the two CTAs (back-pressure beyond)
constexpr int PIPE_LOG = 128;  // recent moves the chain remembers for the windows it picks up
// Every message is ONE store of at most 16 bytes that carries its own sequence number, so no message
// needs a second store to become valid and nothing depends on the order in which remote stores land
// (st.release.cluster compiles to MEMBAR.ALL.GPU on sm_100a: ~1,000 cycles per accepted move).
struct PipeLink {
  // written by the chain's CTA into the BUILDER's copy
  unsigned long long req;      // window request: (first stream position << 16) | (request number & 0xffff)
  int req_exit;
  int pad0;
  // written by the builder into the CHAIN's copy
  unsigned long long rdy;      // window completed: (moves the replica had applied << 32) | its request number
  int mq_tail;                 // moves the builder has taken out of the queue
  int pad1;
  // accepted moves (builder's copy): [0] move number + 1, [1] child | parent << 11 | (type - 1) << 22 |
  // deletion slot << 23 | in-prior << 26 | (move number + 1) << 27, [2..3] the child's new score
  alignas(16) int mq[PIPE_MQ][4];
  int log[PIPE_LOG];           // (chain's copy) node | dropped below MaxPar << 24 | ancestor rows changed << 25 |
                               // set of nodes with parents changed << 26
};
constexpr int PIPE_MAX_NODES = 2048;  // 11-bit node numbers in a move message
constexpr int LOG_NODE = 0xffffff, LOG_UNFULL = 1 << 24, LOG_ANC = 1 << 25, LOG_HP = 1 << 26;

#if defined(__CUDACC__)
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t peer_addr(const void* p, int rank) {  // the same variable in CTA `rank` of the cluster
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr(p)), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_peer(uint32_t a, int v) {
  asm volatile("st.relaxed.cluster.shared::cluster.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory");
}
__device__ __forceinline__ void st_peer64(uint32_t a, unsigned long long v) {
  asm volatile("st.relaxed.cluster.shared::cluster.b64 [%0], %1;" ::"r"(a), "l"(v) : "memory");
}
__device__ __forceinline__ void st_peer128(uint32_t a, int x, int y, int z, int w) {
  asm volatile("st.shared::cluster.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
// polls of this CTA's own mailbox (the peer writes it remotely)
__device__ __forceinline__ int ld_poll(const int* p) {
  int v;
  asm volatile("ld.volatile.shared.b32 %0, [%1];" : "=r"(v) : "r"(smem_addr(p)) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long ld_poll64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.volatile.shared.b64 %0, [%1];" : "=l"(v) : "r"(smem_addr(p)) : "memory");
  return v;
}
__device__ __forceinline__ void ld_poll128(const int* p, int& x, int& y, int& z, int& w) {
  asm volatile("ld.volatile.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(x), "=r"(y), "=r"(z), "=r"(w) : "r"(smem_addr(p)) : "memory");
}
__device__ __forceinline__ int ld_peer(uint32_t a) {
  int v;
  asm volatile("ld.shared::cluster.b32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ long long ld_peer64(uint32_t a) {
  long long v;
  asm volatile("ld.shared::cluster.b64 %0, [%1];" : "=l"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// chain's CTA, lane 0: hand accepted move number `n` to the builder and remember it locally
__device__ __forceinline__ void pipe_publish(const ChainMem& m, int n, int type, int c, int j, int del, int ag,
                                             double score, int flags) {
  PipeLink* lk = m.pipe;
  for (long long spins = 0; n - ld_poll(&lk->mq_tail) >= PIPE_MQ; spins++)
    if (spins > (1ll << 27)) { lk->pad1 = 92; break; }  // (watchdog: the builder is gone -- run_chain reports it)
  const long long sb = __double_as_longlong(score);
  st_peer128(peer_addr(&lk->mq[n % PIPE_MQ][0], 1), n + 1,
             c | (j << 11) | ((type - 1) << 22) | (del << 23) | (ag << 26) | ((n + 1) << 27),
             (int)(sb & 0xffffffffll), (int)(sb >> 32));
  lk->log[n % PIPE_LOG] = c | flags;
}
#endif

// barrier between the rounds of a team operation (all warps of the CTA, or just this warp)
BN_HD void team_sync(const ChainMem& m) {
#if defined(__CUDA_ARCH__)
  if (m.helper) { cta_bar(3); return; }
#endif
  (void)m;
  Warp::sync();
}

BN_HD void anc_after_add(const ChainParams& p, ChainMem& m, int j, int c, int& m_anc_changed) {
  {
    // j (and with it all its ancestors) already an ancestor of c: row j is contained in row c and
    // in the row of every descendant of c -- nothing changes (a redundant edge, common in a
    // dense graph)
    const RowGeom g = row_geom(p);
    const U4* aj = (const U4*)(m.anc + (uint32_t)j * (uint32_t)p.Ws);
    const U4* ac = (const U4*)(m.anc + (uint32_t)c * (uint32_t)p.Ws);
    int news = 0;
    for (int ch = Warp::lane(); ch < g.chunks; ch += Warp::NL) news |= nz4(andn4(aj[ch], ac[ch])) ? 1 : 0;
    BN_STAT(emu_stats().add_total++;)
    if (Warp::ballot(news) == 0u) { BN_STAT(emu_stats().add_trivial++;) m_anc_changed = 0; return; }
  }
  m_anc_changed = 1;
#if defined(__CUDA_ARCH__)
  if (m.helper) {
    if (Warp::lane() == 0) { m.helper[8] = j; m.helper[9] = c; m.helper[0] = HELPER_ANC_ADD; }
    Warp::sync();
    cta_bar(1);
    if (!m.pipe) anc_add_part(p, m, j, c, m.scratch, 0, HELPER_WARPS + 1);  // (two-CTA form: the helper warps own all rows)
    cta_bar(2);
    return;
  }
#else
  anc_add_part(p, m, j, c, m.scratch, 0, 1);
#endif
}


// parents of node d as eight slots (-1 = empty); two 128-bit loads when MaxPar == 8
struct Par8 { int q[8]; };
BN_HD Par8 load_par8(const ChainParams& p, const ChainMem& m, int d) {
  Par8 r;
  const int* pd = m.par + (int64_t)d * p.max_par;
  if (p.max_par == 8) {
    const U4 a = ((const U4*)pd)[0], b = ((const U4*)pd)[1];
    r.q[0] = (int)a.x; r.q[1] = (int)a.y; r.q[2] = (int)a.z; r.q[3] = (int)a.w;
    r.q[4] = (int)b.x; r.q[5] = (int)b.y; r.q[6] = (int)b.z; r.q[7] = (int)b.w;
  } else {
#pragma unroll
    for (int e = 0; e < 8; e++) r.q[e] = (e < p.max_par) ? pd[e] : -1;
  }
  return r;
}

// after removing a parent of child c (par[c] already updated).  The new row of c follows from
// its remaining parents; L = old row & ~new row are the ancestors c lost.  If L is empty nothing
// changes anywhere (the common case in a graph with redundant paths).  Otherwise only bits of L
// can disappear, and only from rows of desc(c).  Those rows are first cleared of L (a lower
// bound of the truth), then the ancestor equations anc[d] = U_q (anc[q] u {q}) over the parents
// q of d are iterated UPWARDS on the bits of L: round 0 evaluates every descendant, round r
// those with a parent that regained a bit in round r-1.  In a DAG the equations have one
// solution and the iteration reaches it from below; most descendants lose L for good, so the
// regain wave is short (a few rounds) where a downward relaxation needs one round per level of
// the loss wave.  Rows are owned by warps (block-cyclic); a row read while its owner updates
// it yields a subset of its final value, which is harmless: the owner marks it dirty and the
// reader is evaluated again next round.
struct DelLayout { int* lists; U4* L; uint32_t* dirty; volatile int* flags; int* nzc; int per; };
BN_HD DelLayout del_layout(const ChainParams& p, const ChainMem& m, int nparts) {
  DelLayout d;
  d.per = rows_per_part(p.P, nparts, Warp::NL);
  int off = (2 * d.per * nparts + 3) / 4 * 4;
  d.lists = m.scratch;
  d.L = (U4*)(m.scratch + off);
  off += (p.W + 3) / 4 * 4;
  d.dirty = (uint32_t*)(m.scratch + off);
  d.flags = (volatile int*)(d.dirty + 3 * p.W);
  d.nzc = (int*)(d.dirty + 3 * p.W + 4);  // [0] = number of chunks where L != 0, then their indices
  return d;
}

BN_HD int anc_del_team(const ChainParams& p, const ChainMem& m, int c, int part, int nparts, long long* dbg = nullptr) {
  const int l = Warp::lane(), W = p.W, MP = p.max_par;
  const DelLayout lay = del_layout(p, m, nparts);
  int* list = lay.lists + (part < 0 ? 0 : part) * 2 * lay.per;
  int* list2 = list + lay.per;
  const long long td0 = cycle_now();
  // (part < 0, two-CTA form: the chain's warp has no rows of its own -- it keeps the round barriers and the bookkeeping)
  const int n = part < 0 ? 0 : collect_desc_part(p, m, c, 0, list, part, nparts);  // old column c: rows this warp owns
  BN_STAT(emu_stats().del_desc += n;)
  const uint32_t lt = (l == 31) ? 0x7fffffffu : ((1u << l) - 1u);
  // L is usually confined to one or two 128-bit chunks: a lane takes one (row, non-zero chunk)
  // pair, so a pass covers 32 / lpr rows with lpr = nnz rounded up to a power of two
  const int nnz = lay.nzc[0];
  int lpr = 1;
  while (lpr < nnz && lpr < Warp::NL) lpr <<= 1;
  const int rpp = Warp::NL / lpr, sub = l / lpr, li = l % lpr;
  const uint32_t gm = (lpr >= 32 ? 0xffffffffu : ((1u << lpr) - 1u)) << (sub * lpr);
  // clear L from the rows of the descendants
  for (int r0 = 0; r0 < n; r0 += rpp) {
    const int r = r0 + sub;
    if (r < n) {
      U4* ad = (U4*)(m.anc + (uint32_t)list[r] * (uint32_t)p.Ws);
      for (int t = li; t < nnz; t += lpr) {
        const int ch = lay.nzc[1 + t];
        ad[ch] = andn4(ad[ch], lay.L[ch]);
      }
    }
  }
  const long long td1 = cycle_now();
  team_sync(m);
  const long long td2 = cycle_now();
  if (dbg) { dbg[6] += td1 - td0; dbg[7] += td2 - td1; }
  int rounds_done = 0;
  for (int round = 0;; round++) {
    const long long tr0 = cycle_now();
    const uint32_t* dprev = lay.dirty + (round % 3) * W;
    uint32_t* dnext = lay.dirty + ((round + 1) % 3) * W;
    if (part <= 0 && (part < 0 || !m.pipe)) {  // nobody reads or writes these during this round
      uint32_t* dclr = lay.dirty + ((round + 2) % 3) * W;
      for (int w = l; w < W; w += Warp::NL) dclr[w] = 0u;
      if (l == 0) lay.flags[(round + 2) % 4] = 0;
    }
    const int* rows = list;
    int nt = n;
    if (round > 0) {
      // rows with a parent that regained a bit last round
      rows = list2;
      nt = 0;
      for (int i0 = 0; i0 < n; i0 += Warp::NL) {
        const int i = i0 + l;
        const int d = (i < n) ? list[i] : -1;
        int touched = 0;
        if (d >= 0) {
          if (MP <= 8) {
            // unused slots of a parent list hold -1: all eight dirty words load independently
            const Par8 pq = load_par8(p, m, d);
#pragma unroll
            for (int e = 0; e < 8; e++)
              if (pq.q[e] >= 0) touched |= (dprev[pq.q[e] >> 5] >> (pq.q[e] & 31)) & 1u;
          } else {
            const int kd = m.npar[d];
            const int* pd = m.par + (int64_t)d * MP;
            for (int e = 0; e < kd; e++) {
              const int q = pd[e];
              touched |= (dprev[q >> 5] >> (q & 31)) & 1u;
            }
          }
        }
        const uint32_t mask = Warp::ballot(touched);
        if (touched) list2[nt + popc32(mask & lt)] = d;
        nt += popc32(mask);
      }
      Warp::sync();
    }
    int any = 0;
    BN_STAT(emu_stats().del_rounds++; emu_stats().del_rows_eval += nt;)
    for (int r0 = 0; r0 < nt; r0 += rpp) {
      const int r = r0 + sub;
      int changed = 0, d = 0;
      if (r < nt) {
        d = rows[r];
        U4* ad = (U4*)(m.anc + (uint32_t)d * (uint32_t)p.Ws);
        for (int t = li; t < nnz; t += lpr) {
          const int ch = lay.nzc[1 + t];
          const U4 Lc = lay.L[ch];
          U4 v = {0u, 0u, 0u, 0u};
          if (MP <= 8) {
            const Par8 pq = load_par8(p, m, d);
#pragma unroll
            for (int e = 0; e < 8; e++) {
              const int q = pq.q[e];
              if (q >= 0) v = or4(v, ((const U4*)(m.anc + (uint32_t)q * (uint32_t)p.Ws))[ch]);
            }
          } else {
            const int kd = m.npar[d];
            const int* pd = m.par + (int64_t)d * MP;
            for (int e = 0; e < kd; e++) {
              const int q = pd[e];
              v = or4(v, ((const U4*)(m.anc + (int64_t)q * p.Ws))[ch]);
            }
          }
          const U4 cur = ad[ch];
          const U4 gain = andn4(and4(v, Lc), cur);
          if (nz4(gain)) { ad[ch] = or4(cur, gain); changed = 1; }
        }
      }
      const uint32_t mask = Warp::ballot(changed);
      if (r < nt && li == 0 && (mask & gm)) atomic_or_u32(&dnext[d >> 5], 1u << (d & 31));
      any |= (mask != 0u);
      Warp::sync();  // later passes of this warp see the new rows
    }
    if (any && l == 0) lay.flags[round % 4] = 1;
    const long long tr1 = cycle_now();
    team_sync(m);
    if (dbg) { dbg[8] += tr1 - tr0; dbg[11] += cycle_now() - tr1; }
    rounds_done++;
    if (lay.flags[round % 4] == 0) break;
  }
  return rounds_done;
}

BN_HD void anc_after_delete(const ChainParams& p, ChainMem& m, int c, int& m_anc_changed, long long* dbg = nullptr) {
  const RowGeom g = row_geom(p);
  const int l = Warp::lane();
  int nparts = 1;
#if defined(__CUDA_ARCH__)
  if (m.helper) nparts = m.pipe ? HELPER_WARPS : HELPER_WARPS + 1;
#endif
  const DelLayout lay = del_layout(p, m, nparts);
  {
    // new row of c from its remaining parents (a subset of the old row); L = what it lost
    U4* ac = (U4*)(m.anc + (int64_t)c * p.Ws);
    const int* pc = m.par + (int64_t)c * p.max_par;
    const int kc = m.npar[c];
    int changed = 0;
    for (int ch = l; ch < g.chunks; ch += Warp::NL) {
      U4 v = {0u, 0u, 0u, 0u};
      if (ch == (c >> 7)) v = with_bit(v, c & 127);
      for (int e = 0; e < kc; e++) {
        const int q = pc[e];
        v = or4(v, ((const U4*)(m.anc + (int64_t)q * p.Ws))[ch]);
      }
      const U4 lost = andn4(ac[ch], v);
      lay.L[ch] = lost;
      if (nz4(lost)) { ac[ch] = v; changed = 1; }
    }
    BN_STAT(emu_stats().del_total++;)
    if (Warp::ballot(changed) == 0u) { BN_STAT(emu_stats().del_trivial++;) m_anc_changed = 0; return; }
  }
  m_anc_changed = 1;
  BN_STAT(for (int ch = 0; ch < g.chunks; ch++) emu_stats().del_lost_bits += popc4(lay.L[ch]);)
  for (int w = l; w < 3 * p.W + 4; w += Warp::NL) lay.dirty[w] = 0u;  // three bitsets + four flags
  Warp::sync();
  {
    // indices of the chunks where something was lost
    const uint32_t lt = (l == 31) ? 0x7fffffffu : ((1u << l) - 1u);
    int nnz = 0;
    for (int ch0 = 0; ch0 < g.chunks; ch0 += Warp::NL) {
      const int ch = ch0 + l;
      const int nz = (ch < g.chunks) && nz4(lay.L[ch]);
      const uint32_t mask = Warp::ballot(nz);
      if (nz) lay.nzc[1 + nnz + popc32(mask & lt)] = ch;
      nnz += popc32(mask);
    }
    if (l == 0) lay.nzc[0] = nnz;
    Warp::sync();
  }
#if defined(__CUDA_ARCH__)
  if (m.helper) {
    if (l == 0) { m.helper[9] = c; m.helper[0] = HELPER_ANC_DEL; }
    Warp::sync();
    cta_bar(1);
    anc_del_team(p, m, c, m.pipe ? -1 : 0, nparts, dbg);
    cta_bar(2);
    return;
  }
#else
  anc_del_team(p, m, c, 0, 1);
#endif
}

// ---------------------------------------------------------------------------
// Posterior ancestor tabulation (ChainMem.anc_freq): anc_freq[a + d*P] counts the iterations, from
// max(drop, iter) on, after which the graph has a directed path a -> ... -> d, i.e. bit a of row d.
// No birth iteration per bit: the count is accumulated with signs.  A bit that turns on at
// iteration t subtracts max(t, drop), one that turns off adds it, and the end of the run adds
// max(end, drop) for every bit still set.  Only accepted moves flip bits (apply_move_vals), and they
// flip only these, in the rows of {c} u desc(c) (the rows holding bit c; desc(c) does not change):
//   addition j -> c   gain N & ~row, N = anc(j) & ~anc(c), read before the update (anc_tab_add)
//   deletion at c     lose L & ~row, L = old anc(c) & ~new anc(c), read after it (anc_tab_del)
// Lanes take (row, chunk) pairs; distinct lanes own distinct counters, so no atomics are needed.
// ---------------------------------------------------------------------------
// v added for every set bit of every row (chain start: -max(drop, iter); end: max(end, drop))
BN_HD void anc_tab_all(const ChainParams& p, const ChainMem& m, int v) {
  const int l = Warp::lane(), P = p.P, W = p.W;
  for (int64_t i = l; i < (int64_t)P * W; i += Warp::NL) {
    const int d = (int)(i / W), w = (int)(i - (int64_t)d * W);
    int* out = m.anc_freq + (int64_t)d * P + 32 * w;
    for (uint32_t b = m.anc[(int64_t)d * p.Ws + w]; b; b &= b - 1u) out[ffs32(b) - 1] += v;
  }
  Warp::sync();
}

// the lost / gained sets live where anc_after_delete keeps L: the chunks lay.L[lay.nzc[1..nnz]]
BN_HD DelLayout anc_tab_layout(const ChainParams& p, const ChainMem& m) {
  int nparts = 1;
#if defined(__CUDA_ARCH__)
  if (m.helper) nparts = m.pipe ? HELPER_WARPS : HELPER_WARPS + 1;
#endif
  return del_layout(p, m, nparts);
}

// v added at (bit a, row d) for every row d holding bit c and every bit a of L & ~row d, L = the chunks
// L4[nzc[1..nnz]].  The rows are first listed (`rows`: lay.lists, free outside the team operations), then
// lanes take (listed row, 32-bit word of a non-zero chunk) pairs, so that one row with many flipped bits (a
// sink gaining a long ancestry) is still spread over lanes.  A lane reads up to eight of its counters before
// it writes them back: the loads are independent and overlap instead of paying a memory round trip per bit.
// Not inlined: its registers (the eight counters in flight) would otherwise raise the register pressure of
// the whole chain loop of the WITH_STATE kernels, which resumable runs without the tabulation share.
BN_NOINLINE void anc_tab_flip(const uint32_t* anc, int Ws, int P, int* anc_freq, int c, const uint32_t* Lw,
                              const int* nzc, int nnz, int* rows, int v) {
  const int l = Warp::lane(), nw = 4 * nnz;
  const uint32_t lt = (l == 31) ? 0x7fffffffu : ((1u << l) - 1u);
  int n = 0;
  for (int d0 = 0; d0 < P; d0 += Warp::NL) {
    const int d = d0 + l;
    const int has = d < P && test_bit(anc + (uint32_t)d * (uint32_t)Ws, c);
    const uint32_t mask = Warp::ballot(has);
    if (has) rows[n + popc32(mask & lt)] = d;
    n += popc32(mask);
  }
  Warp::sync();
  for (int i = l; i < n * nw; i += Warp::NL) {
    const int r = i / nw, k = i - r * nw, d = rows[r];
    const int wd = 4 * nzc[1 + (k >> 2)] + (k & 3);  // word of the row
    uint32_t b = Lw[wd] & ~anc[(uint32_t)d * (uint32_t)Ws + wd];
    int* out = anc_freq + (int64_t)d * P + 32 * wd;
    while (b) {
      int idx[8], x[8];
#pragma unroll
      for (int t = 0; t < 8; t++) { idx[t] = b ? ffs32(b) - 1 : -1; b &= b - 1u; }
#pragma unroll
      for (int t = 0; t < 8; t++) if (idx[t] >= 0) x[t] = out[idx[t]];
#pragma unroll
      for (int t = 0; t < 8; t++) if (idx[t] >= 0) out[idx[t]] = x[t] + v;
    }
  }
  Warp::sync();
}
BN_HD void anc_tab_rows(const ChainParams& p, const ChainMem& m, int c, const DelLayout& lay, int nnz, int v) {
  anc_tab_flip(m.anc, p.Ws, p.P, m.anc_freq, c, (const uint32_t*)lay.L, lay.nzc, nnz, lay.lists, v);
}

// accepted addition j -> c, BEFORE anc_after_add: the bits N = anc(j) & ~anc(c) that rows of {c} u desc(c)
// gain turn on at iteration first_counted (v = -max(t, drop)).  N = 0: a redundant edge, nothing changes.
BN_HD void anc_tab_add(const ChainParams& p, const ChainMem& m, int j, int c, int v) {
  const RowGeom g = row_geom(p);
  const int l = Warp::lane();
  const DelLayout lay = anc_tab_layout(p, m);
  const U4* aj = (const U4*)(m.anc + (uint32_t)j * (uint32_t)p.Ws);
  const U4* ac = (const U4*)(m.anc + (uint32_t)c * (uint32_t)p.Ws);
  const uint32_t lt = (l == 31) ? 0x7fffffffu : ((1u << l) - 1u);
  int nnz = 0;
  for (int ch0 = 0; ch0 < g.chunks; ch0 += Warp::NL) {
    const int ch = ch0 + l;
    U4 n = {0u, 0u, 0u, 0u};
    if (ch < g.chunks) n = andn4(aj[ch], ac[ch]);
    const int nz = nz4(n);
    const uint32_t mask = Warp::ballot(nz);
    if (nz) { lay.L[ch] = n; lay.nzc[1 + nnz + popc32(mask & lt)] = ch; }
    nnz += popc32(mask);
  }
  Warp::sync();
  if (nnz) anc_tab_rows(p, m, c, lay, nnz, v);
}

// accepted deletion at c, AFTER anc_after_delete changed rows (s.anc_changed): the bits of L that rows of
// {c} u desc(c) no longer hold turn off (v = +max(t, drop)).  anc_del_team reads L and nzc but never
// writes them, so they are still those of this deletion.
BN_HD void anc_tab_del(const ChainParams& p, const ChainMem& m, int c, int v) {
  const DelLayout lay = anc_tab_layout(p, m);
  anc_tab_rows(p, m, c, lay, lay.nzc[0], v);
}

// Lane l sums p = l, l+32, ... ascending, then a fixed-order tree: deterministic (sum_base: globalLL).
BN_HD double sum_scores(const double* base, int P) {
  double acc = 0.0;
  for (int c = Warp::lane(); c < P; c += Warp::NL) acc += base[c];
  return Warp::sum(acc);
}

// ---------------------------------------------------------------------------
// Best graph visited (ChainMem.best): the graph with the highest log_lik + log_prior among the graphs
// edge_freq counts.  With D = max(drop, iter0), a graph created at iteration t and replaced at t' (or held
// to the end of the call) is counted iff t' > D (end > D).  log_lik is the graph's globalLL (sum_scores of
// the score cache); log_prior is prior_value of its FP + FN and TotalEdges.  A later graph replaces the best
// only when strictly greater: the first to reach the maximum wins.  Its `iter` is max(t, D).
// No copy of the graph per new best: BestTrack.par / npar equal the current lists of every node outside
// the dirty set, whose members are the nodes accepted moves changed since the last new best.  A new best
// copies the dirty nodes' lists and empties the set; so par / npar always hold the best graph.
// ---------------------------------------------------------------------------
BN_HD void best_init(const ChainParams& p, const ChainMem& m, int64_t it0, int64_t from) {
  const int l = Warp::lane(), MP = p.max_par;
  BestTrack& b = *m.best;
  for (int64_t i = l; i < (int64_t)p.P * MP; i += Warp::NL) b.par[i] = m.par[i];
  for (int i = l; i < p.P; i += Warp::NL) b.npar[i] = m.npar[i];
  for (int w = l; w < p.W; w += Warp::NL) b.dirty[w] = 0u;
  Warp::sync();
  if (l == 0) {
    b.log_post = b.log_lik = b.log_prior = -INFINITY;
    b.iter = -1; b.total_edges = 0; b.found = 0;
    b.from = from; b.born = it0; b.n_dirty = 0;
  }
  Warp::sync();
}

// The current graph is about to be left after iteration `it` (c >= 0: an accepted move at node c, called
// before it changes anything) or held at the end of the call (c = -1, it = end).  With it > D the graph is a
// candidate: its log_lik is *gll when gll_ok, else sum_scores, left in *gll (returns 1 then: the caller keeps
// it as its globalLL, the graph has not changed).  Not inlined: resumable runs without the tracking keep
// the instruction-cache footprint of their chain loop.
BN_NOINLINE int best_visit(BestTrack* bt, const double* base, const int* par, const int* npar, int P, int MP,
                           int te, int ag, int64_t it, int c, int gll_ok, double* gll) {
  const int l = Warp::lane();
  int computed = 0;
  const int64_t D = bt->from;
  int* bpar = bt->par; int* bnpar = bt->npar; uint32_t* dirty = bt->dirty; int* list = bt->list;
  if (it > D) {
    double ll = *gll;
    if (!gll_ok) { ll = sum_scores(base, P); *gll = ll; computed = 1; }
    const double lpr = prior_value(bt->phi, bt->omega, (te - ag) + (bt->n_sim - ag), te);
    const double lp = add_rn(ll, lpr);
    if (!bt->found || lp > bt->log_post) {
      const int nd = bt->n_dirty;
      for (int i = l; i < nd; i += Warp::NL) {
        const int d = list[i];
        bnpar[d] = npar[d];
        for (int e = 0; e < MP; e++) bpar[(int64_t)d * MP + e] = par[(int64_t)d * MP + e];
        dirty[d >> 5] = 0u;  // (every set bit of the word is a listed node)
      }
      Warp::sync();
      if (l == 0) {
        const int64_t born = bt->born;
        bt->log_post = lp; bt->log_lik = ll; bt->log_prior = lpr;
        bt->iter = born > D ? born : D; bt->total_edges = te; bt->found = 1;
        bt->n_dirty = 0;
      }
      Warp::sync();
    }
  }
  if (c >= 0 && l == 0) {  // c's list is about to change: the current graph is born at `it`
    if (!test_bit(dirty, c)) { dirty[c >> 5] |= 1u << (c & 31); list[bt->n_dirty] = c; bt->n_dirty++; }
    bt->born = it;
  }
  Warp::sync();
  return computed;
}

BN_HD void best_check(const ChainParams& p, const ChainMem& m, ChainScalars& s, int64_t it, int c) {
  double g = s.gll;
  if (best_visit(m.best, m.base, m.par, m.npar, p.P, p.max_par, s.te_true, s.agree_true, it, c, s.gll_ok, &g)) {
    s.gll = g; s.gll_ok = 1;
  }
}

// end of the call: the final graph's turn, then -1 / 0 lists when no graph was a candidate (end <= D)
BN_HD void best_finish(const ChainParams& p, const ChainMem& m, ChainScalars& s) {
  best_check(p, m, s, p.n_iter, -1);
  if (!m.best->found) {
    for (int64_t i = Warp::lane(); i < (int64_t)p.P * p.max_par; i += Warp::NL) m.best->par[i] = -1;
    for (int i = Warp::lane(); i < p.P; i += Warp::NL) m.best->npar[i] = 0;
  }
  Warp::sync();
}

// ---------------------------------------------------------------------------
// Posterior Markov blanket tabulation (ChainMem.mb): freq[i + j*P] counts the iterations, from max(drop, iter)
// on, after which i -> j, j -> i, or some node has both i and j as parents; the diagonal counts them all.
// wit[i + j*P] holds the number of such reasons (the edge between i and j counts one, each common child one
// more), so the pair is in the blanket iff wit > 0.  It is a function of the graph: an accepted move j -> c
// changes the pairs (j, c) and (j, q), q a co-parent, by one witness each (mb_move).  The count accumulates
// with signs, as anc_freq does: a pair that enters the blanket at iteration t subtracts max(t, drop), one that
// leaves adds it.  The chain start adds the start graph's nodes one by one (mb_graph, -max(drop, iter)) and the
// end removes them all again (+max(end, drop)), so no pass over all P * P pairs is needed.
// ---------------------------------------------------------------------------
BN_HD void mb_count(int* x, int v) {
#if defined(__CUDA_ARCH__)
  atomicAdd(x, v);  // (result unused: a reduction the lane does not wait for; the lanes' pairs are distinct)
#else
  *x += v;
#endif
}

// One witness more (dw = +1) or less (dw = -1) for each pair listed; a count that leaves or reaches 0 adds
// -dw * v to both halves of the pair.  j >= 0: the pairs (j, pc[0..k)) and (j, c) of a move j -> c.  j < 0: every
// witness node c holds, the pairs (pc[e], pc[f]) for f < e < k and (pc[e], c).  The pairs of one call are
// distinct, so lanes own distinct counters.  Not inlined: resumable runs without the tabulation keep the
// registers and instruction-cache footprint of their chain loop.
BN_NOINLINE void mb_pairs(MbTrack* mt, int P, int c, const int* pc, int k, int j, int dw, int v) {
  int* freq = mt->freq;
  uint16_t* wit = mt->wit;
  const int n = j >= 0 ? k + 1 : k * (k + 1) / 2;
  for (int t = Warp::lane(); t < n; t += Warp::NL) {
    int a, b;
    if (j >= 0) {
      a = j; b = t < k ? pc[t] : c;
    } else {  // row e of the triangle: (pc[e], pc[0..e)), then (pc[e], c)
      int e = 0;
      while ((e + 1) * (e + 2) / 2 <= t) e++;
      const int f = t - e * (e + 1) / 2;
      a = pc[e]; b = f < e ? pc[f] : c;
    }
    const int64_t ab = (int64_t)a + (int64_t)b * P, ba = (int64_t)b + (int64_t)a * P;
    const int w0 = wit[ab], w1 = w0 + dw;
    wit[ab] = (uint16_t)w1; wit[ba] = (uint16_t)w1;
    if (w0 == 0 || w1 == 0) { mb_count(freq + ab, -dw * v); mb_count(freq + ba, -dw * v); }
  }
  Warp::sync();
}

// accepted move j -> c (v = first_counted): an addition with c's list before j is appended, a deletion with the
// list after the shift (dw = +1 / -1)
BN_HD void mb_move(const ChainParams& p, const ChainMem& m, int c, int k, int j, int dw, int v) {
  mb_pairs(m.mb, p.P, c, m.par + (int64_t)c * p.max_par, k, j, dw, v);
}

// every node's witnesses added (chain start, dw = +1, v = max(drop, iter)) or removed (end, dw = -1,
// v = max(end, drop)); the diagonal counts the same iterations (-dw * v).  The nodes go one at a time: two
// nodes may share a pair.
BN_HD void mb_graph(const ChainParams& p, const ChainMem& m, int dw, int v) {
  for (int c = 0; c < p.P; c++) {
    const int k = m.npar[c];
    if (k) mb_pairs(m.mb, p.P, c, m.par + (int64_t)c * p.max_par, k, -1, dw, v);
  }
  for (int i = Warp::lane(); i < p.P; i += Warp::NL) m.mb->freq[(int64_t)i * (p.P + 1)] += -dw * v;
  Warp::sync();
}

// empty graph: every row holds its own node only
BN_HD void anc_reset(const ChainParams& p, ChainMem& m) {
  const int l = Warp::lane();
  for (int64_t i = l; i < (int64_t)p.P * p.Ws; i += Warp::NL) m.anc[i] = 0u;
  Warp::sync();
  for (int d = l; d < p.P; d += Warp::NL) m.anc[(int64_t)d * p.Ws + (d >> 5)] = 1u << (d & 31);
  Warp::sync();
}

// full build (chain start from a non-empty graph): Jacobi sweeps to the fixpoint
BN_HD void anc_build_all(const ChainParams& p, ChainMem& m) {
  const RowGeom g = row_geom(p);
  const int l = Warp::lane(), P = p.P;
  anc_reset(p, m);
  for (int round = 0; round <= P; round++) {
    int changed = 0;
    for (int d = 0; d < P; d++) {
      const int kd = m.npar[d];
      if (kd == 0) continue;
      U4* ad = (U4*)(m.anc + (int64_t)d * p.Ws);
      const int* pd = m.par + (int64_t)d * p.max_par;
      for (int ch = l; ch < g.chunks; ch += Warp::NL) {
        U4 v = {0u, 0u, 0u, 0u};
        if (ch == (d >> 7)) v = with_bit(v, d & 127);
        for (int e = 0; e < kd; e++) {
          const int q = pd[e];
          v = or4(v, ((const U4*)(m.anc + (int64_t)q * p.Ws))[ch]);
        }
        if (ne4(v, ad[ch])) { ad[ch] = v; changed = 1; }
      }
      Warp::sync();
    }
    if (Warp::ballot(changed) == 0u) break;
  }
  Warp::sync();
}

// Kernels with MaxPar > 8 keep a Cholesky factor per node (score_core.cuh): (re)factorise node c
// for its current parent list; returns its score.
template <int KMAX>
BN_HD double factor_current(const ChainParams& p, const ChainMem& m, int c) {
  const int MP = p.max_par, k = m.npar[c];
  double* F = m.fac + (int64_t)c * fac_stride(fac_mp(MP));
  if (k <= 8) {
    Parents8 S;
    const Par8 q = load_par8(p, m, c);
#pragma unroll
    for (int e = 0; e < 8; e++) S.s[e] = q.q[e];
    return factor_node8(p.C, p.ldc, c, S, k, p.sc, F, fac_mp(MP));
  }
  return factor_node(p.C, p.ldc, c, m.par + (int64_t)c * MP, k, p.sc, F, fac_mp(MP));
}

// ---------------------------------------------------------------------------
// Chain start: network::network graph part, src/network.h:115-122,138-170
// ---------------------------------------------------------------------------
// InitialNetwork == 1 (random start).  The reference's version (src/network.h:148-163) writes
// edges[p][s] into vectors sized by the prior graph (out of bounds) and neither avoids duplicate
// parents nor cycles, so it is undefined there; this is the defined variant with the same draw
// order from the chain's uniform stream, before iteration 0: for every node that is not a source,
// Npar = int(MaxPar * u) parents are drawn as int(P * u), re-drawn while the candidate is the node
// itself, a sink, already a parent or an ancestor-closing choice (would create a cycle); a slot
// that finds no parent in 100 draws (the reference's "> 100 tries" remark, :288,298) ends the
// node's list.  Returns the number of uniforms consumed.
template <int KMAX>
BN_HD int64_t random_start(const ChainParams& p, ChainMem& m, RngStream& rng) {
  const int P = p.P, MP = p.max_par;
  int64_t pos = 0;
  int anc_changed = 0;
  for (int c = 0; c < P; c++) {
    if (p.node_type[c] == 1) continue;
    if (pos >= rng.gen_hi) rng_top_up(rng, pos);
    const int want = (int)(MP * rng.ubuf[pos & (RNG_CAP - 1)]);
    pos++;
    for (int slot = 0; slot < want; slot++) {
      int found = -1;
      for (int tries = 0; tries < 100 && found < 0; tries++) {
        if (pos >= rng.gen_hi) rng_top_up(rng, pos);
        const int j = (int)(P * rng.ubuf[pos & (RNG_CAP - 1)]);
        pos++;
        int ok = (j != c && p.node_type[j] != 2 && !test_bit(m.anc + (int64_t)j * p.Ws, c));
        for (int e = 0; e < slot; e++) if (m.par[(int64_t)c * MP + e] == j) ok = 0;
        if (ok) found = j;
      }
      if (found < 0) break;
      Warp::sync();
      if (Warp::lane() == 0) { m.par[(int64_t)c * MP + slot] = found; m.npar[c] = slot + 1; }
      Warp::sync();
      anc_after_add(p, m, found, c, anc_changed);
    }
  }
  return pos;
}

// A supplied start (m.start_par, host-validated: an acyclic graph in list order) replaces the start graph of
// initial_network; with m.start the chain continues at iteration m.start->iter with the scalars the
// stopped run exported, and its stream continues where that run left it (the caller hands the stream
// state in, so the read position starts at 0).  Edges and parent counts of the start graph are tabulated
// from max(drop, iter): the tabulations of consecutive segments add up to the uninterrupted run's.
template <int KMAX>
BN_HD void chain_init(const ChainParams& p, ChainMem& m, ChainScalars& s, RngStream& rng) {
  const int l = Warp::lane(), P = p.P, MP = p.max_par;
  const bool given = m.start_par != nullptr;
  const int64_t it0 = m.start ? m.start->iter : 0;
  const int counted_from = (m.start && it0 > p.drop) ? (int)it0 : p.drop;
  for (int64_t i = l; i < (int64_t)P * MP; i += Warp::NL) {
    // unused slots hold -1 (load_par8 relies on it)
    const int c = (int)(i / MP), e = (int)(i % MP);
    m.par[i] = given ? m.start_par[i]
                     : (p.initial_network == 0 && e < p.prior_npar[c]) ? p.prior_par[(int64_t)c * p.prior_stride + e] : -1;
    if (m.born) m.born[i] = counted_from;  // edges of the start graph are counted from iteration max(drop, iter)
  }
  if (m.npar_freq)
    for (int i = l; i < P; i += Warp::NL) m.npar_since[i] = counted_from;
  for (int i = l; i < P; i += Warp::NL) m.npar[i] = given ? m.start_npar[i] : (p.initial_network == 0) ? p.prior_npar[i] : 0;
  for (int w = l; w < p.W; w += Warp::NL) m.haspar[w] = 0u;
  if (m.nver)
    for (int i = l; i < P; i += Warp::NL) m.nver[i] = 0u;
  Warp::sync();
  int64_t start_pos = 0;
  const bool random = !given && p.initial_network == 1;
  if (random) {
    anc_reset(p, m);
    start_pos = random_start<KMAX>(p, m, rng);
  }
  if (l == 0) {
    int te = 0, ag = 0, nh = 0;
    for (int c = 0; c < P; c++) {
      const int k = m.npar[c];
      if (k) { m.haspar[c >> 5] |= 1u << (c & 31); m.hp_list[nh] = c; nh++; }
      for (int e = 0; e < k; e++) {
        te++;
        if (p.sim_edge[(int64_t)m.par[(int64_t)c * MP + e] + (int64_t)c * P]) ag++;
      }
    }
    s.te_true = te; s.agree_true = ag; s.n_haspar = nh;
  }
  s.te_true = Warp::shfl(s.te_true, 0);
  s.agree_true = Warp::shfl(s.agree_true, 0);
  s.n_haspar = Warp::shfl(s.n_haspar, 0);
  Warp::sync();
  if (random) { /* ancestor rows were kept while the graph was drawn */ }
  else if (s.te_true > 0) anc_build_all(p, m);
  else anc_reset(p, m);
  if (m.anc_freq) anc_tab_all(p, m, -counted_from);  // the start graph's paths are counted from max(drop, iter)
  if (m.mb) mb_graph(p, m, 1, counted_from);         // and its blanket pairs
  // base scores (and the per-node factors of the MaxPar > 8 kernels), or those of the stopped run:
  // after a Givens downdate (MaxPar > 8) they differ from a fresh factorisation in the last bits
  s.n_nonpd = 0;
  for (int c = l; c < P; c += Warp::NL) {
    if (m.base_in) {
      m.base[c] = m.base_in[c];
    } else if (KMAX <= 8) {
      Parents8 S;
      const int k = m.npar[c];
#pragma unroll
      for (int e = 0; e < 8; e++) S.s[e] = (e < k) ? m.par[(int64_t)c * MP + e] : c;
      m.base[c] = score_set8(p.C, p.ldc, c, S, k, p.n_samples);
    } else {
      m.base[c] = factor_current<KMAX>(p, m, c);
    }
  }
  Warp::sync();
  s.iter = it0; s.read_pos = start_pos;
  s.valid = m.start ? m.start->valid : 1;  // src/bayesnet_mcmc.cpp:40
  s.te_m = m.start ? m.start->te_m : 0;    // members start at 0 (src/network.h:49-51,64)
  for (int t = 0; t < 3; t++) { s.proposed[t] = 0; s.reject[t] = 0; s.lane_prop[t] = 0; s.lane_rej[t] = 0; }
  s.lane_nonpd = 0; s.lane_valid = 0; s.lane_bytes = 0;
  s.acc_add = m.start ? m.start->acc_add : 0; s.acc_del = m.start ? m.start->acc_del : 0;
  s.n_rows = 0; s.n_moves = 0; s.valid_iters = 0; s.alg_bytes = 0;
  s.gll_ok = 0; s.gll = 0.0;
  s.win = 4; s.windows = 0; s.status = 0; s.need_full = 0; s.anc_changed = 0;
  s.next_log = 0;
  if (m.start) {  // the first logged iteration at or after it0 (it0 + n_iter <= INT_MAX, host-checked)
    const int64_t nl = (it0 + p.output_every - 1) / p.output_every * p.output_every;
    s.next_log = nl > 0x7fffffff ? 0x7fffffff : (int)nl;
  }
  s.pw_cur = -1; s.pw_seen = 0; s.pw_out_pos = 0; s.pw_out_seq = 0; s.pw_out = 0; s.pw_waits = 0; s.pw_discards = 0; s.pw_rebuilds = 0;
  for (int t = 0; t < 6; t++) s.pw_cyc[t] = 0;
  for (int t = 0; t < 12; t++) s.cyc[t] = 0;
  s.slots_sim = 0;
  if (m.best) best_init(p, m, it0, counted_from);  // the start graph is the current one, born at it0
}

// globalLL = sum_p score(p) of the kept graph (LogLikelihood(1), src/network.h:239-247).
BN_HD double sum_base(const ChainParams& p, const ChainMem& m) { return sum_scores(m.base, p.P); }

// ---------------------------------------------------------------------------
// Phase A: replay the draw order of `nslots` iterations (warp-uniform).
// Returns the number of slots filled; sets *overflow when a single iteration
// outran the ring.
// ---------------------------------------------------------------------------
// `unbounded` (want == 1): the iteration is not speculative, so when it outruns the ring the ring
// slides forward with it (the reference's rejection loops, src/network.h:283-299, have no limit);
// *overflow = 2 when no legal child / parent exists at all (the reference would spin forever),
// 3 when a replayed stream ran out inside a rejection loop.
BN_HD int phase_a(const ChainParams& p, const ChainMem& m, const ChainScalars& s,
                  RngStream& rng, WindowSlots& ws, int want, int* overflow, int unbounded = 0) {
  const int P = p.P, MP = p.max_par;
  int64_t pos = s.read_pos;
  int valid = s.valid, te_m = s.te_m;
  int64_t hi = rng.gen_hi;
  int n = 0;
  *overflow = 0;
#define BN_U(dst)                                        \
  do {                                                   \
    if (pos >= hi && unbounded) { rng_top_up(rng, pos); hi = rng.gen_hi; } \
    if (pos >= hi) { ovf = 1; dst = 0.75; }              \
    else dst = rng.ubuf[pos & (RNG_CAP - 1)];            \
    pos++;                                               \
  } while (0)
  while (n < want) {
    int ovf = 0;
    double u;
    BN_U(u);  // u_move, src/bayesnet_mcmc.cpp:48
    int type, c = 0, j = 0, e = -1;
    if (u > 0.5 || te_m < 3) {
      // propose_addition, src/network.h:281-306
      if (unbounded) {
        int any = 0;
        for (int q = Warp::lane(); q < P; q += Warp::NL) any |= (p.node_type[q] != 1 && m.npar[q] < MP) ? 1 : 0;
        if (Warp::ballot(any) == 0u) { *overflow = 2; return 0; }
      }
      for (;;) {
        BN_U(u);
        c = (int)(P * u);
        if (ovf || (p.node_type[c] != 1 && m.npar[c] < MP)) break;
        if (unbounded && rng.kind == RNG_REPLAY && pos > rng.replay_len) { *overflow = 3; return 0; }
      }
      const int kc = ovf ? 0 : m.npar[c];
      const int* pc = m.par + (int64_t)c * MP;
      if (unbounded) {
        int any = 0;
        for (int q = Warp::lane(); q < P; q += Warp::NL) {
          int ok = (p.node_type[q] != 2 && q != c);
          for (int t = 0; t < kc; t++) if (pc[t] == q) ok = 0;
          any |= ok;
        }
        if (Warp::ballot(any) == 0u) { *overflow = 2; return 0; }
      }
      for (;;) {
        BN_U(u);
        j = (int)(P * u);
        if (ovf) break;
        int ok = (p.node_type[j] != 2 && j != c);
        for (int q = 0; q < kc; q++) if (pc[q] == j) ok = 0;
        if (ok) break;
        if (unbounded && rng.kind == RNG_REPLAY && pos > rng.replay_len) { *overflow = 3; return 0; }
      }
      type = 1;
      te_m = s.te_true;  // OldLogPrior = LogPrior(), :302
      // CheckValidity -> pathExists (src/network.h:366-432): is c an ancestor of j?
      if (!ovf) valid = !(j == c || test_bit(m.anc + (int64_t)j * p.Ws, c));
    } else {
      // propose_deletion, src/network.h:308-328
      BN_U(u);  // drawn and discarded (:309)
      BN_U(u);
      const int idx = (int)(s.n_haspar * u);
      BN_U(u);
      if (!ovf) {
        c = m.hp_list[idx];
        e = (int)(m.npar[c] * u);
        j = m.par[(int64_t)c * MP + e];
      }
      type = 2;
      te_m = s.te_true;  // :323
      // `valid` keeps the previous iteration's value (src/bayesnet_mcmc.cpp:50-52)
    }
    double ua = 0.0;
    if (valid && !ovf) {
      // checker(): NewLogPrior = LogPrior() on the proposed graph (src/network.h:333) leaves
      // TotalEdges at the proposed count; FP/FN need the prior adjacency and do not steer
      // the draw order, so phase B fills them in (one lane per slot)
      te_m = s.te_true + (type == 1 ? 1 : -1);
      BN_U(ua);  // acceptance uniform, :335
    }
    if (ovf) { *overflow = (n == 0); break; }
    if (Warp::lane() == 0) {
      ws.child[n] = c; ws.parent[n] = j; ws.pos[n] = e;
      ws.type[n] = (signed char)type; ws.valid[n] = (signed char)valid;
      ws.te_m[n] = te_m;
      ws.pos_after[n] = pos; ws.u_acc[n] = ua;
    }
    n++;
  }
#undef BN_U
  Warp::sync();
  return n;
}

// ---------------------------------------------------------------------------
// Score of the parent set a proposal would leave at child c (push_back / erase order,
// src/network.h:303,325).
// ---------------------------------------------------------------------------
template <int KMAX>
BN_HD double score_proposal(const ChainParams& p, const ChainMem& m, int type, int c, int j, int del,
                            double* rowout, int* kk_out, int* npd) {
  const int MP = p.max_par;
  const int* pc = m.par + (int64_t)c * MP;
  const int k = m.npar[c];
  *kk_out = k + (type == 1 ? 1 : -1);
  *npd = 0;
  double nw;
  if (KMAX <= 8) {
    // MaxPar <= 8: register-resident Cholesky of the proposed set (push_back / erase order)
    Parents8 S;
    if (type == 1) {
#pragma unroll
      for (int e = 0; e < 8; e++) S.s[e] = (e < k) ? pc[e] : j;
    } else {
#pragma unroll
      for (int e = 0; e < 8; e++) {
        const int src = e + (e >= del ? 1 : 0);
        S.s[e] = (src < k) ? pc[src] : c;
      }
    }
    nw = score_set8(p.C, p.ldc, c, S, *kk_out, p.n_samples);
    *npd = (nw == -INFINITY) ? 1 : 0;
    return nw;
  }
  // MaxPar > 8: O(k^2) on the node's cached factor
  const double* F = m.fac + (int64_t)c * fac_stride(fac_mp(MP));
  int flags = 0;
  if (k <= 8) {
    Parents8 S;
    const Par8 q = load_par8(p, m, c);
#pragma unroll
    for (int e = 0; e < 8; e++) S.s[e] = q.q[e];
    nw = score_move8(p.C, p.ldc, p.diag, c, S, k, type, j, del, p.sc, F, fac_mp(MP), rowout, &flags);
  } else {
    nw = score_move_stream<KMAX>(p.C, p.ldc, p.diag, c, pc, k, type, j, del, p.sc, F, fac_mp(MP), rowout, &flags);
  }
  if (flags == SCORE_NOFACTOR) nw = score_scratch<KMAX>(p.C, p.ldc, c, pc, k, del, p.n_samples, npd);
  else if (flags == SCORE_NPD) *npd = 1;
  return nw;
}

// ---------------------------------------------------------------------------
// Phase B + C for one slot (one lane): score the proposed set and decide.
// ---------------------------------------------------------------------------
template <int KMAX>
BN_HD void phase_bc(const ChainParams& p, const ChainMem& m, const ChainScalars& s,
                    WindowSlots& ws, int i) {
  const int c = ws.child[i], j = ws.parent[i];
  const int fp_true = s.te_true - s.agree_true, fn_true = p.n_sim_edges - s.agree_true;
  if (!ws.valid[i]) {
    // invalid: only OldLogPrior ran, the members describe the current graph
    ws.fp_m[i] = fp_true; ws.fn_m[i] = fn_true;
    ws.accept[i] = 0; ws.nonpd[i] = 0; ws.kk[i] = 0;
    return;
  }
  {
    const int ag = p.sim_edge[(int64_t)j + (int64_t)c * p.P] ? 1 : 0;
    const int ag_new = s.agree_true + (ws.type[i] == 1 ? ag : -ag);
    ws.fp_m[i] = ws.te_m[i] - ag_new;
    ws.fn_m[i] = p.n_sim_edges - ag_new;
  }
  int kk = 0, npd = 0;
  const double nw = score_proposal<KMAX>(p, m, ws.type[i], c, j, ws.pos[i], nullptr, &kk, &npd);
  ws.new_score[i] = nw;
  ws.kk[i] = kk;
  ws.nonpd[i] = (signed char)npd;
  // HR = exp(NewLogLike - OldLogLike + NewLogPrior - OldLogPrior), src/network.h:334
  const double old_prior = prior_value(p.phi, p.omega, fp_true + fn_true, s.te_true);
  const double new_prior = prior_value(p.phi, p.omega, ws.fp_m[i] + ws.fn_m[i], ws.te_m[i]);
  const double arg = sub_rn(add_rn(sub_rn(nw, m.base[c]), new_prior), old_prior);
  const double HR = exp(arg);
  ws.accept[i] = (ws.u_acc[i] > HR) ? 0 : 1;  // reject iff runif > HR (NaN accepts), :335
}

// ---------------------------------------------------------------------------
// Rounds: position-parallel speculation.
//
// The only sequential dependences between iterations are the stream position (each
// iteration consumes a data-dependent number of uniforms), the stale `valid` flag, and the
// graph itself, which changes on the ~5% of iterations that are accepted.  So one thread
// per stream position q in [pos, pos + REPLAY_POS) builds the RECORD of the iteration that
// WOULD start at q: draw replay (move type, rejection-sampled child/parent, uniforms
// consumed, cycle test), the score of the proposed parent set, and the accept decision.
// Roughly one position in five is a real iteration start; the rest is latency-free slack
// of the eight warps.  The chain's own warp then walks the records from the committed
// position (pointer chase over `consumed`), commits rejected iterations in bulk, and on an
// accepted move applies it and REPAIRS the remaining records instead of discarding them:
//   * a record depends on the graph only through its child's parent list (replay of the
//     duplicate test / deletion index, score, base score), the ancestor bit of its
//     (parent, child) pair, and the global counts TotalEdges / Nagree (prior terms);
//   * records of the changed child are stale: the walk stops in front of the first one
//     and the next round starts there;
//   * cycle bits are re-tested by all threads; the accept decisions stand (a move at another
//     node changes the Hastings argument by rounding only; close calls are marked stale).
//     Cyclic additions are never scored: should their cycle bit clear, the record goes stale;
//   * a move that changes the set of nodes with parents (deletion draws index into it) has the
//     deletion records behind the walk redone in place; a child that drops below MaxPar makes
//     stale the draws that skipped it.
// Requires TotalEdges >= 4 so that the `TotalEdges < 3` branch of
// src/bayesnet_mcmc.cpp:48 cannot fire; the sequential window path covers the rest.
// ---------------------------------------------------------------------------
struct RoundCtx {  // warp-uniform, handed to the helper warps through the command block
  int64_t pos, hi;
  int n_haspar, te_true, agree_true;
  int redo_from;  // -1: build every record; >= 0: rebuild records from this slot on, namely ...
  int redo_mode;  // ... 0: the deletion records; 1: the stale records; 2: all of them
};

// draw replay of the iteration that would start at stream position q -> record `slot`
BN_HD void replay_position(const ChainParams& p, const ChainMem& m, int n_haspar, const double* ubuf,
                           int64_t hi, int64_t q, WindowSlots& ws, int slot) {
  const int P = p.P, MP = p.max_par;
  int64_t i = q;
  int ovf = 0, type, c = 0, j = 0, e = -1, cyc = 0, many = 0;
  uint32_t full = 0u;
  double u;
#define BN_UAT(dst)                                    \
  do {                                                 \
    if (i >= hi) { ovf = 1; dst = 0.75; }              \
    else dst = ubuf[i & (RNG_CAP - 1)];                \
    i++;                                               \
  } while (0)
  BN_UAT(u);  // u_move, src/bayesnet_mcmc.cpp:48
  if (u > 0.5) {
    // propose_addition, src/network.h:281-306
    type = 1;
    for (;;) {
      BN_UAT(u);
      c = (int)(P * u);
      if (ovf || p.node_type[c] == 1) { if (ovf) break; continue; }
      if (m.npar[c] < MP) break;
      // skipped for being full: the record goes stale if this node loses a parent
      if (P > 0xfffe || (full >> 16)) many = 1;
      else full = (full << 16) | (uint32_t)(c + 1);
    }
    const int kc = ovf ? 0 : m.npar[c];
    const int* pc = m.par + (int64_t)c * MP;
    Par8 pc8;
    if (MP <= 8) pc8 = load_par8(p, m, c);
    for (;;) {
      BN_UAT(u);
      j = (int)(P * u);
      if (ovf) break;
      int ok = (p.node_type[j] != 2 && j != c);
      if (MP <= 8) {  // unused slots hold -1
#pragma unroll
        for (int t = 0; t < 8; t++) if (pc8.q[t] == j) ok = 0;
      } else {
        for (int t = 0; t < kc; t++) if (pc[t] == j) ok = 0;
      }
      if (ok) break;
    }
    // CheckValidity -> pathExists (src/network.h:366-432): is c an ancestor of j?
    if (!ovf) cyc = test_bit(m.anc + (int64_t)j * p.Ws, c) ? 1 : 0;
  } else {
    // propose_deletion, src/network.h:308-328
    type = 2;
    BN_UAT(u);  // drawn and discarded (:309)
    BN_UAT(u);
    const int idx = (int)(n_haspar * u);
    BN_UAT(u);
    if (!ovf) {
      c = m.hp_list[idx];
      e = (int)(m.npar[c] * u);
      j = m.par[(int64_t)c * MP + e];
    }
  }
#undef BN_UAT
  // the acceptance uniform must be in the ring as well, and the count (+1) must fit the record
  if (i >= hi || i - q >= REC_LEN_MASK) ovf = 1;
  ws.t_c[slot] = c; ws.t_j[slot] = j; ws.t_e[slot] = e; ws.t_full[slot] = full;
  ws.t_rec[slot] = (int)(i - q) | (type == 2 ? REC_TYPE : 0) | (cyc ? REC_CYC : 0) | (ovf ? REC_OVF : 0) |
                   (many ? REC_FULLMANY : 0);  // (REC_AG: build_record)
}

// what the walk needs of a (consumable) record: an addition sets `valid` itself
// (src/bayesnet_mcmc.cpp:50), a deletion inherits it; invalid iterations draw no acceptance uniform
BN_HD int walk_word(int rec) {
  const int cons = rec & REC_LEN_MASK, accept = (rec & REC_ACC) ? 1 : 0;
  if (rec & REC_TYPE) return cons | ((cons + 1) << 8) | (1 << 17) | (accept << 19);
  if (rec & REC_CYC) return cons | (cons << 8);
  const int len = cons + 1;
  return len | (len << 8) | (3 << 16) | (accept << 18) | (accept << 19);
}

// checker() for a record under the current global counts: sets REC_ACC / REC_CLOSE and the walk word
BN_HD void decide_record(const ChainParams& p, const ChainMem& m, const RoundCtx& rc, const double* ubuf,
                         WindowSlots& ws, int slot) {
  int rec = ws.t_rec[slot];
  if (rec & REC_OVF) { ws.t_walk[slot] = WALK_OVF; return; }
  const int c = ws.t_c[slot];
  const int type = (rec & REC_TYPE) ? 2 : 1;
  if (type == 1 && (rec & REC_CYC)) {  // invalid addition: no checker(), no acceptance draw
    ws.t_walk[slot] = walk_word(rec);
    return;
  }
  const int ag = (rec & REC_AG) ? 1 : 0;
  const int te_new = rc.te_true + (type == 1 ? 1 : -1);
  const int ag_new = rc.agree_true + (type == 1 ? ag : -ag);
  const int fp_true = rc.te_true - rc.agree_true, fn_true = p.n_sim_edges - rc.agree_true;
  const double old_prior = prior_value(p.phi, p.omega, fp_true + fn_true, rc.te_true);
  const double new_prior = prior_value(p.phi, p.omega, (te_new - ag_new) + (p.n_sim_edges - ag_new), te_new);
  // HR = exp(NewLogLike - OldLogLike + NewLogPrior - OldLogPrior), src/network.h:334
  const double arg = sub_rn(add_rn(sub_rn(ws.t_score[slot], m.base[c]), new_prior), old_prior);
  // reject iff runif > HR (NaN accepts), :335.  u > exp(arg) <=> log u > arg unless the two are
  // within rounding of each other: then (and for NaN) the reference's own expression decides.
  // A move at ANOTHER node changes arg only by the rounding of the two prior expressions
  // (NewLogPrior - OldLogPrior is -phi (1 - 2 ag) -/+ omega whatever the counts), so outside the
  // 1e-6 band the decision stands for the rest of the round; inside it the record is marked.
  const double d = ws.t_lu[slot] - arg;
  int accept;
  rec &= ~(REC_ACC | REC_CLOSE);
  if (fabs(d) > 1e-6) {
    accept = !(d > 0.0);
  } else {
    const double HR = exp(arg);
    const double u_acc = ubuf[(rc.pos + slot + (rec & REC_LEN_MASK)) & (RNG_CAP - 1)];
    accept = !(u_acc > HR);
    rec |= REC_CLOSE;
  }
  if (accept) rec |= REC_ACC;
  ws.t_rec[slot] = rec;
  ws.t_walk[slot] = walk_word(rec);
}

BN_HD double nan_sentinel() {
#if defined(__CUDA_ARCH__)
  return __longlong_as_double(-1ll);
#else
  return NAN;
#endif
}

// Warp-cooperative O(k^2) scoring of ONE proposal at a node with 9..32 parents (MaxPar > 8 kernels,
// device only).  A single thread streaming the node's factor pays an L2 round trip per row, and the
// slowest record sets the length of a round; here lane l owns row l of the factor (its entries in
// registers, every load of the warp in flight at once) and the forward substitution runs across
// the lanes: step t finalises w_t on lane t, broadcasts it, and the lanes below subtract their
// L[l][t] w_t.  Same arithmetic as score_move_stream up to the order of the two final sums.
// All 32 lanes call it with the same arguments.
#if defined(__CUDACC__)
template <int KMAX>
__device__ __forceinline__ double coop_score(const ChainParams& p, const ChainMem& m, int c, int j, int type, int del,
                                             double* rowout, int* npd) {
  const int l = Warp::lane(), MP = p.max_par, mp = fac_mp(MP);
  const double* F = m.fac + (int64_t)c * fac_stride(mp);
  const int k = m.npar[c];
  const bool mine = l < k;
  const double* Frow = F + fac_row(l);
  D2 r[16];  // own row: L[l][0..l-1] (the reciprocal pivot is read separately)
#pragma unroll
  for (int q = 0; q < 16; q++) {
    r[q].x = 0.0; r[q].y = 0.0;
    if (mine && 2 * q < l) r[q] = ld2_l2(Frow + 2 * q);
  }
  const double rinv = mine ? ld1_l2(Frow + l) : 0.0;
  const double zl = mine ? ld1_l2(F + fac_zoff(mp) + l) : 0.0;
  const D2 tail = ld2_l2(F + fac_tail(mp));
  const double rss = tail.x, icc = tail.y;
  const bool add = type == 1;
  double a = 0.0, d0 = 0.0, e0 = 0.0;
  if (add) {
    if (mine) a = ld_shared_ro(p.C + (int64_t)m.par[(int64_t)c * MP + l] * p.ldc + j);
    d0 = ld_shared_ro(p.diag + j);
    e0 = ld_shared_ro(p.C + (int64_t)c * p.ldc + j);
  }
  double w_own = 0.0;
#pragma unroll
  for (int t = 0; t < 32; t++) {
    if (t < k) {  // (warp-uniform)
      const double cand = (!add && l == del) ? rinv : a * rinv;  // deletion: y_del = 1 / L[del][del], y_t = 0 above it
      const double wt = Warp::shfl(cand, t);
      if (l == t) w_own = wt;
      const double lt = (t & 1) ? r[t >> 1].y : r[t >> 1].x;  // L[l][t] (0 unless t < l)
      if (l > t) a -= lt * wt;
    }
  }
  const double s1 = Warp::sum(w_own * w_own), s2 = Warp::sum(w_own * zl);
  *npd = 0;
  if (add) {
    const double dj = d0 - s1, ej = e0 - s2;
    bool bad = !(rss == rss) || !(dj > 0.0);
    double rss_new = bad ? NAN : rss - ej * ej / dj;
    if (!bad && !(rss_new * icc > RSS_FLOOR)) { bad = true; rss_new = NAN; }
    if (rowout) {
      if (mine) rowout[l] = w_own;
      if (l == 0) { rowout[row_tail(mp)] = dj; rowout[row_tail(mp) + 1] = ej; rowout[row_tail(mp) + 2] = rss_new; }
    }
    if (bad) { *npd = 1; return -INFINITY; }
    return score_from_rss(rss_new, icc, k + 1, p.sc);
  }
  return score_from_rss(rss + s2 * s2 / s1, icc, k - 1, p.sc);
}
#endif

#if defined(__CUDACC__)
template <int KMAX>
__device__ __forceinline__ void build_record_coop(const ChainParams& p, const ChainMem& m, const RoundCtx& rc,
                                                  const double* ubuf, WindowSlots& ws, int slot, bool active) {
  // (`active` false: this thread has no record to build in this call but takes part in the
  // cooperative scoring of its warp)
  int rec = 0, skip = 1, kk = 0, npd = 0, ag = 0, need = 0, big = 0, c = 0, j = 0, e = -1, type = 1;
  double sc = 0.0, cached = nan_sentinel();
  double* cache = nullptr;
  double* rowout = m.rowbuf + (uint32_t)slot * (uint32_t)row_stride(fac_mp(p.max_par));
  if (active) {
    replay_position(p, m, rc.n_haspar, ubuf, rc.hi, rc.pos + slot, ws, slot);
    rec = ws.t_rec[slot];
    if (rec & REC_OVF) {
      ws.t_walk[slot] = WALK_OVF;
    } else if (!(rec & REC_TYPE) && (rec & REC_CYC)) {
      ws.t_rec[slot] = rec | REC_NOSCORE;  // a cyclic addition is never scored (build_record)
      decide_record(p, m, rc, ubuf, ws, slot);
    } else {
      skip = 0;
      c = ws.t_c[slot]; j = ws.t_j[slot]; e = ws.t_e[slot];
      type = (rec & REC_TYPE) ? 2 : 1;
      cache = (m.dscore && (rec & REC_TYPE)) ? m.dscore + (uint32_t)c * (uint32_t)p.max_par + e : nullptr;
      if (cache) cached = ld_shared_ro(cache);
      ag = ld_shared_ro(p.sim_edge + (int64_t)j + (int64_t)c * p.P) ? REC_AG : 0;
      ws.t_lu[slot] = log(ubuf[(rc.pos + slot + (rec & REC_LEN_MASK)) & (RNG_CAP - 1)]);
      if (cached == cached) {
        sc = cached;
        kk = m.npar[c] - 1;
        npd = (sc == -INFINITY) ? 1 : 0;
      } else {
        need = 1;
        const int k = m.npar[c];
        // nodes with 9..32 parents whose block holds a factor: scored by the whole warp below
        big = (k > 8 && k <= 32 && ld1_l2(m.fac + (int64_t)c * fac_stride(fac_mp(p.max_par)) + fac_tail(fac_mp(p.max_par))) ==
                                       ld1_l2(m.fac + (int64_t)c * fac_stride(fac_mp(p.max_par)) + fac_tail(fac_mp(p.max_par)))) ? 1 : 0;
        if (!big) sc = score_proposal<KMAX>(p, m, type, c, j, e, rowout, &kk, &npd);
      }
    }
  }
  uint32_t todo = Warp::ballot(big);
  while (todo) {
    const int src = ffs32(todo) - 1;
    todo &= todo - 1;
    const int b_c = Warp::shfl(c, src), b_j = Warp::shfl(j, src), b_type = Warp::shfl(type, src), b_e = Warp::shfl(e, src);
    const int b_slot = Warp::shfl(slot, src);
    int b_npd = 0;
    const double v = coop_score<KMAX>(p, m, b_c, b_j, b_type, b_e,
                                      m.rowbuf + (uint32_t)b_slot * (uint32_t)row_stride(fac_mp(p.max_par)), &b_npd);
    if (Warp::lane() == src) { sc = v; npd = b_npd; kk = m.npar[c] + (type == 1 ? 1 : -1); }
  }
  if (active && !skip) {
    if (need && cache) *cache = sc;  // (duplicates within a round store the same value)
    ws.t_score[slot] = sc;
    ws.t_rec[slot] = rec | ag | (npd ? REC_NPD : 0) | (kk << REC_KK_SHIFT);
    decide_record(p, m, rc, ubuf, ws, slot);
  }
}
#endif

template <int KMAX>
BN_HD void build_record(const ChainParams& p, const ChainMem& m, const RoundCtx& rc, const double* ubuf,
                        WindowSlots& ws, int slot) {
  bool active = true;
  if (rc.redo_from >= 0) {
    // the set of nodes with parents changed: deletion draws index into it (src/network.h:311-319),
    // so the deletion records behind the walk are replayed and decided again; additions keep theirs
    const int old = ws.t_rec[slot];
    if (slot < rc.redo_from) active = false;
    else if (rc.redo_mode == 0) active = (old & REC_TYPE) && !(old & REC_OVF);
    else if (rc.redo_mode == 1) active = (old & REC_STALE) != 0;
  }
#if defined(__CUDA_ARCH__)
  if constexpr (KMAX > 8) {
    // MaxPar > 8 on the device: the same record, written without early exits so that the whole warp
    // reaches the cooperative scoring of the proposals at nodes with 9..32 parents
    build_record_coop<KMAX>(p, m, rc, ubuf, ws, slot, active);
    return;
  }
#endif
  if (!active) return;
  replay_position(p, m, rc.n_haspar, ubuf, rc.hi, rc.pos + slot, ws, slot);
  const int rec = ws.t_rec[slot];
  if (rec & REC_OVF) { ws.t_walk[slot] = WALK_OVF; return; }
  if (!(rec & REC_TYPE) && (rec & REC_CYC)) {
    // a cyclic addition never reaches checker(): it is not scored; should an accepted deletion
    // clear its cycle bit later in the round, the record goes stale instead
    ws.t_rec[slot] = rec | REC_NOSCORE;
    decide_record(p, m, rc, ubuf, ws, slot);
    return;
  }
  int kk = 0, npd = 0;
  double sc;
  // the score of a deletion is a function of (child, slot) until the child's parents change:
  // it is kept in a per-chain table (L2), which takes half of the records off the sub-Gram
  // gather -- the throughput limit of this phase (one L1TEX wavefront per gathered entry).
  // The two L2 reads of the record (that table, the prior adjacency) are issued first and the
  // logarithm of the acceptance uniform is taken while they are in flight.
  const int rc_c = ws.t_c[slot], rc_j = ws.t_j[slot];
  double* cache = (m.dscore && (rec & REC_TYPE)) ? m.dscore + (uint32_t)rc_c * (uint32_t)p.max_par + ws.t_e[slot] : nullptr;
  double cached = nan_sentinel();
#if defined(__CUDA_ARCH__)
  // two-CTA pipeline: the table holds (score, tag) pairs, tag = the number of accepted moves at the
  // child when the score was computed.  The chain's CTA and the record builder lag each other by a
  // few moves; an entry is valid for whoever holds the same count, and nothing is ever invalidated
  // (a late store of an outdated score carries an outdated tag).
  long long tag = 0;
  if (m.nver && cache) {
    cache += (cache - m.dscore);  // pairs
    tag = (long long)m.nver[rc_c];
    const D2 v = ld2_l2(cache);
    if (__double_as_longlong(v.y) == tag) cached = v.x;
  } else
#endif
  if (cache) cached = ld_shared_ro(cache);
  const int ag = ld_shared_ro(p.sim_edge + (int64_t)rc_j + (int64_t)rc_c * p.P) ? REC_AG : 0;
  ws.t_lu[slot] = log(ubuf[(rc.pos + slot + (rec & REC_LEN_MASK)) & (RNG_CAP - 1)]);
  if (cached == cached) {
    sc = cached;
    kk = m.npar[ws.t_c[slot]] - 1;
    npd = (sc == -INFINITY) ? 1 : 0;
  } else {
    sc = score_proposal<KMAX>(p, m, (rec & REC_TYPE) ? 2 : 1, ws.t_c[slot], ws.t_j[slot], ws.t_e[slot],
                              KMAX > 8 ? m.rowbuf + (uint32_t)slot * (uint32_t)row_stride(fac_mp(p.max_par)) : nullptr,
                              &kk, &npd);
#if defined(__CUDA_ARCH__)
    if (m.nver && cache) {
      D2 w; w.x = sc; w.y = __longlong_as_double(tag);
      *(D2*)cache = w;
    } else
#endif
    if (cache) *cache = sc;  // (duplicates within a round store the same value)
  }
  ws.t_score[slot] = sc;
  ws.t_rec[slot] = rec | ag | (npd ? REC_NPD : 0) | (kk << REC_KK_SHIFT);
  decide_record(p, m, rc, ubuf, ws, slot);
}

// after an accepted move at child c: records that depend on c's parent list go stale (the walk
// stops if it lands on one), as do the close calls; the others keep their decision, and when
// ancestor rows changed (`retest`) the additions get their cycle bit re-tested.
// `unfull`: the move took c from MaxPar to MaxPar - 1 parents, so draws that skipped c differ
BN_HD void repair_record(const ChainParams& p, const ChainMem& m, WindowSlots& ws, int slot, int c, int unfull,
                         int retest, int from) {
  if (slot < from) return;
  int rec = ws.t_rec[slot];
  if (rec & (REC_OVF | REC_STALE)) return;
  bool stale = ws.t_c[slot] == c || (rec & REC_CLOSE);
  if (!stale && unfull && !(rec & REC_TYPE)) {
    const uint32_t f = ws.t_full[slot], cc = (uint32_t)(c + 1);
    stale = (rec & REC_FULLMANY) || (f & 0xffffu) == cc || (f >> 16) == cc;
  }
  if (!stale && retest && !(rec & REC_TYPE)) {
    const int cyc = test_bit(m.anc + (int64_t)ws.t_j[slot] * p.Ws, ws.t_c[slot]) ? 1 : 0;
    if (cyc != ((rec & REC_CYC) ? 1 : 0)) {
      if (!cyc && (rec & REC_NOSCORE)) {
        stale = true;  // it was never scored
      } else {
        rec = (rec & ~REC_CYC) | (cyc ? REC_CYC : 0);
        ws.t_rec[slot] = rec;
        ws.t_walk[slot] = walk_word(rec);
      }
    }
  }
  if (stale) {
    ws.t_rec[slot] = rec | REC_STALE;
    ws.t_walk[slot] = WALK_STALE;
  }
}

#if defined(__CUDACC__)
// Two-CTA pipeline: a window built when the replica had applied `lo` moves is repaired for the moves
// lo .. hi-1 the chain has accepted since -- repair_record's rules for every move of the list, the
// cycle bit re-tested once against the current ancestor rows (`retest`: one of the moves changed them).
__device__ __forceinline__ void repair_record_batch(const ChainParams& p, const ChainMem& m, WindowSlots& ws, int slot,
                                                    int from, int lo, int hi, int retest) {
  if (slot < from) return;
  int rec = ws.t_rec[slot];
  if (rec & (REC_OVF | REC_STALE)) return;
  const int rc_c = ws.t_c[slot];
  const bool add = !(rec & REC_TYPE);
  const uint32_t f = ws.t_full[slot];
  bool stale = (rec & REC_CLOSE) != 0;
  for (int i = lo; i < hi; i++) {
    const int e = m.pipe->log[i % PIPE_LOG];
    const int c = e & LOG_NODE;
    stale |= (c == rc_c);
    if ((e & LOG_UNFULL) && add) {
      const uint32_t cc = (uint32_t)(c + 1);
      stale |= (rec & REC_FULLMANY) || (f & 0xffffu) == cc || (f >> 16) == cc;
    }
  }
  if (!stale && retest && add) {
    const int cyc = test_bit(m.anc + (int64_t)ws.t_j[slot] * p.Ws, rc_c) ? 1 : 0;
    if (cyc != ((rec & REC_CYC) ? 1 : 0)) {
      if (!cyc && (rec & REC_NOSCORE)) {
        stale = true;  // it was never scored
      } else {
        rec = (rec & ~REC_CYC) | (cyc ? REC_CYC : 0);
        ws.t_rec[slot] = rec;
        ws.t_walk[slot] = walk_word(rec);
      }
    }
  }
  if (stale) {
    ws.t_rec[slot] = rec | REC_STALE;
    ws.t_walk[slot] = WALK_STALE;
  }
}

// record `slot` of the window the builder (rank 1) holds -> this CTA's copy, over distributed shared memory
__device__ __forceinline__ void pipe_copy_record(WindowSlots& ws, int slot) {
  const int c = ld_peer(peer_addr(&ws.t_c[slot], 1)), j = ld_peer(peer_addr(&ws.t_j[slot], 1));
  const int e = ld_peer(peer_addr(&ws.t_e[slot], 1)), rec = ld_peer(peer_addr(&ws.t_rec[slot], 1));
  const int full = ld_peer(peer_addr(&ws.t_full[slot], 1)), walk = ld_peer(peer_addr(&ws.t_walk[slot], 1));
  const long long sc = ld_peer64(peer_addr(&ws.t_score[slot], 1)), lu = ld_peer64(peer_addr(&ws.t_lu[slot], 1));
  ws.t_c[slot] = c; ws.t_j[slot] = j; ws.t_e[slot] = e; ws.t_rec[slot] = rec;
  ws.t_full[slot] = (uint32_t)full; ws.t_walk[slot] = walk;
  ws.t_score[slot] = __longlong_as_double(sc); ws.t_lu[slot] = __longlong_as_double(lu);
}
#endif

#if defined(__CUDACC__)
__device__ __forceinline__ void helper_post(const ChainMem& m, int op, const RoundCtx& rc) {
  if (Warp::lane() == 0) {
    m.helper[1] = (int)(rc.pos & 0xffffffffll); m.helper[2] = (int)(rc.pos >> 32);
    m.helper[3] = (int)(rc.hi & 0xffffffffll); m.helper[4] = (int)(rc.hi >> 32);
    m.helper[5] = rc.n_haspar; m.helper[6] = rc.te_true; m.helper[7] = rc.agree_true;
    m.helper[8] = rc.redo_from; m.helper[11] = rc.redo_mode;
    m.helper[0] = op;
  }
  Warp::sync();
}
__device__ __forceinline__ RoundCtx helper_ctx(const ChainMem& m) {
  RoundCtx rc;
  rc.pos = ((int64_t)m.helper[2] << 32) | (uint32_t)m.helper[1];
  rc.hi = ((int64_t)m.helper[4] << 32) | (uint32_t)m.helper[3];
  rc.n_haspar = m.helper[5]; rc.te_true = m.helper[6]; rc.agree_true = m.helper[7];
  rc.redo_from = m.helper[8]; rc.redo_mode = m.helper[11];
  return rc;
}

// Wichmann-Hill by the whole CTA: thread t jumps ahead t + 1 steps from the state in the
// command block ([5..7]) and writes the uniform at stream position [1..2] + t; the last
// thread leaves the new state in [8..10].
struct WhJump { uint32_t mx, my, mz; };
__device__ __forceinline__ WhJump wh_jump_for_thread() {
  WhJump j;
  j.mx = pow_mod(171u, (int)threadIdx.x + 1, 30269u);
  j.my = pow_mod(172u, (int)threadIdx.x + 1, 30307u);
  j.mz = pow_mod(170u, (int)threadIdx.x + 1, 30323u);
  return j;
}
__device__ __forceinline__ void fill_wh_thread(const ChainMem& m, double* ubuf, const WhJump& j) {
  const int64_t pos = ((int64_t)m.helper[2] << 32) | (uint32_t)m.helper[1];
  const uint32_t xs = ((uint32_t)m.helper[5] * j.mx) % 30269u;
  const uint32_t ys = ((uint32_t)m.helper[6] * j.my) % 30307u;
  const uint32_t zs = ((uint32_t)m.helper[7] * j.mz) % 30323u;
  ubuf[(pos + threadIdx.x) & (RNG_CAP - 1)] = wh_combine(xs, ys, zs);
  if (threadIdx.x == (HELPER_WARPS + 1) * 32 - 1) { m.helper[8] = (int)xs; m.helper[9] = (int)ys; m.helper[10] = (int)zs; }
}
// chain warp: append (HELPER_WARPS + 1) * 32 uniforms while they fit in the ring
__device__ __forceinline__ void team_fill_wh(const ChainMem& m, RngStream& r, int64_t read_pos, const WhJump& j) {
  constexpr int TEAM = (HELPER_WARPS + 1) * 32;
  while (r.gen_hi + TEAM <= read_pos + RNG_CAP) {
    if (Warp::lane() == 0) {
      m.helper[1] = (int)(r.gen_hi & 0xffffffffll); m.helper[2] = (int)(r.gen_hi >> 32);
      m.helper[5] = (int)r.x; m.helper[6] = (int)r.y; m.helper[7] = (int)r.z;
      m.helper[0] = HELPER_FILL_WH;
    }
    Warp::sync();
    cta_bar(1);
    fill_wh_thread(m, r.ubuf, j);
    cta_bar(2);
    r.x = (uint32_t)m.helper[8]; r.y = (uint32_t)m.helper[9]; r.z = (uint32_t)m.helper[10];
    r.gen_hi += TEAM;
    Warp::sync();
  }
}

// body of a helper warp (warp index 1..HELPER_WARPS of the chain's CTA)
// PIPE (two-CTA form): the helper warps do ALL the work of a team operation -- slots and row blocks
// are dealt over HELPER_WARPS parts
template <int KMAX, bool PIPE = false>
__device__ __forceinline__ void helper_loop(const ChainParams& p, const ChainMem& m, int part,
                                            double* ubuf, WindowSlots& ws) {
  const WhJump jump = wh_jump_for_thread();
  for (;;) {
    cta_bar(1);
    const int op = m.helper[0];
    if (op == HELPER_EXIT) break;
    const int slot = (PIPE ? part - 1 : part) * 32 + Warp::lane();
    if (op == HELPER_RECORDS) {
      build_record<KMAX>(p, m, helper_ctx(m), ubuf, ws, slot);
    } else if (op == HELPER_REPAIR) {
      repair_record(p, m, ws, slot, m.helper[9], m.helper[11], m.helper[7], m.helper[8]);
    } else if (op == HELPER_ANC_ADD) {
      if (PIPE)
        anc_add_part(p, m, m.helper[8], m.helper[9], m.scratch + (part - 1) * rows_per_part(p.P, HELPER_WARPS, Warp::NL), part - 1,
                     HELPER_WARPS);
      else
        anc_add_part(p, m, m.helper[8], m.helper[9], m.scratch + part * rows_per_part(p.P, HELPER_WARPS + 1, Warp::NL), part,
                     HELPER_WARPS + 1);
    } else if (op == HELPER_ANC_DEL) {
      if (PIPE) anc_del_team(p, m, m.helper[9], part - 1, HELPER_WARPS);
      else anc_del_team(p, m, m.helper[9], part, HELPER_WARPS + 1);
    } else if (op == HELPER_FILL_WH) {
      fill_wh_thread(m, ubuf, jump);
    } else if (op == HELPER_PIPE_COPY) {
      pipe_copy_record(ws, slot);
    } else if (op == HELPER_REPAIR_BATCH) {
      repair_record_batch(p, m, ws, slot, m.helper[8], m.helper[5], m.helper[6], m.helper[7]);
    }
    cta_bar(2);
  }
}
#endif

template <int KMAX, bool PIPE = false>
BN_HD void team_records(const ChainParams& p, const ChainMem& m, const RoundCtx& rc, const double* ubuf,
                        WindowSlots& ws) {
#if defined(__CUDA_ARCH__)
  if (m.helper) {
    helper_post(m, HELPER_RECORDS, rc);
    cta_bar(1);
    if constexpr (!PIPE) build_record<KMAX>(p, m, rc, ubuf, ws, Warp::lane());
    cta_bar(2);
    return;
  }
#else
  for (int slot = Warp::lane(); slot < REPLAY_POS; slot += Warp::NL) build_record<KMAX>(p, m, rc, ubuf, ws, slot);
  Warp::sync();
#endif
}

// `retest` = the move changed ancestor rows: the cycle bits of the additions are re-tested
BN_HD void team_repair(const ChainParams& p, const ChainMem& m, WindowSlots& ws, int c, int unfull, int retest,
                       int from) {
#if defined(__CUDA_ARCH__)
  if (m.helper) {
    if (Warp::lane() == 0) {
      m.helper[8] = from; m.helper[9] = c; m.helper[11] = unfull; m.helper[7] = retest;
      m.helper[0] = HELPER_REPAIR;
    }
    Warp::sync();
    cta_bar(1);
    if (!m.pipe) repair_record(p, m, ws, Warp::lane(), c, unfull, retest, from);
    cta_bar(2);
  }
#else
  for (int slot = Warp::lane(); slot < REPLAY_POS; slot += Warp::NL)
    repair_record(p, m, ws, slot, c, unfull, retest, from);
  Warp::sync();
#endif
}

// ---------------------------------------------------------------------------
// Commit: counters, trace rows, and the accepted move if any (warp-uniform).
// ---------------------------------------------------------------------------
BN_HD void write_row_vals(const ChainParams& p, ChainMem& m, ChainScalars& s, int64_t it, int child,
                          int type, int fn, int fp, int additions, int deletions) {
  if (!s.gll_ok) { s.gll = sum_base(p, m); s.gll_ok = 1; }
  if (s.n_rows < p.trace_capacity) {
    if (Warp::lane() == 0) {
      const int r = s.n_rows;
      m.t_iter[r] = (int)it;
      m.t_changed[r] = child;
      m.t_movetype[r] = type;
      m.t_gll[r] = s.gll;
      m.t_add[r] = additions;
      m.t_del[r] = deletions;
      m.t_fn[r] = fn;
      m.t_fp[r] = fp;
    }
    s.n_rows++;
  }
}
BN_HD void write_row(const ChainParams& p, ChainMem& m, ChainScalars& s, int64_t it,
                     const WindowSlots& ws, int i, int additions, int deletions) {
  write_row_vals(p, m, s, it, ws.child[i], ws.type[i], ws.fn_m[i], ws.fp_m[i], additions, deletions);
}

// `newrow`: the candidate factor row of an accepted addition record (score_core.cuh), or null
// (sequential path): the node is re-factorised instead.
template <int KMAX>
BN_HD void apply_move_vals(const ChainParams& p, ChainMem& m, ChainScalars& s, int64_t it, int type, int c,
                           int j, int del, double new_score, int ag, const double* newrow) {
  const int MP = p.max_par, l = Warp::lane();
#if defined(__CUDA_ARCH__)
  // Consistency guard (two-CTA form): a move that cannot be applied to the graph it arrives at -- an addition at a
  // full node or of a parent already there, a deletion slot that does not hold the parent -- means a record
  // escaped its repair.  The chain stops with status 95 instead of corrupting its state.
  if (m.pipe) {
    const int kk0 = m.npar[c];
    bool bad = (type == 1) ? (kk0 >= MP) : (del < 0 || del >= kk0 || m.par[(int64_t)c * MP + del] != j);
    if (type == 1) for (int e = 0; e < kk0 && e < MP; e++) bad |= m.par[(int64_t)c * MP + e] == j;
    if (bad) { s.status = 95; return; }
  }
#endif
  if (m.best) best_check(p, m, s, it, c);  // the graph left here, before anything changes
  int* pc = m.par + (int64_t)c * MP;
  int* bc = m.born ? m.born + (int64_t)c * MP : nullptr;  // (only read with edge_freq)
  const int k = m.npar[c];
  double* F = KMAX > 8 ? m.fac + (int64_t)c * fac_stride(fac_mp(MP)) : nullptr;
#if defined(__CUDA_ARCH__)
  // (MaxPar > 8) the accepted record's candidate row (score_core.cuh) becomes row k of the factor: one 16-byte
  // pair per lane; the loads are issued here and the stores follow the ancestor update (an L2
  // round trip hidden)
  D2 rv, rd, rr;
  rv.x = rv.y = rd.x = rd.y = rr.x = rr.y = 0.0;
  if (KMAX > 8 && type == 1 && newrow) {
    if (2 * l < k) rv = ld2_l2(newrow + 2 * l);
    rd = ld2_l2(newrow + row_tail(fac_mp(MP)));
    rr = ld2_l2(newrow + row_tail(fac_mp(MP)) + 2);
  }
#endif
  const long long tq0 = cycle_now();
  const int64_t first_counted = (it > p.drop) ? it : p.drop;  // Tabulate(): main.cpp:392
#if defined(__CUDA_ARCH__)
  // two-CTA pipeline: the builder's replica starts on the move while this CTA applies it
  const bool publish = m.pipe && m.pipe_rank == 0 && m.pipe_debug != 2;  // (developer switch BN_B200_PIPE=5: no moves published)
  const long long tp0 = cycle_now();
  if (publish && l == 0)
    pipe_publish(m, s.n_moves, type, c, j, type == 2 ? del : 0, ag, new_score,
                 ((type == 2 && k == MP) ? LOG_UNFULL : 0) | ((type == 1 ? k == 0 : k == 1) ? LOG_HP : 0));
  s.pw_cyc[5] += cycle_now() - tp0;
#endif
  Warp::sync();
  if (l == 0 && m.npar_freq) {
    // freqNpar[p][Npar[p]]++ of Tabulate() (Bayes-networks/main.cpp:291): the old count held
    // from npar_since[c] up to this iteration
    const int64_t cnt = first_counted - m.npar_since[c];
    if (cnt > 0) m.npar_freq[(int64_t)c * (MP + 1) + k] += (int)cnt;
    m.npar_since[c] = (int)first_counted;
  }
  if (type == 1) {
    if (l == 0) {
      pc[k] = j; m.npar[c] = k + 1;
      if (m.edge_freq) bc[k] = (int)first_counted;  // birth iterations only feed the tabulation
      m.base[c] = new_score;
      if (KMAX > 8 && !newrow) factor_current<KMAX>(p, m, c);
    }
    if (k == 0) {
      Warp::sync();
      hp_insert(m, s.n_haspar, c);  // rank from the bitset BEFORE c's bit is set
      if (l == 0) m.haspar[c >> 5] |= 1u << (c & 31);
      s.n_haspar++;
    }
    s.te_true++; s.agree_true += ag;
    Warp::sync();
    const long long tq1 = cycle_now();
    if (m.anc_freq) anc_tab_add(p, m, j, c, -(int)first_counted);  // (reads the rows before the update)
    if (m.mb) mb_move(p, m, c, k, j, 1, (int)first_counted);        // (c's list before j: pc[0..k))
    anc_after_add(p, m, j, c, s.anc_changed);
    (void)tq1;
  } else {
    if (l == 0) {
      if (m.edge_freq) {
        const int64_t cnt = first_counted - bc[del];
        if (cnt > 0) m.edge_freq[(int64_t)j + (int64_t)c * p.P] += (int)cnt;
      }
      for (int e = del; e + 1 < k; e++) pc[e] = pc[e + 1];
      if (m.edge_freq)
        for (int e = del; e + 1 < k; e++) bc[e] = bc[e + 1];
      pc[k - 1] = -1;
      m.npar[c] = k - 1;
      // MaxPar > 8: the node's factor follows by a Givens downdate (a fresh factorisation when the
      // block holds none); later proposals at c are compared with the score of the new factor
      if (KMAX > 8) {
        const double rss_old = F[fac_tail(fac_mp(MP))];
        m.base[c] = (rss_old == rss_old) ? factor_downdate<KMAX>(F, k, del, p.sc, fac_mp(MP)) : factor_current<KMAX>(p, m, c);
      } else {
        m.base[c] = new_score;
      }
    }
    if (k == 1) {
      Warp::sync();
      hp_remove(m, s.n_haspar, c);
      if (l == 0) m.haspar[c >> 5] &= ~(1u << (c & 31));
      s.n_haspar--;
    }
    s.te_true--; s.agree_true -= ag;
    Warp::sync();
    if (m.mb) mb_move(p, m, c, k - 1, j, -1, (int)first_counted);  // (c's list after the shift)
    const long long tq1 = cycle_now();
#if defined(BN_PHASE_CYCLES)
    anc_after_delete(p, m, c, s.anc_changed, s.cyc);   // [6] collect+clear, [7] first barrier, [8] round work, [11] round barriers
#else
    anc_after_delete(p, m, c, s.anc_changed);
#endif
    if (m.anc_freq && s.anc_changed) anc_tab_del(p, m, c, (int)first_counted);
    s.cyc[9] += tq1 - tq0; s.cyc[10] += cycle_now() - tq1;
  }
  if (KMAX > 8 && type == 1 && newrow) {
    const int mp = fac_mp(MP);
#if defined(__CUDA_ARCH__)
    const double r = rsqrt_f64(rd.x);
    if (2 * l <= k) {
      if (2 * l == k) rv.x = r;
      if (2 * l + 1 == k) rv.y = r;
      *(D2*)(F + fac_row(k) + 2 * l) = rv;
    }
    if (l == 0) { F[fac_zoff(mp) + k] = rd.y * r; F[fac_tail(mp)] = rr.x; }
#else
    const double r = rsqrt_f64(newrow[row_tail(mp)]);
    for (int t = 0; t < k; t++) F[fac_row(k) + t] = newrow[t];
    F[fac_row(k) + k] = r;
    F[fac_zoff(mp) + k] = newrow[row_tail(mp) + 1] * r; F[fac_tail(mp)] = newrow[row_tail(mp) + 2];
#endif
  }
  if (m.nver) {  // the deletion scores of c carry the old count: no longer valid
    if (l == 0) m.nver[c]++;
  } else if (m.dscore) {  // the deletion scores of c are no longer valid
    double* dc = m.dscore + (uint32_t)c * (uint32_t)MP;
    for (int e = l; e < MP; e += Warp::NL) dc[e] = nan_sentinel();
  }
#if defined(__CUDA_ARCH__)
  if (publish && l == 0 && s.anc_changed) m.pipe->log[s.n_moves % PIPE_LOG] |= LOG_ANC;
#endif
  if (s.n_moves < p.moves_capacity) {
    if (l == 0) {
      int* mv = m.moves + (int64_t)s.n_moves * 4;
      mv[0] = (int)it; mv[1] = type; mv[2] = c; mv[3] = j;
    }
  }
  s.n_moves++;
  s.gll_ok = 0;
  Warp::sync();
}

template <int KMAX>
BN_HD void apply_move(const ChainParams& p, ChainMem& m, ChainScalars& s, int64_t it,
                      const WindowSlots& ws, int i) {
  const int ag = p.sim_edge[(int64_t)ws.parent[i] + (int64_t)ws.child[i] * p.P] ? 1 : 0;
  apply_move_vals<KMAX>(p, m, s, it, ws.type[i], ws.child[i], ws.parent[i], ws.pos[i], ws.new_score[i], ag, nullptr);
}

// Commit slots [0, ncommit): all but possibly the last are rejections/invalid.
template <int KMAX>
BN_HD void commit(const ChainParams& p, ChainMem& m, ChainScalars& s, const WindowSlots& ws,
                  int ncommit) {
  // One lane per slot: the counters are ballots + popcounts instead of a sequential loop.
  // Only the last committed slot can be an acceptance; rows logged before it see the
  // pre-move graph, its own row (if any) the post-move graph.
  const int l = Warp::lane();
  for (int i0 = 0; i0 < ncommit; i0 += Warp::NL) {
    const int i = i0 + l;
    const bool in = i < ncommit;
    const int64_t it = s.iter + i;
    const bool valid = in && ws.valid[in ? i : 0];
    const int type = in ? ws.type[i] : 0;
    const bool counted = valid && it >= p.drop;  // src/network.h:331, src/bayesnet_mcmc.cpp:58
    const bool acc = valid && ws.accept[in ? i : 0];
    const uint32_t m_valid = Warp::ballot(valid);
    const uint32_t m_inval = Warp::ballot(in && !valid);
    const uint32_t m_p1 = Warp::ballot(counted && type == 1);
    const uint32_t m_p2 = Warp::ballot(counted && type == 2);
    const uint32_t m_r1 = Warp::ballot(counted && type == 1 && !acc);
    const uint32_t m_r2 = Warp::ballot(counted && type == 2 && !acc);
    const uint32_t m_npd = Warp::ballot(valid && ws.nonpd[in ? i : 0]);
    const uint32_t m_acc = Warp::ballot(acc);
    const uint32_t m_log = Warp::ballot(valid && ((int)it % p.output_every == 0));  // :63-65 (n_iter is an int)
    const int kk = valid ? ws.kk[i] : 0;
    const int bytes = Warp::sum(valid ? 4 * (kk + 1) * (kk + 2) + 8 : 0);
    // rows of rejected iterations (pre-move graph), in order
    uint32_t lg = m_log & ~m_acc;
    while (lg) {
      const int b = ffs32(lg) - 1;
      lg &= lg - 1;
      const uint32_t upto = (b == 31) ? 0xffffffffu : ((2u << b) - 1u);
      (void)upto;  // (only the last committed slot can be an acceptance)
      write_row(p, m, s, s.iter + i0 + b, ws, i0 + b, s.acc_add, s.acc_del);
    }
    s.valid_iters += popc32(m_valid);
    s.alg_bytes += bytes;
    s.proposed[1] += popc32(m_p1); s.proposed[2] += popc32(m_p2);
    s.reject[0] += popc32(m_inval);  // notValid(), src/network.h:434-437 (not guarded by drop)
    s.reject[1] += popc32(m_r1); s.reject[2] += popc32(m_r2);
    s.n_nonpd += popc32(m_npd);
    if (m_acc) {
      const int b = ffs32(m_acc) - 1;  // == the last committed slot
      const long long ta = cycle_now();
      apply_move<KMAX>(p, m, s, s.iter + i0 + b, ws, i0 + b);
      const long long dt = cycle_now() - ta;
      s.cyc[ws.type[i0 + b] == 1 ? 4 : 5] += dt;
      s.cyc[3] -= dt;
      if (s.iter + i0 + b >= p.drop) { if (ws.type[i0 + b] == 1) s.acc_add++; else s.acc_del++; }
      if (m_log & m_acc) write_row(p, m, s, s.iter + i0 + b, ws, i0 + b, s.acc_add, s.acc_del);
    }
  }
  const int last = ncommit - 1;
  s.valid = ws.valid[last];
  s.te_m = ws.te_m[last];
  s.read_pos = ws.pos_after[last];
  s.iter += ncommit;
  // lanes are not in lockstep: nobody may still be reading the slots when lane 0
  // starts writing the next window's
  Warp::sync();
}

// One epoch of a round: walk the records from relative position *k_io (at most `want`
// iterations, stopping behind the first accepted one) and commit them -- the same bookkeeping
// as commit(), with the slot of iteration s.iter + q living in the registers of lane q.
// Returns the number of iterations committed; *accepted / *acc_c / *acc_type describe the
// accepted move, *stop (WALK_OVF / WALK_STALE / WALK_END or 0) the record that ended the walk.
template <int KMAX>
BN_HD int round_epoch(const ChainParams& p, ChainMem& m, ChainScalars& s, const WindowSlots& ws, int64_t round_pos,
                      int* k_io, int want, int* stop, int* accepted, int* acc_c, int* acc_type) {
  const int l = Warp::lane();
  int k = *k_io, v = s.valid, n = 0, myk = 0, myvalid = 0, acc = 0, k_acc = 0;
  *stop = 0;
  // pointer chase over the walk words: `valid` is only assigned by additions
  // (src/bayesnet_mcmc.cpp:50-52), the acceptance uniform is drawn for valid iterations only
  // (records that cannot be consumed -- overflow, stale, behind the round -- carry a stop mark,
  // so the loop has one rarely taken exit besides its counter)
  while (n < want) {
    const int w = ws.t_walk[k];
    const int f = w >> (16 + v);  // bit 0 outgoing valid, bit 2 accepted, bit 4 stop mark
    if (f & 0x14) {               // rare: the common path has this one branch besides the counter
      if (f & 0x10) { *stop = w; break; }
      if (l == n) { myk = k; myvalid = 1; }  // an accepted iteration is a valid one
      acc = 1; k_acc = k;
      k += (w >> (v << 3)) & 0xff;
      v = 1;
      n++;
      break;
    }
    if (l == n) { myk = k; myvalid = f & 1; }
    k += (w >> (v << 3)) & 0xff;
    v = f & 1;
    n++;
  }
  *accepted = acc;
  if (n == 0) return 0;
  const long long tc = cycle_now();
  const int last = n - 1;
  const bool in = l < n;
  const int rec = in ? ws.t_rec[myk] : 0;
  const int type = (rec & REC_TYPE) ? 2 : 1;
  const bool valid = in && myvalid;
  const int it0 = (int)s.iter, it = it0 + l;  // n_iter is an int
  const bool counted = valid && it >= p.drop;  // src/network.h:331, src/bayesnet_mcmc.cpp:58
  const bool is_acc = acc && l == last;        // only the last slot can be an acceptance
  // statistics stay lane-private (no ballots or reductions per epoch)
  // (constant indices only: a run-time index would move the scalars to local memory)
  s.lane_prop[1] += (counted && type == 1) ? 1 : 0;
  s.lane_prop[2] += (counted && type == 2) ? 1 : 0;
  s.lane_rej[1] += (counted && type == 1 && !is_acc) ? 1 : 0;
  s.lane_rej[2] += (counted && type == 2 && !is_acc) ? 1 : 0;
  s.lane_rej[0] += (in && !myvalid) ? 1 : 0;  // notValid(), src/network.h:434-437 (not guarded by drop)
  if (valid) {
    const int kk = rec >> REC_KK_SHIFT;
    s.lane_valid++;
    s.lane_bytes += 4 * (kk + 1) * (kk + 2) + 8;
    if (rec & REC_NPD) s.lane_nonpd++;
  }
  // logged iterations (i % output == 0, :63-65): s.next_log is the next multiple at or behind it0
  int log_acc = 0, fn_acc = 0, fp_acc = 0;
  if (s.next_log < it0 + n) {  // rare
    // members left by the last LogPrior(): the proposed graph for valid iterations
    // (checker(), src/network.h:333), the current graph otherwise
    const int ag = (rec & REC_AG) ? 1 : 0;
    const int te_m = valid ? s.te_true + (type == 1 ? 1 : -1) : s.te_true;
    const int ag_new = valid ? s.agree_true + (type == 1 ? ag : -ag) : s.agree_true;
    const int fp_m = te_m - ag_new, fn_m = p.n_sim_edges - ag_new;
    const int child = in ? ws.t_c[myk] : 0;
    do {
      const int b = s.next_log - it0;
      const int b_valid = Warp::shfl(valid ? 1 : 0, b), b_child = Warp::shfl(child, b), b_type = Warp::shfl(type, b);
      const int b_fn = Warp::shfl(fn_m, b), b_fp = Warp::shfl(fp_m, b);
      if (acc && b == last) { log_acc = 1; fn_acc = b_fn; fp_acc = b_fp; }  // its row sees the post-move graph
      else if (b_valid) write_row_vals(p, m, s, it0 + b, b_child, b_type, b_fn, b_fp, s.acc_add, s.acc_del);
      s.next_log += p.output_every;
    } while (s.next_log < it0 + n);
  }
  const int info_last = Warp::shfl((valid ? 4 : 0) | type, last);
  long long dt = 0;
  if (acc) {
    const int c = ws.t_c[k_acc], a_type = (ws.t_rec[k_acc] & REC_TYPE) ? 2 : 1;
    const long long ta = cycle_now();
    apply_move_vals<KMAX>(p, m, s, it0 + last, a_type, c, ws.t_j[k_acc], ws.t_e[k_acc], ws.t_score[k_acc],
                          (ws.t_rec[k_acc] & REC_AG) ? 1 : 0,
                          KMAX > 8 ? m.rowbuf + (uint32_t)k_acc * (uint32_t)row_stride(fac_mp(p.max_par)) : nullptr);
    dt = cycle_now() - ta;
    s.cyc[a_type == 1 ? 4 : 5] += dt;
    if (it0 + last >= p.drop) { if (a_type == 1) s.acc_add++; else s.acc_del++; }
    if (log_acc) write_row_vals(p, m, s, it0 + last, c, a_type, fn_acc, fp_acc, s.acc_add, s.acc_del);
    *acc_c = c; *acc_type = a_type;
    // (the move was applied: te_true already counts it)
    s.te_m = s.te_true;
  } else {
    s.te_m = (info_last & 4) ? s.te_true + ((info_last & 3) == 1 ? 1 : -1) : s.te_true;
  }
  s.valid = v;
  s.read_pos = round_pos + k;
  s.iter += n;
  // the caller charges the whole call to the walk: move the commit part and the move over
  const long long tcommit = cycle_now() - tc;
  s.cyc[3] += tcommit - dt;
  s.cyc[2] -= tcommit;
  *k_io = k;
  return n;
}

// One round: records for REPLAY_POS positions, then walk / commit / repair epochs.
template <int KMAX>
BN_HD void run_round(const ChainParams& p, ChainMem& m, ChainScalars& s, RngStream& rng, WindowSlots& ws) {
  long long t0 = cycle_now();
  RoundCtx rc;
  rc.pos = s.read_pos; rc.hi = rng.gen_hi;
  rc.n_haspar = s.n_haspar; rc.te_true = s.te_true; rc.agree_true = s.agree_true;
  rc.redo_from = -1; rc.redo_mode = 0;
  while (s.next_log < (int)s.iter) s.next_log += p.output_every;  // (after sequential windows; else no step)
  team_records<KMAX>(p, m, rc, rng.ubuf, ws);
  long long t1 = cycle_now();
  s.cyc[1] += t1 - t0;
  int k = 0;
  for (;;) {
    t0 = cycle_now();
    int want = WIN < Warp::NL ? WIN : Warp::NL;  // one lane per iteration of the epoch
    if ((int64_t)want > p.n_iter - s.iter) want = (int)(p.n_iter - s.iter);
    if (want <= 0) break;
    int stop = 0, accepted = 0, c = 0, type = 0;
    const int k0 = k, nh0 = s.n_haspar;
    const int n = round_epoch<KMAX>(p, m, s, ws, rc.pos, &k, want, &stop, &accepted, &c, &type);
    s.cyc[2] += cycle_now() - t0;
    if (n == 0) {
      // one iteration needs more uniforms than a record can count: the sequential path takes it
      if (stop == WALK_OVF && k0 == 0) s.need_full = 1;
      break;
    }
    s.need_full = 0;
    s.slots_sim += n;
    if (stop) break;  // the next record is overflowed, stale or behind this round's positions
    if (accepted) {
      // TotalEdges < 4 ends the rounds (sequential windows take over).  A child that reaches
      // MaxPar only affects its own records; one that drops below it affects the draws that
      // skipped it.
      if (s.te_true < 4) break;
      if (k >= REPLAY_POS) break;
      const int unfull = (type == 2 && m.npar[c] == p.max_par - 1) ? 1 : 0;
      t0 = cycle_now();
      team_repair(p, m, ws, c, unfull, s.anc_changed, k);
      if (s.n_haspar != nh0) {
        // the set of nodes with parents changed: the deletion records behind the walk are redone
        rc.n_haspar = s.n_haspar; rc.te_true = s.te_true; rc.agree_true = s.agree_true;
        rc.redo_from = k; rc.redo_mode = 0;
        team_records<KMAX>(p, m, rc, rng.ubuf, ws);
      }
      s.cyc[2] += cycle_now() - t0;
    }
  }
}

#if defined(__CUDACC__)
// ---------------------------------------------------------------------------
// Two-CTA pipeline, chain side (rank 0; see PipeLink).
// ---------------------------------------------------------------------------
__device__ __forceinline__ void pipe_request(const ChainMem& m, ChainScalars& s, int64_t pos) {
  s.pw_out_seq++; s.pw_out = 1; s.pw_out_pos = pos;
  if (Warp::lane() == 0)
    st_peer64(peer_addr(&m.pipe->req, 1), ((unsigned long long)pos << 16) | (unsigned long long)(s.pw_out_seq & 0xffff));
}

// make ws hold the window that contains s.read_pos: the one the builder was asked for ahead of time
// if the walk arrived there, else a fresh request; then repair it for the moves it has not seen
// (returns the number of moves the builder's replica had applied when it built the window)
template <int KMAX>
__device__ __forceinline__ int pipe_acquire(const ChainParams& p, ChainMem& m, ChainScalars& s, RngStream& rng,
                                            WindowSlots& ws) {
  PipeLink* lk = m.pipe;
  const int l = Warp::lane();
  const int64_t want = (s.pw_cur >= 0 && s.read_pos >= s.pw_cur + PIPE_WIN && s.read_pos < s.pw_cur + 2 * PIPE_WIN)
                           ? s.pw_cur + PIPE_WIN : s.read_pos;
  const long long ta0 = cycle_now();
  int applied = 0;
  for (;;) {
    if (!s.pw_out) pipe_request(m, s, want);
    unsigned long long rdy = 0ull;
    if (l == 0) {
      long long spins = 0;
      while ((int)((rdy = ld_poll64(&lk->rdy)) & 0xffffull) != (s.pw_out_seq & 0xffff))
        if (++spins > (1ll << 27)) { lk->pad1 = 91; break; }  // (watchdog)
      s.pw_waits += spins ? 1 : 0;
    }
    applied = Warp::shfl((int)(rdy >> 32), 0);
    s.pw_out = 0;
    if (s.pw_out_pos == want) break;
    s.pw_discards++;  // (the walk left the grid: a sequential window, an iteration that outran its record)
  }
  const long long ta1 = cycle_now();
  s.pw_cyc[0] += ta1 - ta0;
  if (l == 0) m.helper[0] = HELPER_PIPE_COPY;
  Warp::sync();
  cta_bar(1);
  cta_bar(2);
  s.pw_cur = want;
  pipe_request(m, s, want + PIPE_WIN);  // the builder goes on with the next window of the grid
  s.pw_cyc[1] += cycle_now() - ta1;
  return applied;
}

// The records in ws are right for the graph after `applied` accepted moves; repair them for the moves
// accepted since: the ones the builder had not seen when it built the window, and the ones a
// sequential window applied while the walk stayed inside the window.
template <int KMAX>
__device__ __forceinline__ void pipe_catch_up(const ChainParams& p, ChainMem& m, ChainScalars& s, RngStream& rng,
                                              WindowSlots& ws, int applied, int fresh) {
  PipeLink* lk = m.pipe;
  const int l = Warp::lane();
  const int64_t want = s.pw_cur;
  const int from = (int)(s.read_pos - want), now = s.n_moves;
  const long long ta2 = cycle_now();
  s.pw_seen = now;
  if (now == applied && !(m.pipe_debug && fresh)) return;
  RoundCtx rc;
  rc.pos = want; rc.hi = rng.gen_hi;
  rc.n_haspar = s.n_haspar; rc.te_true = s.te_true; rc.agree_true = s.agree_true;
  rc.redo_from = from;
  if (now - applied > PIPE_LOG || (m.pipe_debug && fresh)) {  // more moves than the chain remembers: every record is built again
    rc.redo_mode = 2;
    s.pw_rebuilds++;
    team_records<KMAX, true>(p, m, rc, rng.ubuf, ws);
    return;
  }
  int flags = 0;
  for (int i = applied + l; i < now; i += Warp::NL) flags |= lk->log[i % PIPE_LOG];
  const int any_anc = Warp::ballot(flags & LOG_ANC) != 0u, any_hp = Warp::ballot(flags & LOG_HP) != 0u;
  if (l == 0) {
    m.helper[8] = from; m.helper[5] = applied; m.helper[6] = now; m.helper[7] = any_anc;
    m.helper[0] = HELPER_REPAIR_BATCH;
  }
  Warp::sync();
  cta_bar(1);
  cta_bar(2);
  const long long ta3 = cycle_now();
  s.pw_cyc[2] += ta3 - ta2;
  if (any_hp) {  // deletion draws index into the set of nodes with parents: those records are redone
    rc.redo_mode = 0;
    team_records<KMAX, true>(p, m, rc, rng.ubuf, ws);
    s.pw_cyc[3] += cycle_now() - ta3;
  }
}

// One pass over (what is left of) a window: walk / commit / repair epochs as in run_round; the
// records come from the builder, and a stale record under the walk is rebuilt in place.
template <int KMAX>
__device__ __forceinline__ void run_round_pipe(const ChainParams& p, ChainMem& m, ChainScalars& s, RngStream& rng,
                                               WindowSlots& ws) {
  long long t0 = cycle_now();
  {
    const bool fresh = s.pw_cur < 0 || s.read_pos < s.pw_cur || s.read_pos >= s.pw_cur + PIPE_WIN;
    const int applied = fresh ? pipe_acquire<KMAX>(p, m, s, rng, ws) : s.pw_seen;
    pipe_catch_up<KMAX>(p, m, s, rng, ws, applied, fresh ? 1 : 0);
  }
  RoundCtx rc;
  rc.pos = s.pw_cur; rc.hi = rng.gen_hi;
  rc.n_haspar = s.n_haspar; rc.te_true = s.te_true; rc.agree_true = s.agree_true;
  rc.redo_from = -1; rc.redo_mode = 0;
  while (s.next_log < (int)s.iter) s.next_log += p.output_every;  // (after sequential windows; else no step)
  s.cyc[1] += cycle_now() - t0;
  int k = (int)(s.read_pos - s.pw_cur);
  for (;;) {
    t0 = cycle_now();
    int want = WIN < Warp::NL ? WIN : Warp::NL;  // one lane per iteration of the epoch
    if ((int64_t)want > p.n_iter - s.iter) want = (int)(p.n_iter - s.iter);
    if (want <= 0) break;
    int stop = 0, accepted = 0, c = 0, type = 0;
    const int nh0 = s.n_haspar;
    const int n = round_epoch<KMAX>(p, m, s, ws, rc.pos, &k, want, &stop, &accepted, &c, &type);
    s.cyc[2] += cycle_now() - t0;
    if (n > 0) { s.need_full = 0; s.slots_sim += n; }
    if (stop) {
      if (stop == WALK_STALE) {
        // an accepted move changed what this record depends on: the stale records behind the walk
        // are built again from the current graph, and the walk goes on
        t0 = cycle_now();
        rc.n_haspar = s.n_haspar; rc.te_true = s.te_true; rc.agree_true = s.agree_true;
        rc.redo_from = k; rc.redo_mode = 1;
        s.pw_rebuilds++;
        team_records<KMAX, true>(p, m, rc, rng.ubuf, ws);
        s.cyc[1] += cycle_now() - t0;
        s.pw_cyc[4] += cycle_now() - t0;
        continue;
      }
      // one iteration needs more uniforms than a record can count: the sequential path takes it
      if (stop == WALK_OVF) s.need_full = 1;
      break;  // WALK_END: the next window
    }
    if (n == 0) break;
    if (accepted) {
      if (s.te_true < 4) break;  // (sequential windows take over)
      if (k >= PIPE_WIN) break;
      const int unfull = (type == 2 && m.npar[c] == p.max_par - 1) ? 1 : 0;
      t0 = cycle_now();
      team_repair(p, m, ws, c, unfull, s.anc_changed, k);
      if (s.n_haspar != nh0) {
        rc.n_haspar = s.n_haspar; rc.te_true = s.te_true; rc.agree_true = s.agree_true;
        rc.redo_from = k; rc.redo_mode = 0;
        team_records<KMAX, true>(p, m, rc, rng.ubuf, ws);
      }
      s.pw_seen = s.n_moves;
      s.cyc[2] += cycle_now() - t0;
    }
  }
}

// ---------------------------------------------------------------------------
// Two-CTA pipeline, builder side (rank 1, its chain warp; the helper warps sit in helper_loop).
// ---------------------------------------------------------------------------
template <int KMAX>
__device__ __forceinline__ void shadow_loop(const ChainParams& p, ChainMem& m, ChainScalars& s, RngStream& rng,
                                            WindowSlots& ws) {
  const int l = Warp::lane();
  chain_init<KMAX>(p, m, s, rng);
  const WhJump jump = wh_jump_for_thread();
  PipeLink* lk = m.pipe;
  int seq = 0;
  for (;;) {
    // the replica follows the chain: same move, same team operations on this CTA's copy
    // ONE lane reads the mailbox and the warp takes its values: 32 lanes polling for themselves are not
    // guaranteed to execute a load together, and a message that lands between two lanes' loads splits the
    // warp for good (some lanes serve the request, the others still wait for it with their own `seq` --
    // the cause of a hang seen in about one launch in fifty before this was fixed)
    int w0 = 0, w1 = 0, w2 = 0, w3 = 0, ex = 0, rq_lo = 0, rq_hi = 0;
    if (l == 0) {
      ld_poll128(&lk->mq[s.n_moves % PIPE_MQ][0], w0, w1, w2, w3);
      ex = ld_poll(&lk->req_exit);
      const unsigned long long rq = ld_poll64(&lk->req);
      rq_lo = (int)(rq & 0xffffffffull); rq_hi = (int)(rq >> 32);
    }
    w0 = Warp::shfl(w0, 0);
    const bool has_move = w0 == s.n_moves + 1;
    if (has_move) { w1 = Warp::shfl(w1, 0); w2 = Warp::shfl(w2, 0); w3 = Warp::shfl(w3, 0); }  // (warp-uniform branch)
    else { ex = Warp::shfl(ex, 0); rq_lo = Warp::shfl(rq_lo, 0); rq_hi = Warp::shfl(rq_hi, 0); }
    if (has_move && ((uint32_t)w1 >> 27) == (uint32_t)((s.n_moves + 1) & 31)) {
      if (l == 0) st_peer(peer_addr(&lk->mq_tail, 0), s.n_moves + 1);  // (the message is in registers)
      const double sc = __longlong_as_double(((long long)w3 << 32) | (long long)(uint32_t)w2);
      apply_move_vals<KMAX>(p, m, s, 0, ((w1 >> 22) & 1) + 1, w1 & 0x7ff, (w1 >> 11) & 0x7ff, (w1 >> 23) & 7, sc,
                            (w1 >> 26) & 1, nullptr);
      if (s.status) break;  // (the move did not fit the replica: stop serving -- the chain's watchdog reports it)
      continue;
    }
    if (ex) break;
    const unsigned long long req = ((unsigned long long)(uint32_t)rq_hi << 32) | (unsigned long long)(uint32_t)rq_lo;
    if ((int)(req & 0xffffull) == seq) continue;
    seq = (int)(req & 0xffffull);
    const int64_t pos = (int64_t)(req >> 16);
    if (rng.kind == RNG_WH) team_fill_wh(m, rng, pos, jump);
    else rng_top_up(rng, pos);
    RoundCtx rc;
    rc.pos = pos; rc.hi = rng.gen_hi;
    rc.n_haspar = s.n_haspar; rc.te_true = s.te_true; rc.agree_true = s.agree_true;
    rc.redo_from = -1; rc.redo_mode = 0;
    team_records<KMAX, true>(p, m, rc, rng.ubuf, ws);
    // (the records are in this CTA's shared memory -- team_records ends with a CTA barrier -- before the flag leaves)
    if (l == 0) st_peer64(peer_addr(&lk->rdy, 0), ((unsigned long long)(uint32_t)s.n_moves << 32) | (unsigned long long)seq);
    Warp::sync();
  }
}
#endif

// ---------------------------------------------------------------------------
// The whole chain.
// ---------------------------------------------------------------------------
// PIPE (device only): the two-CTA form -- the records of a window come from the builder CTA
template <int KMAX, bool PIPE = false>
BN_HD void run_chain(const ChainParams& p, ChainMem& m, ChainScalars& s, RngStream& rng,
                     WindowSlots& ws) {
  const int l = Warp::lane();
  chain_init<KMAX>(p, m, s, rng);
  for (int i = (PIPE ? PIPE_WIN : REPLAY_POS) + l; i < 2 * REPLAY_POS; i += Warp::NL) ws.t_walk[i] = WALK_END;
  Warp::sync();
#if defined(__CUDA_ARCH__)
  const WhJump jump = wh_jump_for_thread();
#endif
  while (s.iter < p.n_iter && s.status == 0) {
    long long t0 = cycle_now();
#if defined(__CUDA_ARCH__)
    if constexpr (PIPE) {
      const int wd = m.pipe->pad1;  // a mailbox watchdog fired (the peer CTA stopped answering): an error, never a hang
      if (wd) { s.status = wd; break; }
    }
    if (rng.kind == RNG_WH && m.helper) {
      // the CTA appends 128 uniforms at a time (>= 385 ahead of the read position afterwards)
      team_fill_wh(m, rng, s.read_pos, jump);
      if (s.need_full) rng_top_up(rng, s.read_pos);
    } else
#endif
      rng_top_up(rng, s.read_pos);
    long long t1 = cycle_now();
    s.cyc[0] += t1 - t0;
    s.windows++;
    // position-parallel rounds need `TotalEdges < 3` to be impossible
    if (s.te_true >= 4 && s.te_m >= 3 && !s.need_full) {
#if defined(__CUDA_ARCH__)
      if constexpr (PIPE) { run_round_pipe<KMAX>(p, m, s, rng, ws); continue; }
#endif
      if constexpr (!PIPE) run_round<KMAX>(p, m, s, rng, ws);
      continue;
    }
    // sequential windows (first iterations of a chain, tiny graphs)
    int want = s.need_full ? 1 : s.win;
    if ((int64_t)want > p.n_iter - s.iter) want = (int)(p.n_iter - s.iter);
    int overflow = 0;
    int n = phase_a(p, m, s, rng, ws, want, &overflow);
    if (n == 0) {
      if (!s.need_full) { s.need_full = 1; continue; }  // top the ring up completely and retry
      // one iteration needs more uniforms than the ring holds (legal nodes are rare): no limit
      n = phase_a(p, m, s, rng, ws, 1, &overflow, 1);
      // BN_ERR_NO_LEGAL_PROPOSAL: no legal node exists at all; BN_ERR_CAPACITY: the replay buffer ran out
      if (n == 0) { s.status = (overflow == 3) ? 6 : 4; break; }
    }
    s.need_full = 0;
    t0 = cycle_now();
    s.cyc[1] += t0 - t1;
    s.slots_sim += n;
    for (int i = l; i < n; i += Warp::NL) phase_bc<KMAX>(p, m, s, ws, i);
    Warp::sync();
    int first = -1;
    for (int i0 = 0; i0 < n && first < 0; i0 += Warp::NL) {
      const int i = i0 + l;
      const uint32_t am = Warp::ballot(i < n && ws.valid[i < n ? i : 0] && ws.accept[i < n ? i : 0]);
      if (am) first = i0 + ffs32(am) - 1;
    }
    t1 = cycle_now();
    s.cyc[2] += t1 - t0;
    const int ncommit = (first >= 0) ? first + 1 : n;
    commit<KMAX>(p, m, s, ws, ncommit);
    s.cyc[3] += cycle_now() - t1;
    if (first >= 0) {
      int w = 2 * (first + 1);
      s.win = w < 2 ? 2 : (w > WIN ? WIN : w);
    } else {
      int w = 2 * s.win;
      s.win = w > WIN ? WIN : w;
    }
  }
  // fold the lane-private statistics of the rounds into the warp-uniform totals
  for (int t = 0; t < 3; t++) { s.proposed[t] += Warp::sum(s.lane_prop[t]); s.reject[t] += Warp::sum(s.lane_rej[t]); }
  s.n_nonpd += Warp::sum(s.lane_nonpd);
  s.valid_iters += Warp::sum(s.lane_valid);
  s.alg_bytes += (int64_t)Warp::sum((long long)s.lane_bytes);
  // flush the posterior tabulation of the surviving edges / parent counts
  if (m.npar_freq) {
    Warp::sync();
    for (int c = l; c < p.P; c += Warp::NL) {
      const int64_t cnt = (int64_t)p.n_iter - m.npar_since[c];
      if (cnt > 0) m.npar_freq[(int64_t)c * (p.max_par + 1) + m.npar[c]] += (int)cnt;
    }
  }
  if (m.edge_freq) {
    Warp::sync();
    for (int c = l; c < p.P; c += Warp::NL) {
      const int k = m.npar[c];
      for (int e = 0; e < k; e++) {
        const int64_t cnt = (int64_t)p.n_iter - m.born[(int64_t)c * p.max_par + e];
        if (cnt > 0) m.edge_freq[(int64_t)m.par[(int64_t)c * p.max_par + e] + (int64_t)c * p.P] += (int)cnt;
      }
    }
  }
  if (m.anc_freq) {
    Warp::sync();
    anc_tab_all(p, m, p.n_iter > p.drop ? p.n_iter : p.drop);  // the paths of the final graph, up to the end
  }
  if (m.mb) {
    Warp::sync();
    mb_graph(p, m, -1, p.n_iter > p.drop ? p.n_iter : p.drop);  // the blanket pairs of the final graph
  }
  if (m.best) {
    Warp::sync();
    best_finish(p, m, s);
  }
  Warp::sync();
}

}  // namespace bn
