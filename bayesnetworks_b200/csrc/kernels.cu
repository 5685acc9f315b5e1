// K2 (batched proposal scoring), K3 (chains), K4 (node scores) -- device entry points.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include <type_traits>

#include "chain_core.cuh"
#include "kernels.h"
#include "sweep_log.cuh"

namespace bn {

// ---------------------------------------------------------------------------
// K3: one CTA of eight warps per chain, persistent for the whole run (chain_core.cuh).  Warp 0
// owns the chain; warps 1-7 park on a named barrier and join the team operations (position
// records, record repair, ancestor-row updates, Wichmann-Hill refill).  The per-chain state
// (parent lists, scores, ancestor bitsets, scratch) lives in the CTA's dynamic shared memory
// when it fits (1,000 nodes x MaxPar 8: 202 KB), else in global memory; the Gram is read with
// L2-only loads.
// ---------------------------------------------------------------------------
// ALL_SMEM: every per-chain array of the plan sits in dynamic shared memory, so the pointers
// have a provable shared-memory provenance and the state accesses compile to LDS/STS
// instead of generic loads.
// WITH_STATE: the chains start from supplied graphs / resume states or export their state, tabulate
// ancestor relations or Markov blankets, or track the best graph (ChainWorkspace.with_state).  Without it the
// start pointers, anc_freq, best and mb stay null at compile time, so chain_init folds to the start of
// initial_network and the steady-state loop compiles as it did before resumable chains existed (a per-chain
// end iteration would hold a register for the whole loop).
template <int KMAX, bool ALL_SMEM, bool WITH_STATE>
__global__ void __launch_bounds__((HELPER_WARPS + 1) * 32, 1) chain_kernel(ChainParams p, ChainWorkspace w, ChainRngArgs ra,
                                                   ChainSmemPlan sm, ChainResult* __restrict__ results) {
  __shared__ double ubuf[RNG_CAP];
  __shared__ WindowSlots ws;
  __shared__ int helper_cmd[HELPER_WORDS];
  __shared__ double dof_ratio[KMAX + 2];
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ch = blockIdx.x;
  const int64_t P = p.P, MP = p.max_par, W = p.W;

  ChainMem m;
  int* g_par = w.par + ch * P * MP;
  int* g_npar = w.npar + ch * P;
  m.born = w.born + ch * P * MP;
  if constexpr (ALL_SMEM) {
    m.par = (int*)(dyn_smem + sm.off_par);
    m.npar = (int*)(dyn_smem + sm.off_npar);
    m.base = (double*)(dyn_smem + sm.off_base);
    m.anc = (uint32_t*)(dyn_smem + sm.off_anc);
    m.haspar = (uint32_t*)(dyn_smem + sm.off_haspar);
    m.hp_list = (int*)(dyn_smem + sm.off_hplist);
    m.scratch = (int*)(dyn_smem + sm.off_scratch);
  } else {
    m.par = sm.off_par >= 0 ? (int*)(dyn_smem + sm.off_par) : g_par;
    m.npar = sm.off_npar >= 0 ? (int*)(dyn_smem + sm.off_npar) : g_npar;
    m.base = sm.off_base >= 0 ? (double*)(dyn_smem + sm.off_base) : w.base + ch * P;
    m.anc = sm.off_anc >= 0 ? (uint32_t*)(dyn_smem + sm.off_anc) : w.anc + ch * P * (int64_t)p.Ws;
    m.haspar = sm.off_haspar >= 0 ? (uint32_t*)(dyn_smem + sm.off_haspar) : w.haspar + ch * W;
    m.hp_list = sm.off_hplist >= 0 ? (int*)(dyn_smem + sm.off_hplist) : w.hp_list + ch * P;
    m.scratch = sm.off_scratch >= 0 ? (int*)(dyn_smem + sm.off_scratch) : w.scratch + (int64_t)ch * w.scratch_n;
  }
  const int64_t cap = p.trace_capacity;
  m.t_iter = w.t_iter + ch * cap; m.t_changed = w.t_changed + ch * cap;
  m.t_movetype = w.t_movetype + ch * cap; m.t_gll = w.t_gll + ch * cap;
  m.t_add = w.t_add + ch * cap; m.t_del = w.t_del + ch * cap;
  m.t_fn = w.t_fn + ch * cap; m.t_fp = w.t_fp + ch * cap;
  m.moves = w.moves ? w.moves + (int64_t)ch * p.moves_capacity * 4 : nullptr;
  m.edge_freq = w.edge_freq ? w.edge_freq + ch * P * P : nullptr;
  m.npar_freq = w.npar_freq ? w.npar_freq + ch * P * (MP + 1) : nullptr;
  m.npar_since = w.npar_since ? w.npar_since + ch * P : nullptr;
  m.dscore = w.dscore ? w.dscore + ch * P * MP : nullptr;
  m.fac = w.fac ? w.fac + ch * P * fac_stride(fac_mp(p.max_par)) : nullptr;   // (MaxPar > 8 only)
  m.rowbuf = w.rowbuf ? w.rowbuf + (int64_t)ch * REPLAY_POS * row_stride(fac_mp(p.max_par)) : nullptr;
  m.helper = helper_cmd;
  if constexpr (WITH_STATE) {
    if (w.start_par) { m.start_par = w.start_par + ch * P * MP; m.start_npar = w.start_npar + ch * P; }
    if (w.start) m.start = w.start + ch;
    if (w.scores_in) m.base_in = w.base + ch * P;
    if (w.anc_freq) m.anc_freq = w.anc_freq + ch * P * P;
    if (w.best) m.best = w.best + ch;
    if (w.mb) m.mb = w.mb + ch;
  }

  RngStream rng;
  if (ra.kind == RNG_WH)
    rng_init_wh(rng, ra.seeds[3 * ch], ra.seeds[3 * ch + 1], ra.seeds[3 * ch + 2], ubuf);
  else if (ra.kind == RNG_RMT)
    rng_init_rmt(rng, ra.mt_states + (int64_t)ch * 624, ra.mt_pos[ch], ubuf);
  else
    rng_init_replay(rng, ra.replay + (int64_t)ch * ra.replay_len, ra.replay_len, ubuf);

  ChainParams pp = p;
  set_row_geom(pp);
  // (N - 1) / (N - k - 1), src/network.h:232-234 (int N, int Npar)
  for (int k = threadIdx.x; k < KMAX + 2; k += blockDim.x)
    dof_ratio[k] = (double)(p.n_samples - 1) / (double)(p.n_samples - k - 1);
  pp.sc.half_n = (double)p.n_samples / 2.0;
  pp.sc.ratio = dof_ratio;
  if (!m.moves) pp.moves_capacity = 0;
  if constexpr (WITH_STATE)
    if (w.start) pp.n_iter = (int)(w.start[ch].iter + p.n_iter);  // the chain ends n_iter iterations after its start
  if (ALL_SMEM || sm.off_types >= 0) {
    uint8_t* t = (uint8_t*)(dyn_smem + sm.off_types);
    for (int i = threadIdx.x; i < p.P; i += blockDim.x) t[i] = p.node_type[i];
    pp.node_type = t;
  }
  __syncthreads();
  if (warp != 0) {  // helper warps: parked on a named barrier until the chain needs them
    helper_loop<KMAX>(pp, m, warp, ubuf, ws);
    return;
  }
  ChainScalars s;
  const long long clk0 = clock64();
  run_chain<KMAX>(pp, m, s, rng, ws);
  const long long clk1 = clock64();
  if (lane == 0) helper_cmd[0] = HELPER_EXIT;
  __syncwarp();
  cta_bar(1);

  // final graph back to global memory when it lived in shared memory
  if (ALL_SMEM || sm.off_par >= 0)
    for (int64_t i = lane; i < P * MP; i += 32) g_par[i] = m.par[i];
  if (ALL_SMEM || sm.off_npar >= 0)
    for (int64_t i = lane; i < P; i += 32) g_npar[i] = m.npar[i];
  if constexpr (WITH_STATE)
    if (w.scores_out && (ALL_SMEM || sm.off_base >= 0))
      for (int64_t i = lane; i < P; i += 32) w.base[ch * P + i] = m.base[i];

  if (lane == 0) {
    ChainResult& r = results[ch];
    if constexpr (WITH_STATE) {
      r.end.iter = s.iter; r.end.valid = s.valid; r.end.te_m = s.te_m;
      r.end.acc_add = s.acc_add; r.end.acc_del = s.acc_del;
    }
    r.uniforms = s.read_pos;
    r.valid_iters = s.valid_iters;
    r.alg_bytes = s.alg_bytes;
    for (int t = 0; t < 3; t++) { r.proposed[t] = s.proposed[t]; r.reject[t] = s.reject[t]; }
    r.n_nonpd = s.n_nonpd;
    r.total_edges = s.te_true;
    r.status = s.status;
    r.windows = s.windows;
    r.n_rows = s.n_rows;
    r.n_moves = s.n_moves;
    for (int t = 0; t < 12; t++) r.cyc[t] = s.cyc[t];
    r.slots_sim = s.slots_sim;
    r.cyc_total = clk1 - clk0;
    for (int t = 0; t < 4; t++) r.pipe[t] = 0;
    for (int t = 0; t < 6; t++) r.pipe_cyc[t] = 0;
  }
}

// ---------------------------------------------------------------------------
// K3, two-CTA form (chain_core.cuh: "Two-CTA pipeline"): a chain is a cluster of two CTAs on two
// SMs.  Rank 0 is the chain (walk, commit, accepted moves); rank 1 keeps a replica of the graph
// state and builds the position records of the next window meanwhile.  Only launched when the whole
// per-chain state fits in shared memory (each CTA holds its own copy) and MaxPar <= 8.
// The two roles are separate __noinline__ functions: compiled into one body, the register allocation
// of either role suffers from the other (measured: the ancestor updates of the chain ran at half
// speed).  Everything the roles share sits in DYNAMIC shared memory at plan offsets, so that each
// function derives its pointers from the shared-memory symbol itself (LDS/STS, and the same
// address in both CTAs for mapa).
// ---------------------------------------------------------------------------
struct PipeRoleMem {
  ChainMem m;
  double* ubuf; WindowSlots* ws; double* dof_ratio; uint8_t* types;
};

template <int KMAX>
__device__ __forceinline__ PipeRoleMem pipe_role_setup(const ChainParams& p, const ChainWorkspace& w, const ChainSmemPlan& sm,
                                                      int rank, int ch, unsigned char* dyn_smem) {
  PipeRoleMem r;
  ChainMem& m = r.m;
  const int64_t P = p.P, MP = p.max_par;
  m.par = (int*)(dyn_smem + sm.off_par);
  m.npar = (int*)(dyn_smem + sm.off_npar);
  m.base = (double*)(dyn_smem + sm.off_base);
  m.anc = (uint32_t*)(dyn_smem + sm.off_anc);
  m.haspar = (uint32_t*)(dyn_smem + sm.off_haspar);
  m.hp_list = (int*)(dyn_smem + sm.off_hplist);
  m.scratch = (int*)(dyn_smem + sm.off_scratch);
  m.nver = (uint32_t*)(dyn_smem + sm.off_nver);
  const int64_t cap = p.trace_capacity;
  m.t_iter = w.t_iter + ch * cap; m.t_changed = w.t_changed + ch * cap;
  m.t_movetype = w.t_movetype + ch * cap; m.t_gll = w.t_gll + ch * cap;
  m.t_add = w.t_add + ch * cap; m.t_del = w.t_del + ch * cap;
  m.t_fn = w.t_fn + ch * cap; m.t_fp = w.t_fp + ch * cap;
  // the replica keeps no books: no birth iterations, tabulations, move log
  m.born = rank == 0 ? w.born + ch * P * MP : nullptr;
  m.moves = (rank == 0 && w.moves) ? w.moves + (int64_t)ch * p.moves_capacity * 4 : nullptr;
  m.edge_freq = (rank == 0 && w.edge_freq) ? w.edge_freq + ch * P * P : nullptr;
  m.npar_freq = (rank == 0 && w.npar_freq) ? w.npar_freq + ch * P * (MP + 1) : nullptr;
  m.npar_since = (rank == 0 && w.npar_since) ? w.npar_since + ch * P : nullptr;
  m.dscore = w.dscore + ch * P * MP * 2;  // (score, tag) pairs, shared by the two CTAs
  m.fac = nullptr; m.rowbuf = nullptr;
  m.helper = (volatile int*)(dyn_smem + sm.off_helper);
  m.pipe = (PipeLink*)(dyn_smem + sm.off_link);
  m.pipe_rank = rank;
  m.pipe_debug = w.pipeline == 3 ? 1 : (w.pipeline == 5 ? 2 : 0);
  r.ubuf = (double*)(dyn_smem + sm.off_ubuf);
  r.ws = (WindowSlots*)(dyn_smem + sm.off_ws);
  r.dof_ratio = (double*)(dyn_smem + sm.off_dof);
  r.types = (uint8_t*)(dyn_smem + sm.off_types);
  return r;
}

__device__ __forceinline__ RngStream pipe_role_rng(const ChainRngArgs& ra, int rank, int ch, int n_chains, double* ubuf) {
  RngStream rng;  // each CTA generates the chain's stream for itself
  if (ra.kind == RNG_WH)
    rng_init_wh(rng, ra.seeds[3 * ch], ra.seeds[3 * ch + 1], ra.seeds[3 * ch + 2], ubuf);
  else if (ra.kind == RNG_RMT)
    rng_init_rmt(rng, ra.mt_states + ((int64_t)rank * n_chains + ch) * 624, ra.mt_pos[ch], ubuf);
  else
    rng_init_replay(rng, ra.replay + (int64_t)ch * ra.replay_len, ra.replay_len, ubuf);
  return rng;
}

template <int KMAX>
__device__ __forceinline__ void pipe_role_chain(ChainParams p, ChainWorkspace w, ChainRngArgs ra, ChainSmemPlan sm,
                                             ChainResult* results) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ch = blockIdx.x >> 1;
  PipeRoleMem r = pipe_role_setup<KMAX>(p, w, sm, 0, ch, dyn_smem);
  ChainMem& m = r.m;
  RngStream rng = pipe_role_rng(ra, 0, ch, gridDim.x >> 1, r.ubuf);
  set_row_geom(p);
  p.sc.half_n = (double)p.n_samples / 2.0;
  p.sc.ratio = r.dof_ratio;
  if (!m.moves) p.moves_capacity = 0;
  p.node_type = r.types;
  if (warp != 0) {  // helper warps: parked on a named barrier until the chain needs them
    helper_loop<KMAX, true>(p, m, warp, r.ubuf, *r.ws);
    return;
  }
  ChainScalars s;
  const long long clk0 = clock64();
  run_chain<KMAX, true>(p, m, s, rng, *r.ws);
  const long long clk1 = clock64();
  if (lane == 0) { st_peer(peer_addr(&m.pipe->req_exit, 1), 1); m.helper[0] = HELPER_EXIT; }
  __syncwarp();
  cta_bar(1);
  const int64_t P = p.P, MP = p.max_par;
  int* g_par = w.par + ch * P * MP;
  int* g_npar = w.npar + ch * P;
  for (int64_t i = lane; i < P * MP; i += 32) g_par[i] = m.par[i];
  for (int64_t i = lane; i < P; i += 32) g_npar[i] = m.npar[i];
  if (lane == 0) {
    ChainResult& o = results[ch];
    o.uniforms = s.read_pos;
    o.valid_iters = s.valid_iters;
    o.alg_bytes = s.alg_bytes;
    for (int t = 0; t < 3; t++) { o.proposed[t] = s.proposed[t]; o.reject[t] = s.reject[t]; }
    o.n_nonpd = s.n_nonpd;
    o.total_edges = s.te_true;
    o.status = s.status;
    o.windows = s.windows;
    o.n_rows = s.n_rows;
    o.n_moves = s.n_moves;
    for (int t = 0; t < 12; t++) o.cyc[t] = s.cyc[t];
    o.slots_sim = s.slots_sim;
    o.cyc_total = clk1 - clk0;
    for (int t = 0; t < 6; t++) o.pipe_cyc[t] = s.pw_cyc[t];
    o.pipe[0] = s.pw_out_seq; o.pipe[1] = s.pw_waits; o.pipe[2] = s.pw_discards; o.pipe[3] = s.pw_rebuilds;
  }
}

template <int KMAX>
__device__ __forceinline__ void pipe_role_builder(ChainParams p, ChainWorkspace w, ChainRngArgs ra, ChainSmemPlan sm) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ch = blockIdx.x >> 1;
  PipeRoleMem r = pipe_role_setup<KMAX>(p, w, sm, 1, ch, dyn_smem);
  ChainMem& m = r.m;
  RngStream rng = pipe_role_rng(ra, 1, ch, gridDim.x >> 1, r.ubuf);
  set_row_geom(p);
  p.sc.half_n = (double)p.n_samples / 2.0;
  p.sc.ratio = r.dof_ratio;
  p.moves_capacity = 0;
  p.node_type = r.types;
  if (warp != 0) {
    helper_loop<KMAX, true>(p, m, warp, r.ubuf, *r.ws);
    return;
  }
  ChainScalars s;
  shadow_loop<KMAX>(p, m, s, rng, *r.ws);
  if (lane == 0) m.helper[0] = HELPER_EXIT;
  __syncwarp();
  cta_bar(1);
}

template <int KMAX>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__((HELPER_WARPS + 1) * 32, 1)
    chain_pipe_kernel(ChainParams p, ChainWorkspace w, ChainRngArgs ra, ChainSmemPlan sm, ChainResult* __restrict__ results) {
  extern __shared__ __align__(16) unsigned char dyn_smem[];
  uint32_t rank;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(rank));
  {
    // (N - 1) / (N - k - 1), src/network.h:232-234; node types; an empty mailbox
    double* dof = (double*)(dyn_smem + sm.off_dof);
    for (int k = threadIdx.x; k < KMAX + 2; k += blockDim.x) dof[k] = (double)(p.n_samples - 1) / (double)(p.n_samples - k - 1);
    uint8_t* t = (uint8_t*)(dyn_smem + sm.off_types);
    for (int i = threadIdx.x; i < p.P; i += blockDim.x) t[i] = p.node_type[i];
    int* lk = (int*)(dyn_smem + sm.off_link);
    for (int i = threadIdx.x; i < (int)(sizeof(PipeLink) / 4); i += blockDim.x) lk[i] = 0;
  }
  __syncthreads();
  cluster_sync_all();  // both mailboxes are initialised before anybody writes into the peer's
  if (rank == 0) pipe_role_chain<KMAX>(p, w, ra, sm, results);
  else pipe_role_builder<KMAX>(p, w, ra, sm);
  cluster_sync_all();  // nobody leaves while the peer may still touch its shared memory
}

// Greedy placement of the per-chain arrays into the CTA's dynamic shared memory, hottest
// and smallest first; the ancestor bitsets get an odd row stride so that the column scan
// of anc_after_add/delete (one row per lane) is bank-conflict free.
static ChainSmemPlan plan_chain_smem(ChainParams& p, int scratch_n, int budget, bool with_nver = false) {
  ChainSmemPlan sm;
  int used = 0;
  auto place = [&](int64_t bytes) -> int {
    const int64_t b = (bytes + 15) / 16 * 16;
    if (used + b > budget) return -1;
    const int off = used;
    used += (int)b;
    return off;
  };
  const int64_t P = p.P, MP = p.max_par, W = p.W;
  sm.off_types = place(P);
  sm.off_ubuf = sm.off_ws = sm.off_helper = sm.off_dof = sm.off_link = -1;
  if (with_nver) {  // two-CTA form: what the one-CTA kernel keeps in static shared memory
    sm.off_ubuf = place(RNG_CAP * 8);
    sm.off_ws = place(sizeof(WindowSlots));
    sm.off_helper = place(HELPER_WORDS * 4);
    sm.off_dof = place((8 + 2) * 8);
    sm.off_link = place(sizeof(PipeLink));
  }
  sm.off_npar = place(P * 4);
  sm.off_nver = with_nver ? place(P * 4) : -1;
  sm.off_base = place(P * 8);
  sm.off_haspar = place(W * 4);
  sm.off_hplist = place(P * 4);
  sm.off_par = place(P * MP * 4);
  sm.off_scratch = place((int64_t)scratch_n * 4);
  // in shared memory, keep the row stride off a multiple of 32 words so that the column
  // scan (one row per lane, same word) spreads over the banks
  int64_t Ws = anc_stride((int)W);
  if (Ws % 32 == 0) Ws += 4;
  sm.off_anc = place(P * Ws * 4);
  p.Ws = sm.off_anc >= 0 ? (int)Ws : anc_stride((int)W);
  sm.total_bytes = used;
  return sm;
}

// the two-CTA form, when the whole state (plus the move counts) fits next to its static shared memory
template <int KMAX>
static bool plan_pipe(ChainParams& p, int scratch_n, ChainSmemPlan* out) {
  cudaFuncAttributes fa;
  if (cudaFuncGetAttributes(&fa, chain_pipe_kernel<KMAX>) != cudaSuccess) { cudaGetLastError(); return false; }
  int dev = 0, max_optin = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  const int budget = max_optin - (int)fa.sharedSizeBytes - 1024;
  ChainParams q = p;
  const ChainSmemPlan sm = plan_chain_smem(q, scratch_n, budget > 0 ? budget : 0, true);
  const bool all = sm.off_link >= 0 && sm.off_types >= 0 && sm.off_npar >= 0 && sm.off_nver >= 0 && sm.off_base >= 0 && sm.off_haspar >= 0 &&
                   sm.off_hplist >= 0 && sm.off_par >= 0 && sm.off_scratch >= 0 && sm.off_anc >= 0;
  if (!all || p.P > PIPE_MAX_NODES) return false;
  p = q;
  *out = sm;
  return true;
}

bool chains_can_pipeline(ChainParams p, int scratch_n) {
  if (p.max_par > 8) return false;
  ChainSmemPlan sm;
  return plan_pipe<8>(p, scratch_n, &sm);
}

template <int KMAX>
static const char* launch_chains_t(ChainParams p, const ChainWorkspace& w, const ChainRngArgs& ra,
                                   ChainResult* d_results, int n_chains, cudaStream_t stream) {
  if constexpr (KMAX <= 8) {
    ChainSmemPlan psm;
    if (w.pipeline && plan_pipe<KMAX>(p, w.scratch_n, &psm)) {
      if (cudaFuncSetAttribute(chain_pipe_kernel<KMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, psm.total_bytes) != cudaSuccess)
        return "cudaFuncSetAttribute(chain_pipe_kernel) failed";
      chain_pipe_kernel<KMAX><<<2 * n_chains, (HELPER_WARPS + 1) * 32, psm.total_bytes, stream>>>(p, w, ra, psm, d_results);
      return nullptr;
    }
    if (w.pipeline) return "two-CTA chains requested but the state does not fit in shared memory";
  }
  cudaFuncAttributes fa;
  if (cudaFuncGetAttributes(&fa, chain_kernel<KMAX, true, false>) != cudaSuccess) return "cudaFuncGetAttributes failed";
  int dev = 0, max_optin = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  const int budget = max_optin - (int)fa.sharedSizeBytes - 1024;
  ChainSmemPlan sm = plan_chain_smem(p, w.scratch_n, budget > 0 ? budget : 0);
  const bool all_smem = sm.off_types >= 0 && sm.off_npar >= 0 && sm.off_base >= 0 && sm.off_haspar >= 0 &&
                        sm.off_hplist >= 0 && sm.off_par >= 0 && sm.off_scratch >= 0 && sm.off_anc >= 0;
  auto kernel = w.with_state ? (all_smem ? chain_kernel<KMAX, true, true> : chain_kernel<KMAX, false, true>)
                             : (all_smem ? chain_kernel<KMAX, true, false> : chain_kernel<KMAX, false, false>);
  if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, sm.total_bytes) != cudaSuccess)
    return "cudaFuncSetAttribute(chain_kernel) failed";
  if (getenv("BN_B200_CLUSTER_EXPERIMENT") && n_chains % 2 == 0) {
    // (experiment) the one-CTA kernel launched as clusters of two independent chains
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(n_chains); cfg.blockDim = dim3((HELPER_WARPS + 1) * 32);
    cfg.dynamicSmemBytes = sm.total_bytes; cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    if (cudaLaunchKernelEx(&cfg, kernel, p, w, ra, sm, d_results) != cudaSuccess) return "cluster launch failed";
    return nullptr;
  }
  kernel<<<n_chains, (HELPER_WARPS + 1) * 32, sm.total_bytes, stream>>>(p, w, ra, sm, d_results);
  return nullptr;
}

const char* launch_chains(ChainParams p, const ChainWorkspace& w, const ChainRngArgs& ra,
                          ChainResult* d_results, int n_chains, cudaStream_t stream) {
  if (p.max_par <= 8) return launch_chains_t<8>(p, w, ra, d_results, n_chains, stream);
#if !defined(BN_DEV_BUILD_K8_ONLY)  // (developer switch of build.py: compile the MaxPar <= 8 kernels only)
  if (p.max_par <= 16) return launch_chains_t<16>(p, w, ra, d_results, n_chains, stream);
  if (p.max_par <= 64) return launch_chains_t<64>(p, w, ra, d_results, n_chains, stream);
#endif
  return "max_par > 64 is not supported";
}

// ---------------------------------------------------------------------------
// K4: score(child | parent list) for explicit lists, one thread per item.
// ---------------------------------------------------------------------------
template <int KMAX>
__global__ void __launch_bounds__(128) score_nodes_kernel(const double* __restrict__ C, int64_t ldc,
                                                          int n_samples, int max_par, int n_items,
                                                          const int* __restrict__ child,
                                                          const int* __restrict__ parents,
                                                          const int* __restrict__ n_par,
                                                          double* __restrict__ out, int* __restrict__ nonpd_count) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_items) return;
  double L[KMAX * (KMAX + 1) / 2], z[KMAX];
  int S[KMAX];
  const int k = n_par[i];
  for (int e = 0; e < k; e++) S[e] = parents[(int64_t)i * max_par + e];
  int npd = 0;
  out[i] = score_set(C, ldc, child[i], S, k, n_samples, L, z, &npd);
  if (npd) atomicAdd(nonpd_count, 1);
}

const char* launch_score_nodes(const double* C, int64_t ldc, int n_samples, int max_par, int n_items,
                               const int* d_child, const int* d_parents, const int* d_npar, double* d_out,
                               int* d_nonpd, cudaStream_t stream) {
  const int grid = (n_items + 127) / 128;
  if (max_par <= 8)
    score_nodes_kernel<8><<<grid, 128, 0, stream>>>(C, ldc, n_samples, max_par, n_items, d_child, d_parents, d_npar, d_out, d_nonpd);
  else if (max_par <= 16)
    score_nodes_kernel<16><<<grid, 128, 0, stream>>>(C, ldc, n_samples, max_par, n_items, d_child, d_parents, d_npar, d_out, d_nonpd);
  else if (max_par <= 64)
    score_nodes_kernel<64><<<grid, 128, 0, stream>>>(C, ldc, n_samples, max_par, n_items, d_child, d_parents, d_npar, d_out, d_nonpd);
  else return "max_par > 64 is not supported";
  return nullptr;
}

// ---------------------------------------------------------------------------
// K2: every single-edge add/delete proposal of a DAG in one launch.
// One warp per candidate parent set (graph g, child c): the warp gathers the
// sub-Gram of the current parents S (+ the child's cross-covariances as an
// augmented row) into shared memory, factorises it once (warp-parallel
// right-looking Cholesky), then its lanes sweep the candidate parents j:
//   add    j not in S: one more Cholesky row by forward substitution against the
//          shared factor, O(k^2) -- the same arithmetic a fresh factorisation of
//          S + [j] (push_back order, src/network.h:303) performs for its last row
//   delete j in S:     fresh factorisation of S without j (erase order, :325)
// Source/sink/max-parent masks (src/network.h:285,293) and the Potts prior
// (src/network.h:254-279,334) are applied before the store.
// Reads per add proposal: C[S_i][j] (k coalesced row segments), C[c][j], diag[j];
// writes: score + log Hastings ratio.
// ---------------------------------------------------------------------------
__global__ void graph_counts_kernel(int P, int max_par, int n_graphs, const int* __restrict__ parents,
                                    const int* __restrict__ n_par, const uint8_t* __restrict__ sim_edge,
                                    int* __restrict__ te, int* __restrict__ agree) {
  const int g = blockIdx.x;
  if (g >= n_graphs) return;
  int t = 0, a = 0;
  for (int c = threadIdx.x; c < P; c += blockDim.x) {
    const int k = n_par[(int64_t)g * P + c];
    t += k;
    for (int e = 0; e < k; e++)
      a += sim_edge[(int64_t)parents[((int64_t)g * P + c) * max_par + e] + (int64_t)c * P] ? 1 : 0;
  }
  __shared__ int st[256], sa[256];
  st[threadIdx.x] = t; sa[threadIdx.x] = a;
  __syncthreads();
  for (int o = blockDim.x / 2; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) { st[threadIdx.x] += st[threadIdx.x + o]; sa[threadIdx.x] += sa[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { te[g] = st[0]; agree[g] = sa[0]; }
}

// one more row of the factor for candidate j: w = L^-1 C[S,j]; returns the
// updated (d_j, e_j) = (C_jj - w'w, C_jc - w'z)
template <int KMAX>
__device__ __forceinline__ void border_row(const double* __restrict__ C, int64_t ldc, const int* S, int k,
                                           int j, const double* A, const double* zrow, double& dj,
                                           double& ej) {
  double w[KMAX];
  if constexpr (KMAX <= 16) {
    // fully unrolled with guards so that w[] stays in registers
#pragma unroll
    for (int i = 0; i < KMAX; i++) {
      if (i < k) {
        double acc = __ldcg(C + (int64_t)S[i] * ldc + j);
        const double* Li = A + i * (i + 1) / 2;
#pragma unroll
        for (int t = 0; t < KMAX; t++)
          if (t < i) acc -= Li[t] * w[t];
        acc *= Li[i];  // the diagonal slot holds 1 / L[i][i]
        w[i] = acc;
        dj -= acc * acc;
        ej -= acc * zrow[i];
      }
    }
  } else {
    for (int i = 0; i < k; i++) {
      double acc = __ldcg(C + (int64_t)S[i] * ldc + j);
      const double* Li = A + i * (i + 1) / 2;
      for (int t = 0; t < i; t++) acc -= Li[t] * w[t];
      acc *= Li[i];
      w[i] = acc;
      dj -= acc * acc;
      ej -= acc * zrow[i];
    }
  }
}

template <int KMAX, int SWEEP_WARPS>
__global__ void __launch_bounds__(SWEEP_WARPS * 32, KMAX <= 8 ? 8 : 2) sweep_kernel(SweepParams sp) {
  constexpr int TRI = (KMAX + 1) * (KMAX + 2) / 2;  // augmented (k+1) lower triangle
  __shared__ double sA[SWEEP_WARPS][TRI];
  __shared__ int sS[SWEEP_WARPS][KMAX];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t wslot = (int64_t)blockIdx.x * SWEEP_WARPS + warp;
  const int P = sp.P, MP = sp.max_par;
  if (wslot >= (int64_t)sp.n_graphs * P) return;
  // candidate sets are visited in order of falling parent count (sweep_order_kernel): the addition loop is
  // specialised on that count, and warps that run the same specialisation at the same time share its
  // code in the instruction cache (the kernel was starved of instructions: ncu no_instruction 4.6 per issue)
  const int64_t wg = sp.order ? (int64_t)sp.order[wslot] : wslot;
  const int g = (int)(wg / P), c = (int)(wg % P);
  const int k = sp.n_par[wg];
  const int* plist = sp.parents + wg * MP;
  double* A = sA[warp];
  int* S = sS[warp];
  const double* __restrict__ C = sp.C;
  const int64_t ldc = sp.ldc;

  for (int e = lane; e < k; e += 32) S[e] = plist[e];
  __syncwarp();
  // gather: rows 0..k-1 = C[S_i][S_t] (t <= i); row k = C[S_t][c] (t < k), C[c][c]
  const int tri = (k + 1) * (k + 2) / 2;
  for (int idx = lane; idx < tri; idx += 32) {
    int i = 0;
    while ((i + 1) * (i + 2) / 2 <= idx) i++;
    const int t = idx - i * (i + 1) / 2;
    const int ri = (i < k) ? S[i] : c;
    const int rt = (t < k) ? S[t] : c;
    A[idx] = __ldcg(C + (int64_t)ri * ldc + rt);
  }
  __syncwarp();
  const double Ccc = A[tri - 1];
  // right-looking Cholesky over the first k columns; the augmented row k ends as
  // (z_0 .. z_{k-1}, RSS)
  bool pd = true;
  for (int m = 0; m < k; m++) {
    double d = A[m * (m + 1) / 2 + m];
    if (!(d > 0.0)) { pd = false; break; }
    d = sqrt(d);
    __syncwarp();
    if (lane == 0) A[m * (m + 1) / 2 + m] = d;
    for (int i = m + 1 + lane; i <= k; i += 32) A[i * (i + 1) / 2 + m] /= d;
    __syncwarp();
    for (int i = m + 1 + lane; i <= k; i += 32) {
      const double lim = A[i * (i + 1) / 2 + m];
      for (int t = m + 1; t <= i; t++) A[i * (i + 1) / 2 + t] -= lim * A[t * (t + 1) / 2 + m];
    }
    __syncwarp();
  }
  // the candidate rows multiply by the reciprocal pivots
  for (int i = lane; i < k; i += 32) A[i * (i + 1) / 2 + i] = 1.0 / A[i * (i + 1) / 2 + i];
  __syncwarp();
  const double n = (double)sp.n_samples;
  const double neg_half_n = -(n / 2.0);
  const double syy = Ccc / (n - 1.0);
  const double rss = A[tri - 1];
  const double add_scale = 1.0 / ((n - (double)k - 2.0) * syy);  // 1 / (dof * SYY) of an addition
  const double* zrow = A + k * (k + 1) / 2;
  if (!(rss > Ccc * RSS_FLOOR)) pd = false;
  const double base = pd ? -(n / 2.0) * log((rss / (n - (double)k - 1.0)) / syy) : -INFINITY;
  if (lane == 0 && sp.out_base) sp.out_base[wg] = base;
  // an addition that leaves no residual degrees of freedom (k + 1 parents, N - k - 2 <= 0) scores -inf, as
  // the chain's (N - 1) / (N - k - 2) = inf does (add_scale would be inf or negative and its log NaN): no RSS
  // passes an infinite floor
  const double add_floor = (k + 2 < sp.n_samples) ? Ccc * RSS_FLOOR : INFINITY;

  // prior bookkeeping of this graph
  const int te = sp.te[g], ag = sp.agree[g];
  const double old_prior = prior_value(sp.phi, sp.omega, (te - ag) + (sp.n_sim_edges - ag), te);
  const uint8_t type_c = sp.node_type[c];
  const bool can_add = (type_c != 1) && (k < MP);
  const double nan = __longlong_as_double(0x7ff8000000000000ULL);
  // NewLogPrior of an addition only depends on whether the new edge is in the prior graph
  const double add_prior0 = prior_value(sp.phi, sp.omega, (te + 1 - ag) + (sp.n_sim_edges - ag), te + 1);
  const double add_prior1 = prior_value(sp.phi, sp.omega, (te + 1 - (ag + 1)) + (sp.n_sim_edges - (ag + 1)), te + 1);
  const uint8_t* sim_row = sp.sim_edge + (int64_t)c * P;
  double* out_s = sp.out_score ? sp.out_score + wg * P : nullptr;
  double* out_h = sp.out_log_hr ? sp.out_log_hr + wg * P : nullptr;

  // ---- additions: lanes sweep j ----
  // The loop is specialised on the number of current parents (a compile-time KK up to 8: the border
  // row unrolls without guards and the parent list sits in registers); larger sets take the generic
  // form.  `KK < 0` = generic.
  auto sweep_adds = [&](auto kk_tag) {
    constexpr int KK = decltype(kk_tag)::value;
    int Sr[KK > 0 ? KK : 1];
    if constexpr (KK > 0) {
#pragma unroll
      for (int e = 0; e < KK; e++) Sr[e] = S[e];
    }
    for (int j0 = 0; j0 < P; j0 += 32) {
      const int j = j0 + lane;
      if (j >= P) break;
      bool member = false;
      if constexpr (KK >= 0) {
#pragma unroll
        for (int e = 0; e < KK; e++) member |= (Sr[e] == j);
      } else {
        for (int e = 0; e < k; e++) member |= (S[e] == j);
      }
      if (member) continue;  // deletions below
      double sc = nan, hr = nan;
      if (can_add && j != c && sp.node_type[j] != 2) {
        const int a1 = sim_row[j];
        if (!pd) {
          sc = -INFINITY;
        } else {
          double dj = sp.diag[j];
          double ej = __ldcg(C + (int64_t)c * ldc + j);
          if constexpr (KK >= 0) {
            double g[KK > 0 ? KK : 1], w[KK > 0 ? KK : 1];
#pragma unroll
            for (int i = 0; i < KK; i++) g[i] = __ldcg(C + (int64_t)Sr[i] * ldc + j);
#pragma unroll
            for (int i = 0; i < KK; i++) {
              double acc = g[i];
#pragma unroll
              for (int t = 0; t < i; t++) acc -= A[i * (i + 1) / 2 + t] * w[t];
              acc *= A[i * (i + 1) / 2 + i];  // the diagonal slot holds 1 / L[i][i]
              w[i] = acc;
              dj -= acc * acc;
              ej -= acc * zrow[i];
            }
          } else {
            border_row<KMAX>(C, ldc, S, k, j, A, zrow, dj, ej);
          }
          const double rss_new = rss - ej * ej * __drcp_rn(dj);
          if (dj > 0.0 && rss_new > add_floor) sc = neg_half_n * sweep_log(rss_new * add_scale);
          else sc = -INFINITY;   // not positive definite / an exact fit the Gram route cannot resolve
        }
        hr = sub_rn(add_rn(sub_rn(sc, base), a1 ? add_prior1 : add_prior0), old_prior);
      }
      if (out_s) out_s[j] = sc;
      if (out_h) out_h[j] = hr;
    }
  };
  switch (k) {
    case 0: sweep_adds(std::integral_constant<int, 0>{}); break;
    case 1: sweep_adds(std::integral_constant<int, 1>{}); break;
    case 2: sweep_adds(std::integral_constant<int, 2>{}); break;
    case 3: sweep_adds(std::integral_constant<int, 3>{}); break;
    case 4: sweep_adds(std::integral_constant<int, 4>{}); break;
    case 5: sweep_adds(std::integral_constant<int, 5>{}); break;
    case 6: sweep_adds(std::integral_constant<int, 6>{}); break;
    case 7: sweep_adds(std::integral_constant<int, 7>{}); break;
    case 8: sweep_adds(std::integral_constant<int, 8>{}); break;
    default: sweep_adds(std::integral_constant<int, -1>{}); break;
  }
  // ---- deletions: one lane per current parent, O(k^2) on the shared factor ----
  // RSS without parent e = RSS + (y'z)^2 / (y'y), y = column e of L^-1 (forward substitution from
  // row e on): the drop-one-regressor identity instead of a fresh factorisation of S without e
  // (erase order, src/network.h:325, changes the result by rounding only)
  for (int e = lane; e < k; e += 32) {
    double y[KMAX];
    double yy, yz;
    {
      const double re = A[e * (e + 1) / 2 + e];  // 1 / L[e][e]
      y[e] = re; yy = re * re; yz = re * zrow[e];
    }
    if constexpr (KMAX <= 16) {
#pragma unroll
      for (int i = 1; i < KMAX; i++) {
        if (i > e && i < k) {
          const double* Li = A + i * (i + 1) / 2;
          double acc = 0.0;
#pragma unroll
          for (int t = 0; t < KMAX; t++)
            if (t >= e && t < i) acc -= Li[t] * y[t];
          acc *= Li[i];
          y[i] = acc; yy += acc * acc; yz += acc * zrow[i];
        }
      }
    } else {
      for (int i = e + 1; i < k; i++) {
        const double* Li = A + i * (i + 1) / 2;
        double acc = 0.0;
        for (int t = e; t < i; t++) acc -= Li[t] * y[t];
        acc *= Li[i];
        y[i] = acc; yy += acc * acc; yz += acc * zrow[i];
      }
    }
    const double rss_del = rss + yz * yz / yy;
    double sc = -(n / 2.0) * log((rss_del / (n - (double)k)) / syy);
    // no factor of a parent Gram that is not positive definite: the reduced set is scored from scratch
    if (!pd) sc = score_scratch<KMAX>(C, ldc, c, S, k, e, sp.n_samples, nullptr);
    const int j = S[e];
    const int a1 = sp.sim_edge[(int64_t)j + (int64_t)c * P] ? 1 : 0;
    const int te_n = te - 1, ag_n = ag - a1;
    const double new_prior = prior_value(sp.phi, sp.omega, (te_n - ag_n) + (sp.n_sim_edges - ag_n), te_n);
    if (out_s) out_s[j] = sc;
    if (out_h) out_h[j] = sub_rn(add_rn(sub_rn(sc, base), new_prior), old_prior);
  }
}

__global__ void diag_kernel(const double* __restrict__ C, int64_t ldc, int P, double* __restrict__ diag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < P) diag[i] = C[(int64_t)i * ldc + i];
}

void launch_diag(const double* C, int64_t ldc, int P, double* d_diag, cudaStream_t stream) {
  diag_kernel<<<(P + 127) / 128, 128, 0, stream>>>(C, ldc, P, d_diag);
}

// order[] = the (graph, child) items sorted by falling parent count: one block, counting sort (the order
// inside a count is whatever the atomics give -- every item writes its own output rows, so the result
// does not depend on it)
__global__ void __launch_bounds__(1024) sweep_order_kernel(int n_items, int max_par, const int* __restrict__ n_par,
                                                          int* __restrict__ order) {
  __shared__ int cnt[66], cur[66];
  for (int k = threadIdx.x; k < 66; k += blockDim.x) cnt[k] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < n_items; i += blockDim.x) atomicAdd(&cnt[min(n_par[i], 65)], 1);
  __syncthreads();
  if (threadIdx.x == 0) {
    int acc = 0;
    for (int k = 65; k >= 0; k--) { cur[k] = acc; acc += cnt[k]; }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n_items; i += blockDim.x) order[atomicAdd(&cur[min(n_par[i], 65)], 1)] = i;
  (void)max_par;
}

const char* launch_sweep(const SweepParams& sp, cudaStream_t stream) {
  graph_counts_kernel<<<sp.n_graphs, 256, 0, stream>>>(sp.P, sp.max_par, sp.n_graphs, sp.parents, sp.n_par,
                                                       sp.sim_edge, sp.te, sp.agree);
  if (sp.order) sweep_order_kernel<<<1, 1024, 0, stream>>>(sp.n_graphs * sp.P, sp.max_par, sp.n_par, sp.order);
  const int64_t warps = (int64_t)sp.n_graphs * sp.P;
  if (sp.max_par <= 8) sweep_kernel<8, 4><<<(unsigned)((warps + 3) / 4), 128, 0, stream>>>(sp);
  else if (sp.max_par <= 16) sweep_kernel<16, 4><<<(unsigned)((warps + 3) / 4), 128, 0, stream>>>(sp);
  else if (sp.max_par <= 64) sweep_kernel<64, 2><<<(unsigned)((warps + 1) / 2), 64, 0, stream>>>(sp);
  else return "max_par > 64 is not supported";
  return nullptr;
}

}  // namespace bn
