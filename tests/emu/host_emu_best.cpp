// TEST-ONLY host instantiation of the chain core (one-lane "warp") with the best-graph tracking
// (bn_run_args.best) on, and a supplied start as in host_emu_state.cpp: the graph, the scalars of a
// resumed chain and the score block go in, the same come out.  It lets the CPU suite check the best graph
// against a replay of the move log and the trace, and that the segments of a resumed run combine to the
// uninterrupted run's best.  Built by tests/test_best_graph.py into tests/emu/_build/; never part of
// libbn_b200.so.
#include <cstdlib>
#include <cstring>
#include <vector>

#include "chain_core.cuh"

using namespace bn;

// bn_chain_state of include/bn_b200.h, plus the R Mersenne-Twister state (.Random.seed[2:626] layout)
struct EmuChainState {
  long long iter;
  int valid, total_edges_member, additions, deletions;
  int wh_state[3];
  long long uniforms;
  int mt[625];
};

// bn_best_graph of include/bn_b200.h
struct EmuBestGraph {
  double log_post, log_lik, log_prior;
  long long iter;
  int total_edges, found;
};

extern "C" long long emu_best_score_state_len(int P, int max_par) {
  return (long long)P + (max_par > 8 ? (long long)P * fac_stride(fac_mp(max_par)) : 0);
}

// start_par == null: the start graph of initial_network.  st_in == null: a fresh chain (WH from
// seeds, R-MT from st_mt_fresh at position 624).  score_in == null: scores computed from the graph.
// best == null: no tracking (best_par / best_npar are not touched).
extern "C" int emu_run_chain_best(
    int P, int max_par, int n_samples, const double* C, const unsigned char* node_type,
    const unsigned char* sim_edge, int n_sim_edges, double phi, double omega,
    int initial_network, int drop, int n_iter, int output_every,
    const int* prior_par, const int* prior_npar,
    int rng_kind, const int* seeds, const unsigned int* mt_fresh, const double* replay,
    long replay_len, int capacity,
    int* t_iter, int* t_changed, int* t_movetype, double* t_gll, int* t_add, int* t_del,
    int* t_fn, int* t_fp, int moves_capacity, int* moves, int* edge_freq, int* npar_freq,
    int* final_par, int* final_npar, long* out_counters /*[12]*/,
    const int* start_par, const int* start_npar, const EmuChainState* st_in, EmuChainState* st_out,
    const double* score_in, double* score_out,
    int* best_par /* [P][max_par] */, int* best_npar /* [P] */, EmuBestGraph* best) {
  ChainStart start;
  if (st_in) {
    start.iter = st_in->iter; start.valid = st_in->valid; start.te_m = st_in->total_edges_member;
    start.acc_add = st_in->additions; start.acc_del = st_in->deletions;
  }
  ChainParams p;
  p.P = P; p.max_par = max_par; p.W = (P + 31) / 32; p.Ws = (p.W + 3) / 4 * 4; p.n_samples = n_samples;
  std::vector<double> diag(P);
  for (int i = 0; i < P; i++) diag[i] = C[(size_t)i * P + i];
  p.C = C; p.ldc = P; p.diag = diag.data(); p.node_type = node_type; p.sim_edge = sim_edge;
  p.n_sim_edges = n_sim_edges; p.phi = phi; p.omega = omega;
  p.initial_network = initial_network; p.drop = drop;
  p.n_iter = (int)((st_in ? start.iter : 0) + n_iter);  // as chain_kernel: n_iter more iterations
  p.output_every = output_every; p.trace_capacity = capacity; p.moves_capacity = moves_capacity;
  p.prior_par = prior_par; p.prior_npar = prior_npar; p.prior_stride = max_par;
  set_row_geom(p);
  std::vector<double> ratio(max_par + 10);
  for (int k = 0; k < (int)ratio.size(); k++) ratio[k] = (double)(n_samples - 1) / (double)(n_samples - k - 1);
  p.sc.half_n = (double)n_samples / 2.0;
  p.sc.ratio = ratio.data();

  std::vector<int> par((size_t)P * max_par), npar(P), born((size_t)P * max_par);
  std::vector<int> scratch((size_t)scratch_words(P, 1, 1)), hp_list(P);
  std::vector<double> base(P), base_in(P);
  std::vector<uint32_t> anc_store((size_t)P * p.Ws + 4), haspar(p.W);
  uint32_t* anc = (uint32_t*)(((uintptr_t)anc_store.data() + 15) & ~(uintptr_t)15);
  ChainMem m;
  m.par = par.data(); m.npar = npar.data(); m.born = born.data(); m.base = base.data();
  m.anc = anc; m.haspar = haspar.data();
  m.scratch = scratch.data(); m.hp_list = hp_list.data(); m.helper = nullptr;
  m.t_iter = t_iter; m.t_changed = t_changed; m.t_movetype = t_movetype; m.t_gll = t_gll;
  m.t_add = t_add; m.t_del = t_del; m.t_fn = t_fn; m.t_fp = t_fp;
  m.moves = moves; m.edge_freq = edge_freq;
  std::vector<int> npar_since(P);
  m.npar_freq = npar_freq; m.npar_since = npar_since.data();
  std::vector<double> dscore((size_t)P * max_par, NAN);
  m.dscore = dscore.data();
  const size_t fac_n = (size_t)P * fac_stride(fac_mp(max_par));
  std::vector<double> fac(fac_n + 2), rowbuf((size_t)REPLAY_POS * row_stride(fac_mp(max_par)) + 2);
  m.fac = (double*)(((uintptr_t)fac.data() + 15) & ~(uintptr_t)15);
  m.rowbuf = (double*)(((uintptr_t)rowbuf.data() + 15) & ~(uintptr_t)15);
  m.start_par = start_par; m.start_npar = start_npar;
  m.start = st_in ? &start : nullptr;
  BestTrack track;
  std::vector<uint32_t> dirty(p.W);
  std::vector<int> dirty_list(P);
  if (best) {
    track.n_sim = n_sim_edges; track.phi = phi; track.omega = omega;
    track.par = best_par; track.npar = best_npar; track.dirty = dirty.data(); track.list = dirty_list.data();
    m.best = &track;
  }
  if (score_in) {
    memcpy(base_in.data(), score_in, sizeof(double) * P);
    if (max_par > 8) memcpy(m.fac, score_in + P, sizeof(double) * fac_n);
    m.base_in = base_in.data();
  }

  // the stream: where the stopped run left it, or fresh
  int wh[3] = {seeds[0], seeds[1], seeds[2]};
  std::vector<uint32_t> mt(624), mt0(624);
  int mti = 624;
  if (st_in && rng_kind == RNG_WH) memcpy(wh, st_in->wh_state, sizeof(wh));
  if (st_in && rng_kind == RNG_RMT) {
    mti = st_in->mt[0];
    for (int i = 0; i < 624; i++) mt[i] = (uint32_t)st_in->mt[1 + i];
  } else if (mt_fresh) {
    memcpy(mt.data(), mt_fresh, 624 * 4);
  }
  mt0 = mt;
  std::vector<double> ubuf(RNG_CAP);
  RngStream rng;
  if (rng_kind == RNG_WH) rng_init_wh(rng, wh[0], wh[1], wh[2], ubuf.data());
  else if (rng_kind == RNG_RMT) rng_init_rmt(rng, mt.data(), mti, ubuf.data());
  else rng_init_replay(rng, replay, replay_len, ubuf.data());

  ChainScalars s;
  WindowSlots ws;
  if (max_par <= 8) run_chain<8>(p, m, s, rng, ws);
  else if (max_par <= 16) run_chain<16>(p, m, s, rng, ws);
  else if (max_par <= 64) run_chain<64>(p, m, s, rng, ws);
  else return 7;

  memcpy(final_par, par.data(), sizeof(int) * par.size());
  memcpy(final_npar, npar.data(), sizeof(int) * P);
  out_counters[0] = s.read_pos; out_counters[1] = s.valid_iters;
  for (int t = 0; t < 3; t++) { out_counters[2 + t] = s.proposed[t]; out_counters[5 + t] = s.reject[t]; }
  out_counters[8] = s.n_rows; out_counters[9] = s.n_moves; out_counters[10] = s.n_nonpd;
  out_counters[11] = s.windows;
  if (st_out) {
    memset(st_out, 0, sizeof(*st_out));
    st_out->iter = s.iter; st_out->valid = s.valid; st_out->total_edges_member = s.te_m;
    st_out->additions = s.acc_add; st_out->deletions = s.acc_del;
    st_out->uniforms = (st_in ? st_in->uniforms : 0) + s.read_pos;
    if (rng_kind == RNG_WH) wh_advance(wh, s.read_pos, st_out->wh_state);
    if (rng_kind == RNG_RMT) {
      int pos = st_in ? st_in->mt[0] : 624;
      rmt_advance(mt0.data(), pos, s.read_pos);
      st_out->mt[0] = pos;
      for (int i = 0; i < 624; i++) st_out->mt[1 + i] = (int)mt0[i];
    }
  }
  if (score_out) {
    memcpy(score_out, base.data(), sizeof(double) * P);
    if (max_par > 8) memcpy(score_out + P, m.fac, sizeof(double) * fac_n);
  }
  if (best) {
    best->log_post = track.log_post; best->log_lik = track.log_lik; best->log_prior = track.log_prior;
    best->iter = track.iter; best->total_edges = track.total_edges; best->found = track.found;
  }
  return s.status;
}
