// TEST-ONLY reference of the posterior ancestor tabulation (bn_run_args.anc_freq), independent of the
// chain core: it replays an accepted-move log from the start graph, recomputes the whole ancestor
// closure FROM SCRATCH after every move (Kahn order, each row = itself OR the rows of its parents), and
// integrates every row over the iterations it held its value.  Built by tests/test_ancestor_tab.py into
// tests/emu/_build/.
#include <cstdint>
#include <cstring>
#include <vector>

namespace {

using Row = std::vector<uint64_t>;

// closure[d] = {d} u ancestors of d; false if the graph is cyclic
bool closure(int P, const std::vector<std::vector<int>>& par, std::vector<Row>& out) {
  const int nw = (P + 63) / 64;
  std::vector<int> indeg(P), order;
  std::vector<std::vector<int>> kids(P);
  order.reserve(P);
  for (int c = 0; c < P; c++) {
    indeg[c] = (int)par[c].size();
    for (int q : par[c]) kids[q].push_back(c);
    if (!indeg[c]) order.push_back(c);
  }
  for (size_t i = 0; i < order.size(); i++)
    for (int k : kids[order[i]])
      if (--indeg[k] == 0) order.push_back(k);
  if ((int)order.size() != P) return false;
  out.assign(P, Row(nw, 0));
  for (int d : order) {
    Row& r = out[d];
    r[d >> 6] |= 1ull << (d & 63);
    for (int q : par[d])
      for (int w = 0; w < nw; w++) r[w] |= out[q][w];
  }
  return true;
}

}  // namespace

// start_par / start_npar: [P][max_par] (-1 padded) and [P]; moves: n_moves rows (iter, movetype 1 = addition /
// 2 = deletion, child, parent); the run covers iterations [it0, end).  out: [P][P] int64 (zeroed by the
// caller), out[a + d*P] += the iterations i >= drop in [it0, end) after which a is an ancestor of d.
// stats (may be NULL): [0] the moves after which the closure differs from the one before, [1] the
// (ancestor, descendant) bits those moves flipped.
// Returns 0; 1 if the start graph is cyclic; 2 + k if move k made the graph cyclic or was not applicable.
extern "C" int anc_replay(int P, int max_par, const int* start_par, const int* start_npar, const int* moves,
                          int n_moves, long long it0, long long end, int drop, long long* out, long long* stats) {
  std::vector<std::vector<int>> par(P);
  for (int c = 0; c < P; c++)
    for (int e = 0; e < start_npar[c]; e++) par[c].push_back(start_par[(size_t)c * max_par + e]);
  std::vector<Row> cur, next;
  if (!closure(P, par, cur)) return 1;
  std::vector<long long> since(P, it0);  // each row has held its value since this iteration
  if (stats) stats[0] = stats[1] = 0;
  auto counted = [drop](long long lo, long long hi) {
    lo = lo > drop ? lo : drop;
    hi = hi > drop ? hi : drop;
    return hi - lo;
  };
  auto flush = [&](int d, long long t) {
    const long long n = counted(since[d], t);
    if (n > 0)
      for (int a = 0; a < P; a++)
        if ((cur[d][a >> 6] >> (a & 63)) & 1ull) out[(size_t)d * P + a] += n;
    since[d] = t;
  };
  for (int k = 0; k < n_moves; k++) {
    const int* mv = moves + 4 * (size_t)k;
    const long long t = mv[0];
    const int c = mv[2], j = mv[3];
    std::vector<int>& pc = par[c];
    if (mv[1] == 1) {
      pc.push_back(j);
    } else {
      size_t e = 0;
      while (e < pc.size() && pc[e] != j) e++;
      if (e == pc.size()) return 2 + k;
      pc.erase(pc.begin() + e);
    }
    if (!closure(P, par, next)) return 2 + k;
    // the graph after the move holds from iteration t on: rows that differ close their interval at t
    bool changed = false;
    for (int d = 0; d < P; d++) {
      if (next[d] == cur[d]) continue;
      if (stats)
        for (size_t w = 0; w < next[d].size(); w++) stats[1] += __builtin_popcountll(next[d][w] ^ cur[d][w]);
      flush(d, t);
      cur[d] = next[d];
      changed = true;
    }
    if (stats && changed) stats[0]++;
  }
  for (int d = 0; d < P; d++) flush(d, end);
  return 0;
}
