// TEST-ONLY reference of the posterior Markov blanket tabulation (bn_run_args.mb_freq), independent of the
// chain core and of its witness counts: it replays an accepted-move log from the start graph, recomputes every
// node's blanket FROM SCRATCH after every move (children from the parent lists, then parents u children u the
// children's other parents), and integrates every row over the iterations it held its value.  Built by
// tests/test_markov_blanket.py into tests/emu/_build/.
#include <cstdint>
#include <cstring>
#include <vector>

namespace {

using Row = std::vector<uint64_t>;

void set(Row& r, int b) { r[b >> 6] |= 1ull << (b & 63); }

// out[i] = {i} u parents(i) u children(i) u the other parents of i's children
void blankets(int P, const std::vector<std::vector<int>>& par, std::vector<Row>& out) {
  const int nw = (P + 63) / 64;
  std::vector<std::vector<int>> kids(P);
  for (int c = 0; c < P; c++)
    for (int q : par[c]) kids[q].push_back(c);
  out.assign(P, Row(nw, 0));
  for (int i = 0; i < P; i++) {
    Row& r = out[i];
    set(r, i);
    for (int q : par[i]) set(r, q);
    for (int ch : kids[i]) {
      set(r, ch);
      for (int q : par[ch]) set(r, q);  // (i itself is among them: already set)
    }
  }
}

}  // namespace

// start_par / start_npar: [P][max_par] (-1 padded) and [P]; moves: n_moves rows (iter, movetype 1 = addition /
// 2 = deletion, child, parent); the run covers iterations [it0, end).  out: [P][P] int64 (zeroed by the
// caller), out[j + i*P] += the iterations t >= drop in [it0, end) after which j is in the blanket of i (the
// diagonal: all of them).  stats (may be NULL): [0] the moves after which some blanket differs from the one
// before, [1] the ordered (i, j) entries those moves flipped.
// Returns 0; 2 + k if move k was not applicable (a duplicate parent, or a deletion of an absent one).
extern "C" int mb_replay(int P, int max_par, const int* start_par, const int* start_npar, const int* moves,
                         int n_moves, long long it0, long long end, int drop, long long* out, long long* stats) {
  std::vector<std::vector<int>> par(P);
  for (int c = 0; c < P; c++)
    for (int e = 0; e < start_npar[c]; e++) par[c].push_back(start_par[(size_t)c * max_par + e]);
  std::vector<Row> cur, next;
  blankets(P, par, cur);
  std::vector<long long> since(P, it0);  // each row has held its value since this iteration
  if (stats) stats[0] = stats[1] = 0;
  auto counted = [drop](long long lo, long long hi) {
    lo = lo > drop ? lo : drop;
    hi = hi > drop ? hi : drop;
    return hi - lo;
  };
  auto flush = [&](int i, long long t) {
    const long long n = counted(since[i], t);
    if (n > 0)
      for (int j = 0; j < P; j++)
        if ((cur[i][j >> 6] >> (j & 63)) & 1ull) out[(size_t)i * P + j] += n;
    since[i] = t;
  };
  for (int k = 0; k < n_moves; k++) {
    const int* mv = moves + 4 * (size_t)k;
    const long long t = mv[0];
    const int c = mv[2], j = mv[3];
    std::vector<int>& pc = par[c];
    size_t e = 0;
    while (e < pc.size() && pc[e] != j) e++;
    if (mv[1] == 1) {
      if (e != pc.size() || j == c || (int)pc.size() >= max_par) return 2 + k;
      pc.push_back(j);
    } else {
      if (e == pc.size()) return 2 + k;
      pc.erase(pc.begin() + e);
    }
    blankets(P, par, next);
    // the graph after the move holds from iteration t on: rows that differ close their interval at t
    bool changed = false;
    for (int i = 0; i < P; i++) {
      if (next[i] == cur[i]) continue;
      if (stats)
        for (size_t w = 0; w < next[i].size(); w++) stats[1] += __builtin_popcountll(next[i][w] ^ cur[i][w]);
      flush(i, t);
      cur[i] = next[i];
      changed = true;
    }
    if (stats && changed) stats[0]++;
  }
  for (int i = 0; i < P; i++) flush(i, end);
  return 0;
}
