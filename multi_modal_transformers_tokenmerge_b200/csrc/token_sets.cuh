// Token sets of the matching kernels (tome_token_sets_t): matching and merging run inside each set, the per-set plan
// arrays are concatenated set by set.  SetTable is the form the kernels take it in -- the table plus the prefix offsets of
// every per-set array -- built and validated once on the host; a NULL tome_token_sets_t* is one set spanning the sequence,
// whose offsets are all zero, so the one-set kernels index exactly as before the table existed.
#pragma once

#include "../../include/tome_b200.h"
#include "host_util.h"

namespace tome {

struct SetTable {
  int n;                                    // sets
  int start[TOME_MAX_TOKEN_SETS], len[TOME_MAX_TOKEN_SETS], r[TOME_MAX_TOKEN_SETS];
  // prefix sums over the sets (entry n = total): even tokens (plane A rows, node_max / edge_idx), odd tokens (plane B rows),
  // merged tokens (dst_idx / dst_src), dst_off entries (odd + 1), output rows (n - r), score-dump entries (even * odd)
  int a_off[TOME_MAX_TOKEN_SETS + 1], b_off[TOME_MAX_TOKEN_SETS + 1], r_off[TOME_MAX_TOKEN_SETS + 1];
  int off_off[TOME_MAX_TOKEN_SETS + 1], out_off[TOME_MAX_TOKEN_SETS + 1];
  long long sc_off[TOME_MAX_TOKEN_SETS + 1];
  // K1 a-row tiles per set (prefix sums for the tile size of the launch: set_tiles)
  int tile_off[TOME_MAX_TOKEN_SETS + 1];
  int max_ta, max_tb;                       // largest set's even / odd token counts (K2 shared memory)
};

// Validates `sets` against a sequence of `tokens` tokens and fills `t`.  r_total >= 0: the set r's must add up to it
// (plan / merge shapes); r_total < 0: not checked (metric descriptors carry no r).  Returns TOME_OK or TOME_ERR_INVALID
// with the message set, before any CUDA call.
inline int make_set_table(const tome_token_sets_t* sets, int tokens, int r_total, int class_token, int distill_token,
                          SetTable* t, const char* who) {
  memset(t, 0, sizeof(*t));
  if (!sets) {
    t->n = 1;
    t->start[0] = 0;
    t->len[0] = tokens;
    t->r[0] = r_total > 0 ? r_total : 0;
  } else {
    TOME_CHECK(!class_token && !distill_token, TOME_ERR_INVALID,
               "%s: token sets cannot be combined with a class or distill token", who);
    TOME_CHECK(sets->n_sets >= 1 && sets->n_sets <= TOME_MAX_TOKEN_SETS, TOME_ERR_INVALID, "%s: n_sets (%d) must be in [1, %d]",
               who, sets->n_sets, TOME_MAX_TOKEN_SETS);
    t->n = sets->n_sets;
    long long next = 0, rsum = 0;
    for (int s = 0; s < t->n; ++s) {
      TOME_CHECK(sets->set_start[s] == next, TOME_ERR_INVALID,
                 "%s: token set %d starts at %d, expected %lld (sets must be consecutive, without gaps or overlaps)", who, s,
                 sets->set_start[s], next);
      TOME_CHECK(sets->set_n[s] >= 1, TOME_ERR_INVALID, "%s: token set %d is empty", who, s);
      TOME_CHECK(sets->set_r[s] >= 0 && sets->set_r[s] <= sets->set_n[s] / 2, TOME_ERR_INVALID,
                 "%s: token set %d: r = %d out of range [0, %d]", who, s, sets->set_r[s], sets->set_n[s] / 2);
      t->start[s] = sets->set_start[s];
      t->len[s] = sets->set_n[s];
      t->r[s] = sets->set_r[s];
      next += sets->set_n[s];
      rsum += sets->set_r[s];
    }
    TOME_CHECK(next == tokens, TOME_ERR_INVALID, "%s: the token sets cover %lld tokens, the sequence has %d", who, next, tokens);
    TOME_CHECK(r_total < 0 || rsum == r_total, TOME_ERR_INVALID, "%s: r (%d) must equal the sum of the sets' r (%lld)", who,
               r_total, rsum);
  }
  for (int s = 0; s < t->n; ++s) {
    const int ta = (t->len[s] + 1) / 2, tb = t->len[s] / 2;
    t->a_off[s + 1] = t->a_off[s] + ta;
    t->b_off[s + 1] = t->b_off[s] + tb;
    t->r_off[s + 1] = t->r_off[s] + t->r[s];
    t->off_off[s + 1] = t->off_off[s] + tb + 1;
    t->out_off[s + 1] = t->out_off[s] + t->len[s] - t->r[s];
    t->sc_off[s + 1] = t->sc_off[s] + (long long)ta * tb;
    if (ta > t->max_ta) t->max_ta = ta;
    if (tb > t->max_tb) t->max_tb = tb;
  }
  return TOME_OK;
}

// tile_off for K1 launches over (a-row tile of a set, set): returns the number of tiles
inline int set_tiles(SetTable* t, int tile_rows) {
  for (int s = 0; s < t->n; ++s) t->tile_off[s + 1] = t->tile_off[s] + ceil_div((t->len[s] + 1) / 2, tile_rows);
  return t->tile_off[t->n];
}

#ifdef __CUDACC__
// the set `v` falls in, given the prefix array off[0..n] (off[0] = 0, v < off[n]): a linear scan of at most 16 entries
__device__ __forceinline__ int set_of(const int* off, int n, int v) {
  int s = 0;
  while (s + 1 < n && v >= off[s + 1]) ++s;
  return s;
}

// plane row of token t of a batch row: its set's even (A) or odd (B) row, relative to the start of the batch row's plane
__device__ __forceinline__ int set_plane_row(const SetTable& tab, int t, bool& odd) {
  const int s = set_of(tab.start, tab.n, t);   // set_of reads start[1 .. n-1] only: no total entry needed
  const int l = t - tab.start[s];
  odd = l & 1;
  return (odd ? tab.b_off[s] : tab.a_off[s]) + (l >> 1);
}
#endif

}  // namespace tome
