// pbk_fdmt_tables.h -- host-side index tables of the fast dispersion measure transform (FDMT,
// DESIGN.md 5.4h).  Built in float64 in exactly the order of the definition, in its own
// translation unit compiled without floating-point contraction (pbk_fdmt_tables.cu), so that
// f_lo + c * df and d * K stay two roundings on every host and tests/fdmt_oracle.py reproduces them.
#pragma once

#include <vector>

namespace pbk_fdmt {

// One row of a merged level: A[row, t] = A'[l, t] + A'[u, t - h], or A'[l, t] when u < 0 (a
// carried node).  l and u are rows of the level below, numbered across its nodes.
struct Entry {
  int l, u, h, s;        // s: the output shift s_d (root rows of the last level only, else 0)
};

struct Tables {
  int C = 0, L = 0;                       // channels, merges to the root (ceil(log2 C))
  std::vector<int> nnodes;                // [L + 1] nodes per level
  std::vector<std::vector<int>> row0;     // [L + 1][nnodes + 1] first row of each node
  std::vector<std::vector<Entry>> ent;    // [L + 1]: ent[l] = rows of level l (l >= 1)
  std::vector<Entry> last;                // root rows d_min..D with their s_d; for C == 1
                                          // (no merge) carries of the leaf rows
  long long t_lo = 0, rows = 0;           // output geometry
  int s_min = 0, s_max = 0;               // over the output rows
};

// Returns 0, or 1 when a row count or shift does not fit 32-bit indices.
int build_tables(long long nsamp, int C, double f_lo, double f_hi, double ref, long long D,
                 long long d_min, Tables* t);

}  // namespace pbk_fdmt
