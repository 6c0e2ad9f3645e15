// pbk_fdmt_tables.cu -- the FDMT tree, its row counts and merge shifts, and the output shifts,
// in float64 in the order written in DESIGN.md 5.4h.  Compiled with -ffp-contract=off (Makefile):
// an FMA in f_lo + c * df or d * K would move a rounded shift by one on some hosts.
#include "pbk_fdmt_tables.h"

#include <algorithm>
#include <climits>
#include <cmath>

namespace pbk_fdmt {

static double K(double a, double b) { return 1.0 / (a * a) - 1.0 / (b * b); }

// rint in the default rounding mode: round half to even, as numpy.rint
static long long rnd(double v) { return (long long)std::nearbyint(v); }

int build_tables(long long nsamp, int C, double f_lo, double f_hi, double ref, long long D,
                 long long d_min, Tables* t) {
  const double df = (f_hi - f_lo) / C;
  std::vector<double> fe(C + 1);
  for (int c = 0; c <= C; ++c) fe[c] = f_lo + (double)c * df;
  // tree: lo[l][n] = first channel of node n at level l; level l + 1 merges (2m, 2m + 1)
  std::vector<std::vector<int>> lo(1), hi(1);
  for (int c = 0; c < C; ++c) lo[0].push_back(c), hi[0].push_back(c + 1);
  while (lo.back().size() > 1) {
    const std::vector<int>& pl = lo.back();
    const std::vector<int>& ph = hi.back();
    std::vector<int> nl, nh;
    for (size_t i = 0; i < pl.size(); i += 2) {
      nl.push_back(pl[i]);
      nh.push_back(i + 1 < pl.size() ? ph[i + 1] : ph[i]);
    }
    lo.push_back(nl);
    hi.push_back(nh);
  }
  const int L = (int)lo.size() - 1;
  t->C = C;
  t->L = L;
  t->nnodes.assign(L + 1, 0);
  for (int l = 0; l <= L; ++l) t->nnodes[l] = (int)lo[l].size();
  // row counts, top down; h of every merged row
  std::vector<std::vector<long long>> nrows(L + 1);
  for (int l = 0; l <= L; ++l) nrows[l].assign(lo[l].size(), 0);
  nrows[L][0] = D + 1;
  std::vector<std::vector<std::vector<long long>>> hs(L + 1);
  for (int l = L - 1; l >= 0; --l) {
    hs[l + 1].resize(lo[l + 1].size());
    for (size_t m = 0; m < lo[l + 1].size(); ++m) {
      const long long nS = nrows[l + 1][m];
      if (2 * m + 1 >= lo[l].size()) {           // carried
        nrows[l][2 * m] = nS;
        continue;
      }
      const int c0 = lo[l][2 * m], cm = lo[l][2 * m + 1], c1 = hi[l][2 * m + 1];
      const double kl = K(fe[c0], fe[cm]), ks = K(fe[c0], fe[c1]);
      std::vector<long long>& h = hs[l + 1][m];
      h.resize(nS);
      long long hmax = 0, umax = 0;
      for (long long d = 0; d < nS; ++d) {
        h[d] = rnd(((double)d * kl) / ks);
        hmax = std::max(hmax, h[d]);
        umax = std::max(umax, d - h[d]);
      }
      nrows[l][2 * m] = hmax + 1;
      nrows[l][2 * m + 1] = umax + 1;
    }
  }
  t->row0.assign(L + 1, {});
  for (int l = 0; l <= L; ++l) {
    std::vector<int>& r = t->row0[l];
    r.assign(lo[l].size() + 1, 0);
    long long acc = 0;
    for (size_t n = 0; n < lo[l].size(); ++n) {
      r[n] = (int)acc;
      acc += nrows[l][n];
      if (acc > INT_MAX) return 1;
    }
    r[lo[l].size()] = (int)acc;
  }
  t->ent.assign(L + 1, {});
  for (int l = 1; l <= L; ++l) {
    std::vector<Entry>& e = t->ent[l];
    e.reserve(t->row0[l].back());
    const std::vector<int>& rb = t->row0[l - 1];
    for (size_t m = 0; m < lo[l].size(); ++m)
      for (long long d = 0; d < nrows[l][m]; ++d) {
        if (2 * m + 1 >= lo[l - 1].size()) {
          e.push_back({rb[2 * m] + (int)d, -1, 0, 0});
          continue;
        }
        const long long h = hs[l][m][d];
        e.push_back({rb[2 * m] + (int)h, rb[2 * m + 1] + (int)(d - h), (int)h, 0});
      }
  }
  // output rows d_min..D of the root
  const double kr = K(f_lo, ref), kb = K(f_lo, f_hi);
  long long tl = LLONG_MIN, smax = LLONG_MIN, smin = LLONG_MAX;
  t->last.clear();
  for (long long d = d_min; d <= D; ++d) {
    const long long s = rnd(((double)d * kr) / kb);
    if (s > INT_MAX || s < INT_MIN) return 1;
    tl = std::max(tl, d - s);
    smax = std::max(smax, s);
    smin = std::min(smin, s);
    Entry e = L > 0 ? t->ent[L][d] : Entry{(int)d, -1, 0, 0};
    e.s = (int)s;
    t->last.push_back(e);
  }
  t->t_lo = tl;
  t->rows = std::max(0LL, nsamp - smax - tl);
  t->s_min = (int)smin;
  t->s_max = (int)smax;
  return 0;
}

}  // namespace pbk_fdmt
