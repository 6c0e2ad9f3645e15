// pbk_search.cuh -- single-pulse search of a stack of time series (a DM x time plane): float64
// statistics per series, boxcar S/N at up to 32 widths and the maximum over windows of starts.
//
//   x (nser, rows, ncols) float32; series (s, c) is x[s, :, c].
//   snr(s, c, t, w) = (sum_{i<w} x[s, t+i, c] - w * mean) / (std * sqrt(w)),  t + w <= rows
//   out[s, j, c] = the best (snr, t, w) over the starts t of window j, ties to the smallest t, then
//   the smallest w.  No atomics anywhere: every output has one owner and every sum a fixed order,
//   so executions are bit for bit reproducible (DESIGN.md 5.4f).
//
// Statistics: stats_partial_kernel merges float64 (n, mean, M2) partials per (series, column,
// chunk of rows) -- two-pass over batches of 8 values held in registers, then Chan's update --
// and stats_combine_kernel merges the chunks of one series in a fixed order (one warp each).
//
// Boxcar: one CTA owns the windows of one run of starts of one series and CW adjacent columns.
// It walks the run in tiles of T = 1024 / CW samples per column: lanes load consecutive rows (or,
// for CW > 1, consecutive columns of a row), the tile's inclusive prefix of (x - K) is formed in
// float64 by warp shuffles and one warp per column over the 32 lane groups, and written into a
// ring of R (power of two) prefix values per column.  The starts evaluated in a tile lag the loads
// by LR >= w_max samples, so every P[t + w] is already in the ring; each input float is read once
// except for the LR samples that start a run.  K is the mean rounded to a multiple of
// 2^(ilogb(std) - 12): integer-valued data then gives exact integer prefix differences, so equal
// sums give equal S/N, while the drift of the prefix stays below std * 2^-12 per sample.
//   snr = fma(P[t+w] - P[t], inv[w], -cw[w]),  inv[w] = 1 / (std sqrt(w)),  cw[w] = w (mean - K) inv[w]
// Starts compare in float64; the windowed maximum is a segmented max-scan (warp shuffles, then
// one warp per column over the groups, then the carry of the window that straddles tiles).
#pragma once

#include <cuda_runtime.h>
#include <math_constants.h>

namespace pbk_search {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kV = 4;                 // samples (and starts) per thread per tile
constexpr int kGroups = kV * kWarps;  // lane groups per column per tile
constexpr int kMaxWidths = 32;
constexpr int kMaxWidth = 4096;       // widths above this return PBK_ERR_UNSUPPORTED
constexpr int kStatBatch = 8;         // values merged per Chan step
constexpr int kStatPer = 64;          // values per thread per statistics chunk

struct StatArgs {
  const float* x;
  double* part;          // [nser * ncols * nchunks * 3] (n, mean, M2)
  double* stats;         // [nser * ncols * 2] (mean, std)
  long long rows, ncols, nseries;   // nseries = nser * ncols
  int ngroups, nchunks;
};

struct BoxArgs {
  const float* x;
  const double* stats;
  float* snr;
  int* start;
  int* width;
  long long rows, ncols;
  int window;            // min(window, rows)
  int nwin;
  int ngroups, runs, wpr;   // column groups, runs per series, windows per run
  int nw, wmax, lr, mask, rs;   // widths; ring lag, R - 1, per-column stride (R + 1)
  int widths[kMaxWidths];
};

// Chan et al.: merge (nb, mb, m2b) into (n, m, m2)
__device__ __forceinline__ void chan_merge(double& n, double& m, double& m2, double nb, double mb,
                                           double m2b) {
  if (nb == 0.0) return;
  const double nn = n + nb, d = mb - m, f = nb / nn;
  m = m + d * f;
  m2 = m2 + m2b + d * d * n * f;
  n = nn;
}

// one chunk of TPC * kStatPer rows of CW columns; lanes walk consecutive rows (CW = 1) or the
// consecutive columns of a row
template <int CW>
__global__ void __launch_bounds__(kThreads) stats_partial_kernel(StatArgs a) {
  constexpr int TPC = kThreads / CW;
  __shared__ double sh[3][kThreads];
  const int tid = threadIdx.x, cl = tid % CW, r = tid / CW;
  long long bid = blockIdx.x;
  const int k = (int)(bid % a.nchunks);
  bid /= a.nchunks;
  const int g = (int)(bid % a.ngroups);
  const long long s = bid / a.ngroups;
  const long long c = (long long)g * CW + cl;
  const long long t0 = (long long)k * TPC * kStatPer + r;
  double n = 0.0, m = 0.0, m2 = 0.0;
  if (c < a.ncols) {
    const float* src = a.x + s * a.rows * a.ncols + c;
    for (int b = 0; b < kStatPer; b += kStatBatch) {
      double v[kStatBatch];
      int nb = 0;
#pragma unroll
      for (int i = 0; i < kStatBatch; ++i) {
        const long long t = t0 + (long long)(b + i) * TPC;
        v[i] = t < a.rows ? (double)__ldg(src + t * a.ncols) : 0.0;
        nb += t < a.rows;
      }
      if (nb == 0) break;
      double sum = 0.0;
#pragma unroll
      for (int i = 0; i < kStatBatch; ++i) sum += v[i];
      const double mb = sum / nb;
      double m2b = 0.0;
#pragma unroll
      for (int i = 0; i < kStatBatch; ++i)
        if (i < nb) m2b += (v[i] - mb) * (v[i] - mb);
      chan_merge(n, m, m2, (double)nb, mb, m2b);
    }
  }
  sh[0][tid] = n, sh[1][tid] = m, sh[2][tid] = m2;
  __syncthreads();
  for (int st = TPC / 2; st >= 1; st >>= 1) {
    if (r < st) {
      const int o = tid + st * CW;
      chan_merge(n, m, m2, sh[0][o], sh[1][o], sh[2][o]);
      sh[0][tid] = n, sh[1][tid] = m, sh[2][tid] = m2;
    }
    __syncthreads();
  }
  if (r == 0 && c < a.ncols) {
    double* p = a.part + ((s * a.ncols + c) * a.nchunks + k) * 3;
    p[0] = n, p[1] = m, p[2] = m2;
  }
}

// one warp per series: lane l merges chunks l, l + 32, ... in order, then a fixed shuffle tree
__global__ void __launch_bounds__(kThreads) stats_combine_kernel(StatArgs a) {
  const int lane = threadIdx.x & 31;
  const long long sc = (long long)blockIdx.x * kWarps + (threadIdx.x >> 5);
  if (sc >= a.nseries) return;
  const double* p = a.part + sc * a.nchunks * 3;
  double n = 0.0, m = 0.0, m2 = 0.0;
  for (int k = lane; k < a.nchunks; k += 32) chan_merge(n, m, m2, p[3 * k], p[3 * k + 1], p[3 * k + 2]);
  for (int o = 16; o >= 1; o >>= 1) {
    const double nb = __shfl_down_sync(0xffffffffu, n, o);
    const double mb = __shfl_down_sync(0xffffffffu, m, o);
    const double m2b = __shfl_down_sync(0xffffffffu, m2, o);
    if (lane + o < 32) chan_merge(n, m, m2, nb, mb, m2b);
  }
  if (lane == 0) {
    a.stats[2 * sc] = m;
    a.stats[2 * sc + 1] = sqrt(m2 / n);
  }
}

// dynamic shared memory of one boxcar CTA, in bytes
__host__ __device__ inline size_t boxcar_smem(int CW, int rs) {
  return sizeof(double) * ((size_t)CW * rs + (size_t)CW * kGroups * 3 + (size_t)CW * kMaxWidths * 2 +
                           5 * (size_t)CW) +
         sizeof(int) * kMaxWidths;
}

template <int CW>
__global__ void __launch_bounds__(kThreads, 2) boxcar_kernel(BoxArgs a) {
  constexpr int TPC = kThreads / CW, G = 32 / CW, T = kV * TPC;
  extern __shared__ double sm[];
  double* ring = sm;                                        // [CW][rs] prefix values
  double* gsum = ring + (size_t)CW * a.rs;                  // [CW][kGroups] group sums / prefixes
  double* gms = gsum + CW * kGroups;                        // [CW][kGroups] group maxima
  long long* gmk = (long long*)(gms + CW * kGroups);        //   and their (t << 5 | width index)
  double* sinv = (double*)(gmk + CW * kGroups);             // [CW][kMaxWidths]
  double* scw = sinv + CW * kMaxWidths;
  double* csn = scw + CW * kMaxWidths;                      // [2][CW] carry of the open window,
  long long* ckey = (long long*)(csn + 2 * CW);             //   by tile parity
  double* kshift = (double*)(ckey + 2 * CW);                // [CW] K
  int* swid = (int*)(kshift + CW);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int cl = tid % CW, r = tid / CW, lr = lane / CW;    // lr: rank among the column's lanes
  long long bid = blockIdx.x;
  const int g = (int)(bid % a.ngroups);
  bid /= a.ngroups;
  const int run = (int)(bid % a.runs);
  const long long s = bid / a.runs;
  const long long c = (long long)g * CW + cl;
  const bool cok = c < a.ncols;
  const long long tb = (long long)run * a.wpr * a.window;
  const long long run_len = min(a.rows, tb + (long long)a.wpr * a.window) - tb;
  const long long lim = min(a.rows, tb + run_len + a.wmax - 1);

  if (tid < CW) {
    const long long cc = (long long)g * CW + tid;
    double mean = 0.0, sd = 0.0;
    if (cc < a.ncols) {
      mean = a.stats[(s * a.ncols + cc) * 2];
      sd = a.stats[(s * a.ncols + cc) * 2 + 1];
    }
    const bool ok = sd > 0.0;                 // false for zero, negative and NaN
    double K = 0.0;
    if (ok) {
      const double q = ldexp(1.0, ilogb(sd) - 12);
      K = rint(mean / q) * q;
      if (!isfinite(K)) K = 0.0;
    }
    kshift[tid] = K;
    for (int k = 0; k < a.nw; ++k) {
      const double w = (double)a.widths[k];
      const double inv = ok ? 1.0 / (sd * sqrt(w)) : 0.0;
      sinv[tid * kMaxWidths + k] = inv;
      scw[tid * kMaxWidths + k] = ok ? w * (mean - K) * inv : 0.0;
    }
    ring[(size_t)tid * a.rs] = 0.0;           // P[0]
    csn[tid] = csn[CW + tid] = -CUDART_INF;
    ckey[tid] = ckey[CW + tid] = -1;
  }
  if (tid < a.nw) swid[tid] = a.widths[tid];
  __syncthreads();
  const double K = kshift[cl];
  const float* src = a.x + (s * a.rows + tb) * a.ncols + (cok ? c : 0);
  double* rc = ring + (size_t)cl * a.rs;

  float xv[kV];
  auto load = [&](long long b) {
#pragma unroll
    for (int v = 0; v < kV; ++v) {
      const long long t = b + v * TPC + r;
      xv[v] = (cok && tb + t < lim) ? __ldg(src + t * a.ncols) : 0.f;
    }
  };
  load(0);
  const long long nit = (run_len + a.lr + T - 1) / T;
  for (long long it = 0; it < nit; ++it) {
    const long long b = it * T;
    // ---- prefix of the tile: P[b + j + 1] for j = v * TPC + r = (v * kWarps + warp) * G + lr
    double pv[kV];
#pragma unroll
    for (int v = 0; v < kV; ++v) {
      const long long t = tb + b + v * TPC + r;
      pv[v] = (cok && t < lim) ? (double)xv[v] - K : 0.0;
#pragma unroll
      for (int d = 1; d < G; d <<= 1) {
        const double y = __shfl_up_sync(0xffffffffu, pv[v], d * CW);
        if (lr >= d) pv[v] += y;
      }
      if (lr == G - 1) gsum[cl * kGroups + v * kWarps + warp] = pv[v];
    }
    __syncthreads();
    for (int cc = warp; cc < CW; cc += kWarps) {
      double inc = gsum[cc * kGroups + lane];
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const double y = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += y;
      }
      const double ex = __shfl_up_sync(0xffffffffu, inc, 1);
      gsum[cc * kGroups + lane] = ring[(size_t)cc * a.rs + (b & a.mask)] + (lane ? ex : 0.0);
    }
    __syncthreads();
#pragma unroll
    for (int v = 0; v < kV; ++v)
      rc[(b + v * TPC + r + 1) & a.mask] = gsum[cl * kGroups + v * kWarps + warp] + pv[v];
    if (it + 1 < nit) load(b + T);
    __syncthreads();

    // ---- starts ts + j, j = v * TPC + r, lag LR behind the loads
    const long long ts = b - a.lr;
    if (ts < 0 || ts >= run_len) continue;   // uniform over the CTA
    const long long abs0 = tb + ts;
    const int par = (int)(it & 1) * CW;
    const int offs0 = (int)(abs0 % a.window), win0 = (int)(abs0 / a.window);
    double bs[kV], p0[kV];
    long long bk[kV];
    int room[kV], offs[kV];
#pragma unroll
    for (int v = 0; v < kV; ++v) {
      const int j = v * TPC + r;
      const long long p = ts + j;
      bs[v] = -CUDART_INF;
      bk[v] = -1;
      p0[v] = rc[p & a.mask];
      room[v] = p < run_len ? (int)(a.rows - (tb + p)) : 0;
      offs[v] = (int)((unsigned)(offs0 + j) % (unsigned)a.window);
    }
    for (int k = 0; k < a.nw; ++k) {
      const int w = swid[k];
      const double iv = sinv[cl * kMaxWidths + k], cv = scw[cl * kMaxWidths + k];
#pragma unroll
      for (int v = 0; v < kV; ++v) {
        if (w <= room[v]) {
          const double dsum = rc[(ts + v * TPC + r + w) & a.mask] - p0[v];
          const double sn = fma(dsum, iv, -cv);
          if (sn > bs[v]) bs[v] = sn, bk[v] = k;
        }
      }
    }
    // segmented max over the starts of each window: earlier entries win ties
#pragma unroll
    for (int v = 0; v < kV; ++v) {
      if (bk[v] >= 0) bk[v] |= (abs0 + v * TPC + r) << 5;
#pragma unroll
      for (int d = 1; d < G; d <<= 1) {
        const double ys = __shfl_up_sync(0xffffffffu, bs[v], d * CW);
        const long long yk = __shfl_up_sync(0xffffffffu, bk[v], d * CW);
        if (lr >= d && offs[v] >= d && !(bs[v] > ys)) bs[v] = ys, bk[v] = yk;
      }
      if (lr == G - 1) {
        gms[cl * kGroups + v * kWarps + warp] = bs[v];
        gmk[cl * kGroups + v * kWarps + warp] = bk[v];
      }
    }
    __syncthreads();
    for (int cc = warp; cc < CW; cc += kWarps) {
      double ms = gms[cc * kGroups + lane];
      long long mk = gmk[cc * kGroups + lane];
      // offset in its window of this group's last start
      const int ol = (int)((unsigned)(offs0 + lane * G + G - 1) % (unsigned)a.window);
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const double ys = __shfl_up_sync(0xffffffffu, ms, d);
        const long long yk = __shfl_up_sync(0xffffffffu, mk, d);
        if (lane >= d && ol >= d * G && !(ms > ys)) ms = ys, mk = yk;
      }
      // the window opened in an earlier tile
      if (ol >= (lane + 1) * G && !(ms > csn[par + cc])) ms = csn[par + cc], mk = ckey[par + cc];
      gms[cc * kGroups + lane] = ms;
      gmk[cc * kGroups + lane] = mk;
      // the last start of the tile carries its window into the next tile
      if (lane == 31) csn[(CW - par) + cc] = ms, ckey[(CW - par) + cc] = mk;
    }
    __syncthreads();
#pragma unroll
    for (int v = 0; v < kV; ++v) {
      const int j = v * TPC + r, grp = v * kWarps + warp;
      double ps = -CUDART_INF;
      long long pk = -1;
      bool has = false;
      if (grp > 0 && offs[v] >= lr + 1) {
        ps = gms[cl * kGroups + grp - 1], pk = gmk[cl * kGroups + grp - 1], has = true;
      } else if (offs[v] >= j + 1) {
        ps = csn[par + cl], pk = ckey[par + cl], has = true;
      }
      if (has && !(bs[v] > ps)) bs[v] = ps, bk[v] = pk;
      const long long p = ts + j, t = tb + p;
      if (p < run_len && cok && (offs[v] == a.window - 1 || t == a.rows - 1)) {
        const int jw = win0 + (int)((unsigned)(offs0 + j) / (unsigned)a.window);
        const long long o = (s * a.nwin + jw) * a.ncols + c;
        a.snr[o] = (float)bs[v];
        a.start[o] = bk[v] >= 0 ? (int)(bk[v] >> 5) : -1;
        a.width[o] = bk[v] >= 0 ? swid[bk[v] & 31] : -1;
      }
    }
  }
}

inline const void* boxcar_kernel_of(int CW) {
  switch (CW) {
    case 32: return (const void*)boxcar_kernel<32>;
    case 16: return (const void*)boxcar_kernel<16>;
    case 8: return (const void*)boxcar_kernel<8>;
    case 4: return (const void*)boxcar_kernel<4>;
    case 2: return (const void*)boxcar_kernel<2>;
    default: return (const void*)boxcar_kernel<1>;
  }
}

inline cudaError_t launch_boxcar(int CW, const BoxArgs& a, unsigned grid, size_t smem, cudaStream_t st) {
  switch (CW) {
    case 32: boxcar_kernel<32><<<grid, kThreads, smem, st>>>(a); break;
    case 16: boxcar_kernel<16><<<grid, kThreads, smem, st>>>(a); break;
    case 8: boxcar_kernel<8><<<grid, kThreads, smem, st>>>(a); break;
    case 4: boxcar_kernel<4><<<grid, kThreads, smem, st>>>(a); break;
    case 2: boxcar_kernel<2><<<grid, kThreads, smem, st>>>(a); break;
    default: boxcar_kernel<1><<<grid, kThreads, smem, st>>>(a); break;
  }
  return cudaGetLastError();
}

inline cudaError_t launch_stats(int CW, const StatArgs& a, cudaStream_t st) {
  const unsigned grid = (unsigned)(a.nseries / a.ncols * a.ngroups * a.nchunks);
  switch (CW) {
    case 32: stats_partial_kernel<32><<<grid, kThreads, 0, st>>>(a); break;
    case 16: stats_partial_kernel<16><<<grid, kThreads, 0, st>>>(a); break;
    case 8: stats_partial_kernel<8><<<grid, kThreads, 0, st>>>(a); break;
    case 4: stats_partial_kernel<4><<<grid, kThreads, 0, st>>>(a); break;
    case 2: stats_partial_kernel<2><<<grid, kThreads, 0, st>>>(a); break;
    default: stats_partial_kernel<1><<<grid, kThreads, 0, st>>>(a); break;
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  stats_combine_kernel<<<(unsigned)((a.nseries + kWarps - 1) / kWarps), kThreads, 0, st>>>(a);
  return cudaGetLastError();
}

}  // namespace pbk_search
