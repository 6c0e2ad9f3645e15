// pbk_fdmt.cuh -- fast dispersion measure transform (FDMT) of a (nsamp, C, P) float32 filterbank
// (DESIGN.md 5.4h; index tables from pbk_fdmt_tables.cu).
//
// State.  Level l holds, for every row of every node, one row of `stride` floats: the window's
// times with P interleaved, time-major, so a shift of h samples is a shift of h * P floats.  A
// chunk's window starts at input time ws; every value before it reads as +0, which is exactly the
// definition's x[t < 0] = 0 when ws == 0, and is never part of a kept output otherwise (each root
// row d at time t reads only x[t - d .. t], and the window starts D samples before the earliest
// kept time).  Every output is a fixed tree of float32 adds: no atomics, bit-for-bit repeatable.
//
// Kernels.
// - fused_kernel: one CTA per (level-k node, time tile).  It stages the input rows its subtree
//   reads, builds the leaves and k merges in shared memory over the tile plus a halo of the node's
//   largest row, and writes level k's rows for the tile.  At k = 0 it builds the leaves alone in
//   registers and writes them straight out; that form measured fastest on B200 (DESIGN.md 5.4h)
//   and is the default.
// - pass_kernel: one merged level, state to state.  A CTA is one row and a run of times; rows vary
//   fastest in the grid, so adjacent rows, which mostly share h, read their L row from L2.  The
//   L row and the output are 16-byte vectors; the U row, shifted by h * P floats, is read as
//   coalesced scalars.
// - last_kernel: the root's rows d_min..D, written straight into the caller's (ndm, rows, P).
#pragma once

#include <cuda_runtime.h>

#include "pbk_fdmt_tables.h"

namespace pbk_fdmt {

constexpr int kThreads = 256;
constexpr int kPassFloats = 4 * kThreads;          // floats per pass CTA and grid-y step
constexpr int kFusedThreads = 256;                 // fused kernel: blockDim (32, 8)

struct FusedArgs {
  const float* x;        // input (nsamp, C, P)
  float* out;            // level-k state
  long long xrow;        // C * P
  long long ws;          // input time of window time 0
  long long stride;      // floats per state row
  int wlen;              // window times
  int P, k, T, nnodes;   // floats per cell, fused merges, tile times, level-k nodes
  const int* row0;       // levels 0..k, concatenated [nnodes_l + 1] arrays
  const int* row0_off;   // [k + 1] offset of level l's array in row0
  const int* nnodes_l;   // [k + 1]
  const int4* ent;       // levels 1..k, concatenated (l, u, h, s)
  const int* ent_off;    // [k + 1] offset of level l's entries in ent (index 0 unused)
  int bufB_floats;       // offset of the second shared buffer
};

__global__ void __launch_bounds__(kFusedThreads) fdmt_fused_kernel(FusedArgs a) {
  extern __shared__ float sm[];
  const int n = (int)(blockIdx.x % (unsigned)a.nnodes);
  const int tile = (int)(blockIdx.x / (unsigned)a.nnodes);
  const int t0 = tile * a.T;
  const int P = a.P;
  const int* r0k = a.row0 + a.row0_off[a.k];
  if (a.k == 0) {
    // leaves only: each thread runs down the rows of one (time, p) of channel n in registers and
    // writes them straight to the state; x is read from L1 / L2, no shared memory
    const int nr = r0k[n + 1] - r0k[n];
    const int ntp = min(a.T, a.wlen - t0) * P;
    const float* xc = a.x + a.ws * a.xrow + (long long)n * P;
    float* dst = a.out + (long long)r0k[n] * a.stride + (long long)t0 * P;
    for (int e = threadIdx.y * blockDim.x + threadIdx.x; e < ntp; e += kFusedThreads) {
      const int tau = e / P, p = e - tau * P;
      const int wt = t0 + tau;
      float v = xc[(long long)wt * a.xrow + p];
      dst[e] = v;
      for (int r = 1; r < nr; ++r) {
        v = v + (wt - r >= 0 ? xc[(long long)(wt - r) * a.xrow + p] : 0.f);
        dst[(long long)r * a.stride + e] = v;
      }
    }
    return;
  }
  const int H = r0k[n + 1] - r0k[n] - 1;              // halo: the node's largest row
  const int WT = a.T + H, WTP = WT * P;
  // leaves of the subtree
  const int ca = n << a.k, cb = min((n + 1) << a.k, a.nnodes_l[0]);
  const int nch = cb - ca;
  const int* r00 = a.row0;
  int nl = 1;
  for (int c = ca; c < cb; ++c) nl = max(nl, r00[c + 1] - r00[c]);
  float* bufA = sm;
  float* bufB = sm + a.bufB_floats;
  // stage x at window times [t0 - H - (nl - 1), t0 + T) for channels [ca, cb): bufB
  const int XT = WT + nl - 1, xw = nch * P;
  const long long tx0 = (long long)t0 - H - (nl - 1);
  const int tid = threadIdx.y * blockDim.x + threadIdx.x;
  for (int i = tid; i < XT * xw; i += kFusedThreads) {
    const int tt = i / xw, q = i - tt * xw;
    const long long wt = tx0 + tt;
    bufB[i] = wt >= 0 && wt < a.wlen ? a.x[(a.ws + wt) * a.xrow + (long long)ca * P + q] : 0.f;
  }
  __syncthreads();
  // leaves: A_c[0, t] = x[t], A_c[i, t] = A_c[i - 1, t] + x[t - i]; local time tau is staged row
  // tau + nl - 1.  Loops run over flattened (row, time) so that no thread idles at a row's end.
  const int ra0 = r00[ca];
  for (int i = tid; i < nch * WTP; i += kFusedThreads) {
    const int cc = i / WTP, e = i - cc * WTP;
    const int tau = e / P, p = e - tau * P;
    const int c = ca + cc;
    const int nr = r00[c + 1] - r00[c];
    float* dst = bufA + (r00[c] - ra0) * WTP + e;
    const float* src = bufB + (tau + nl - 1) * xw + cc * P + p;
    float v = src[0];
    dst[0] = v;
    for (int r = 1; r < nr; ++r) {
      v = v + src[-r * xw];
      dst[r * WTP] = v;
    }
  }
  __syncthreads();
  // merges 1..k, ping-ponging between the two buffers
  float* src = bufA;
  float* dstb = bufB;
  for (int l = 1; l <= a.k; ++l) {
    const int* rp = a.row0 + a.row0_off[l - 1];
    const int* rl = a.row0 + a.row0_off[l];
    const int span = a.k - l;
    const int pa = rp[n << (span + 1)];
    const int la = rl[n << span], lb = rl[min((n + 1) << span, a.nnodes_l[l])];
    const int4* ent = a.ent + a.ent_off[l];
    for (int i = tid; i < (lb - la) * WTP; i += kFusedThreads) {
      const int r = i / WTP, e = i - r * WTP;
      const int4 en = ent[la + r];
      float v = src[(en.x - pa) * WTP + e];
      if (en.y >= 0) {
        const int eu = e - en.z * P;
        v = v + (eu >= 0 ? src[(en.y - pa) * WTP + eu] : 0.f);
      }
      dstb[r * WTP + e] = v;
    }
    __syncthreads();
    float* tmp = src;
    src = dstb;
    dstb = tmp;
  }
  // level k rows of the node, tile times only
  const int ka = r0k[n];
  const int nt = min(a.T, a.wlen - t0);
  const int nrow = H + 1, ntp = nt * P;
  for (int i = tid; i < nrow * ntp; i += kFusedThreads) {
    const int r = i / ntp, e = i - r * ntp;
    a.out[(long long)(ka + r) * a.stride + (long long)t0 * P + e] = src[r * WTP + H * P + e];
  }
}

struct PassArgs {
  const float* src;
  float* dst;
  const int4* ent;       // rows of this level
  long long stride;
  int n;                 // floats per row in use (wlen * P)
  int P;
};

__global__ void __launch_bounds__(kThreads) fdmt_pass_kernel(PassArgs a) {
  const int4 en = a.ent[blockIdx.x];
  const float* L = a.src + (long long)en.x * a.stride;
  const float* U = a.src + (long long)max(en.y, 0) * a.stride;
  float* D = a.dst + (long long)blockIdx.x * a.stride;
  const int sh = en.z * a.P;
  for (int e = blockIdx.y * kPassFloats + threadIdx.x * 4; e < a.n; e += gridDim.y * kPassFloats) {
    float4 v = *reinterpret_cast<const float4*>(L + e);     // stride and bases are 16-byte aligned
    if (en.y >= 0) {
      const int eu = e - sh;
      v.x = v.x + (eu >= 0 ? U[eu] : 0.f);
      v.y = v.y + (eu + 1 >= 0 ? U[eu + 1] : 0.f);
      v.z = v.z + (eu + 2 >= 0 ? U[eu + 2] : 0.f);
      v.w = v.w + (eu + 3 >= 0 ? U[eu + 3] : 0.f);
    }
    *reinterpret_cast<float4*>(D + e) = v;   // floats past n stay inside the padded row
  }
}

struct LastArgs {
  const float* src;
  float* out;            // (ndm, rows, P)
  const int4* ent;       // [ndm] (l, u, h, s_d)
  long long stride;
  long long rows;        // output rows of the whole plane
  long long base;        // window time of output row ja with s = 0: t_lo + ja - ws
  long long ja;          // first output row of the chunk
  int n;                 // floats of the chunk per trial (jn * P)
  int P;
};

__global__ void __launch_bounds__(kThreads) fdmt_last_kernel(LastArgs a) {
  const int4 en = a.ent[blockIdx.x];
  const long long e0 = (a.base + en.w) * a.P;
  const float* L = a.src + (long long)en.x * a.stride + e0;
  const float* U = a.src + (long long)max(en.y, 0) * a.stride + e0;
  float* o = a.out + ((long long)blockIdx.x * a.rows + a.ja) * a.P;
  const long long sh = (long long)en.z * a.P;
  for (int e = blockIdx.y * kThreads + threadIdx.x; e < a.n; e += gridDim.y * kThreads) {
    float v = L[e];
    if (en.y >= 0) v = v + (e0 + e - sh >= 0 ? U[e - sh] : 0.f);
    o[e] = v;
  }
}

}  // namespace pbk_fdmt
