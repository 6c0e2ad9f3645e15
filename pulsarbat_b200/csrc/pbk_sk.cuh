// pbk_sk.cuh -- spectral kurtosis (Nita & Gary 2010) per block of M samples of every column, the
// flag of each (block, channel) cell and the zeroing of flagged cells (DESIGN.md 5.4g).
//
//   x (nsamp, nchan, npol) of complex64, int8 (re, im) pairs or float32; column (c, p) is one series
//   p = re^2 + im^2 (voltages) or x (float32 power), S1 = sum p, S2 = sum p^2 over rows
//   [b M, (b+1) M) -- int64 for int8 (exact), float64 otherwise -- and
//   SK = F (M S2 / (S1 S1) - 1),  F = (M nd + 1) / (M - 1),  NaN when S1 == 0
//   cell (b, c) is flagged when the SK of any p is outside [lo, hi] (NaN included).
//
// sk_partial_kernel: one CTA sums a run of rows of one block over CW adjacent lanes of V columns.
// Lanes walk consecutive columns of a row (CW > 1) or consecutive rows (CW = 1) with loads of V
// elements (16 bytes when the arrays allow it), each lane keeps kUnroll loads in flight, and the
// TPC row lanes of a column merge in a fixed tree.  Out of place, the same loads are written to
// the output, so the copy costs no second read.  A block is split into nsplit runs of rows when
// there are too few (block, column group) tiles to fill the GPU.
// sk_finalize_kernel: one thread per (b, c) adds the nsplit partials of its npol columns in order
// and writes SK and the flag.
// sk_zap_kernel: the grid of the estimate pass again; CTAs with a flagged cell zero it, the others
// return after reading the flags.
// No atomics: every output is bit for bit reproducible, and the int8 sums are exact.
#pragma once

#include <cuda_runtime.h>

namespace pbk_sk {

constexpr int kThreads = 256;
constexpr int kUnroll = 8;            // loads in flight per thread
constexpr int kMinRowsPerLane = 16;   // a run of rows gives each row lane at least this many rows
constexpr long long kTargetCtas = 1024;   // split blocks until the estimate grid has this many CTAs

struct PartArgs {
  const void* in;
  void* out;        // sk_partial_kernel: out-of-place copy target or nullptr; sk_zap_kernel: zapped
  void* part;       // [nblk][nsplit][W] (S1, S2)
  const unsigned char* flags;   // [nblk][nchan], read by sk_zap_kernel
  long long W;      // nchan * npol elements per row
  long long m;      // rows per block
  long long chunk;  // rows per split
  long long nchan, npol;
  int nsplit, ngroups;
};

struct FinArgs {
  const void* part;
  float* sk;               // [nblk][nchan][npol] or nullptr
  unsigned char* mask;     // [nblk][nchan] or nullptr
  unsigned char* flags;    // [nblk][nchan], always written
  long long ncells;        // nblk * nchan
  long long nchan, npol, W;
  int nsplit;
  double mf, f, lo, hi;    // M, F and the thresholds
};

// per input type: accumulator and the power of one element
template <typename T> struct Elem;
template <> struct Elem<float2> {
  using Acc = double;
  static __device__ __forceinline__ void add(float2 v, double& s1, double& s2) {
    // re^2 and im^2 of widened floats are exact in float64: the sum rounds once, with or without FMA
    const double re = v.x, im = v.y;
    const double p = re * re + im * im;
    s1 = __dadd_rn(s1, p);
    s2 = __dadd_rn(s2, __dmul_rn(p, p));
  }
};
template <> struct Elem<char2> {
  using Acc = long long;
  static __device__ __forceinline__ void add(char2 v, long long& s1, long long& s2) {
    const int p = (int)v.x * v.x + (int)v.y * v.y;   // <= 2 * 128^2
    s1 += p;
    s2 += (long long)p * p;
  }
};
template <> struct Elem<float> {
  using Acc = double;
  static __device__ __forceinline__ void add(float v, double& s1, double& s2) {
    const double p = v;
    s1 = __dadd_rn(s1, p);
    s2 = __dadd_rn(s2, __dmul_rn(p, p));
  }
};

// V consecutive elements moved as one load / store of V * sizeof(T) bytes
template <int B> struct Raw;
template <> struct Raw<2> { using U = unsigned short; };
template <> struct Raw<4> { using U = unsigned int; };
template <> struct Raw<8> { using U = uint2; };
template <> struct Raw<16> { using U = uint4; };
template <typename T, int V> union Pack {
  typename Raw<sizeof(T) * V>::U u;
  T t[V];
};

__device__ __forceinline__ double to_double(double v) { return v; }
__device__ __forceinline__ double to_double(long long v) { return __ll2double_rn(v); }

// Grid (block b, split k, column group g); lane (r, cl) owns columns c .. c + V - 1 and rows
// r0 + r, r0 + r + TPC, ... of the split.  The column order of the sums does not depend on V: V > 1
// only widens the loads of arrays aligned to V elements, so every alignment gives the same bits.
template <typename T, int V, int CW>
__global__ void __launch_bounds__(kThreads) sk_partial_kernel(PartArgs a) {
  using E = Elem<T>;
  using Acc = typename E::Acc;
  using U = typename Raw<sizeof(T) * V>::U;
  constexpr int TPC = kThreads / CW;
  __shared__ Acc sh[2][V][kThreads];
  const int tid = threadIdx.x, cl = tid % CW, r = tid / CW;
  long long bid = blockIdx.x;
  const int g = (int)(bid % a.ngroups);
  bid /= a.ngroups;
  const int k = (int)(bid % a.nsplit);
  const long long b = bid / a.nsplit;
  const long long c = ((long long)g * CW + cl) * V, ws = a.W / V;
  const long long r0 = (long long)k * a.chunk, r1 = min(a.m, r0 + a.chunk);
  Acc s1[V], s2[V];
#pragma unroll
  for (int j = 0; j < V; ++j) s1[j] = 0, s2[j] = 0;
  if (c < a.W) {
    const long long base = b * a.m * a.W + c;
    const U* src = reinterpret_cast<const U*>(reinterpret_cast<const T*>(a.in) + base);
    U* dst = a.out ? reinterpret_cast<U*>(reinterpret_cast<T*>(a.out) + base) : nullptr;
    for (long long t = r0 + r; t < r1; t += (long long)TPC * kUnroll) {
      Pack<T, V> v[kUnroll];
#pragma unroll
      for (int i = 0; i < kUnroll; ++i) {
        const long long tt = t + (long long)i * TPC;
        if (tt < r1) v[i].u = __ldg(src + tt * ws);
      }
#pragma unroll
      for (int i = 0; i < kUnroll; ++i) {
        const long long tt = t + (long long)i * TPC;
        if (tt < r1) {
#pragma unroll
          for (int j = 0; j < V; ++j) E::add(v[i].t[j], s1[j], s2[j]);
          if (dst) dst[tt * ws] = v[i].u;
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < V; ++j) sh[0][j][tid] = s1[j], sh[1][j][tid] = s2[j];
  __syncthreads();
  for (int st = TPC / 2; st >= 1; st >>= 1) {
    if (r < st) {
#pragma unroll
      for (int j = 0; j < V; ++j) {
        s1[j] += sh[0][j][tid + st * CW];
        s2[j] += sh[1][j][tid + st * CW];
        sh[0][j][tid] = s1[j], sh[1][j][tid] = s2[j];
      }
    }
    __syncthreads();
  }
  if (r == 0 && c < a.W) {
    Acc* p = reinterpret_cast<Acc*>(a.part) + ((b * a.nsplit + k) * a.W + c) * 2;
#pragma unroll
    for (int j = 0; j < V; ++j) p[2 * j] = s1[j], p[2 * j + 1] = s2[j];
  }
}

template <typename T>
__global__ void __launch_bounds__(kThreads) sk_finalize_kernel(FinArgs a) {
  using Acc = typename Elem<T>::Acc;
  const long long cell = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (cell >= a.ncells) return;
  const long long b = cell / a.nchan, c = cell - b * a.nchan;
  const Acc* part = reinterpret_cast<const Acc*>(a.part);
  bool flag = false;
  for (long long p = 0; p < a.npol; ++p) {
    const long long col = c * a.npol + p;
    Acc s1 = 0, s2 = 0;
    for (int k = 0; k < a.nsplit; ++k) {
      const Acc* q = part + ((b * a.nsplit + k) * a.W + col) * 2;
      s1 += q[0];
      s2 += q[1];
    }
    const double d1 = to_double(s1), d2 = to_double(s2);
    // SK = F (M S2 / (S1 S1) - 1) in exactly this order, without contraction
    const double sk = d1 == 0.0 ? __longlong_as_double(0x7ff8000000000000LL)
                                : __dmul_rn(a.f, __dadd_rn(__ddiv_rn(__dmul_rn(a.mf, d2),
                                                                     __dmul_rn(d1, d1)), -1.0));
    if (a.sk) a.sk[cell * a.npol + p] = (float)sk;
    flag |= !(sk >= a.lo && sk <= a.hi);
  }
  a.flags[cell] = flag ? 1 : 0;
  if (a.mask) a.mask[cell] = flag ? 1 : 0;
}

// Same grid as sk_partial_kernel: a CTA none of whose columns belongs to a flagged cell of its block
// returns after reading the flags, so unflagged cells cost no write.
template <typename T, int V, int CW>
__global__ void __launch_bounds__(kThreads) sk_zap_kernel(PartArgs a) {
  using U = typename Raw<sizeof(T) * V>::U;
  constexpr int TPC = kThreads / CW;
  const int tid = threadIdx.x, cl = tid % CW, r = tid / CW;
  long long bid = blockIdx.x;
  const int g = (int)(bid % a.ngroups);
  bid /= a.ngroups;
  const int k = (int)(bid % a.nsplit);
  const long long b = bid / a.nsplit;
  const long long c = ((long long)g * CW + cl) * V, ws = a.W / V;
  const long long r0 = (long long)k * a.chunk, r1 = min(a.m, r0 + a.chunk);
  bool fj[V];
  bool any = false, all = true;
#pragma unroll
  for (int j = 0; j < V; ++j) {
    fj[j] = c + j < a.W && a.flags[b * a.nchan + (c + j) / a.npol];
    any |= fj[j];
    all &= fj[j];
  }
  if (!__syncthreads_or(any) || !any) return;
  T* base = reinterpret_cast<T*>(a.out) + b * a.m * a.W + c;
  Pack<T, V> z;
  z.u = U{};
  for (long long t = r0 + r; t < r1; t += TPC) {
    if (all) {
      reinterpret_cast<U*>(base)[t * ws] = z.u;
    } else {
#pragma unroll
      for (int j = 0; j < V; ++j)
        if (fj[j]) base[t * a.W + j] = z.t[j];
    }
  }
}

// column lanes of a CTA: the widest power of two <= min(lanes, 32)
inline int columns_per_cta(long long lanes) {
  int cw = 32;
  while (cw > lanes) cw /= 2;
  return cw;
}

// elements per load of an aligned row: 2 complex64 or 4 float32 (16 bytes), 4 int8 pairs (8 bytes:
// 8 pairs would double the int64 accumulators and leave one CTA per SM)
template <typename T> constexpr int vector_width() { return sizeof(T) == 2 ? 4 : 16 / sizeof(T); }
inline int vector_width(int esize) { return esize == 2 ? 4 : 16 / esize; }

template <typename T, int V>
inline cudaError_t launch_v(bool zap, int CW, const PartArgs& a, unsigned grid, cudaStream_t st) {
#define PBK_SK_CASE(cw)                                                             \
  case cw:                                                                          \
    if (zap) sk_zap_kernel<T, V, cw><<<grid, kThreads, 0, st>>>(a);                 \
    else sk_partial_kernel<T, V, cw><<<grid, kThreads, 0, st>>>(a);                 \
    break;
  switch (CW) {
    PBK_SK_CASE(32)
    PBK_SK_CASE(16)
    PBK_SK_CASE(8)
    PBK_SK_CASE(4)
    PBK_SK_CASE(2)
    default:
      if (zap) sk_zap_kernel<T, V, 1><<<grid, kThreads, 0, st>>>(a);
      else sk_partial_kernel<T, V, 1><<<grid, kThreads, 0, st>>>(a);
  }
#undef PBK_SK_CASE
  return cudaGetLastError();
}

template <typename T>
inline cudaError_t launch_pass(bool zap, bool vec, int CW, const PartArgs& a, unsigned grid,
                               cudaStream_t st) {
  constexpr int VW = vector_width<T>();
  return vec ? launch_v<T, VW>(zap, CW, a, grid, st) : launch_v<T, 1>(zap, CW, a, grid, st);
}

// esize: 8 (complex64), 2 (int8 pairs) or 4 (float32); zap: the partial grid of the zap pass
inline cudaError_t launch_pass(int esize, bool zap, bool vec, int CW, const PartArgs& a,
                               unsigned grid, cudaStream_t st) {
  if (esize == 8) return launch_pass<float2>(zap, vec, CW, a, grid, st);
  if (esize == 2) return launch_pass<char2>(zap, vec, CW, a, grid, st);
  return launch_pass<float>(zap, vec, CW, a, grid, st);
}

inline cudaError_t launch_finalize(int esize, const FinArgs& a, unsigned grid, cudaStream_t st) {
  if (esize == 8) sk_finalize_kernel<float2><<<grid, kThreads, 0, st>>>(a);
  else if (esize == 2) sk_finalize_kernel<char2><<<grid, kThreads, 0, st>>>(a);
  else sk_finalize_kernel<float><<<grid, kThreads, 0, st>>>(a);
  return cudaGetLastError();
}

}  // namespace pbk_sk
