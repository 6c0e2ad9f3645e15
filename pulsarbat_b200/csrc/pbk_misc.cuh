// pbk_misc.cuh -- bandwidth-bound companions of the FFT passes: detection, time integration and
// phase-binned folding.
//   detect      core.py:766-774 (re^2+im^2 per pol) and core.py:948/960 (Stokes I = AA+BB)
//   downsample  builder-defined time sum (SURVEY 8a row R)
//   fold        builder-defined (SURVEY 8a row F) on top of the phase polynomial returned by
//               pulsar/predictor.py:149-160 (phasepol); numpy polyval order, FP64, no FMA.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace pbk {

constexpr int kFoldMaxCoef = 16;

// out[j, e] = sum_{m<M} in[(j*M+m), e]      float32 in/out, float32 accumulation in time order
__global__ void __launch_bounds__(256) downsample_kernel(const float* __restrict__ in,
                                                         float* __restrict__ out, long long rows,
                                                         long long E, long long M) {
  const long long total = rows * E;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long j = i / E, e = i - j * E;
    const float* src = in + (j * M) * E + e;
    float acc = 0.f;
#pragma unroll 8
    for (long long m = 0; m < M; ++m) acc += __ldg(src + m * E);
    out[i] = acc;
  }
}

// float4-wide variant when E % 4 == 0 and pointers are 16-byte aligned
__global__ void __launch_bounds__(256) downsample_kernel_v4(const float4* __restrict__ in,
                                                            float4* __restrict__ out,
                                                            long long rows, long long E4,
                                                            long long M) {
  const long long total = rows * E4;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long j = i / E4, e = i - j * E4;
    const float4* src = in + (j * M) * E4 + e;
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 8
    for (long long m = 0; m < M; ++m) {
      const float4 v = __ldg(src + m * E4);
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
    out[i] = acc;
  }
}

static inline cudaError_t launch_downsample(const float* in, float* out, long long rows,
                                            long long E, long long M, cudaStream_t st) {
  if (rows <= 0) return cudaSuccess;
  const bool v4 = (E % 4 == 0) && ((((uintptr_t)in | (uintptr_t)out) & 15) == 0);
  const long long total = v4 ? rows * (E / 4) : rows * E;
  long long blocks = (total + 255) / 256;
  if (blocks > 148ll * 32) blocks = 148ll * 32;
  if (v4)
    downsample_kernel_v4<<<(unsigned)blocks, 256, 0, st>>>(reinterpret_cast<const float4*>(in),
                                                           reinterpret_cast<float4*>(out), rows,
                                                           E / 4, M);
  else
    downsample_kernel<<<(unsigned)blocks, 256, 0, st>>>(in, out, rows, E, M);
  return cudaGetLastError();
}

// one (A, B) pol pair of complex64 as (Are, Aim, Bre, Bim): a 128-bit load when the array is
// 16-byte aligned (V4), two 64-bit loads when it is only aligned to its complex64 elements
template <bool V4>
__device__ __forceinline__ float4 ld_pair(const float2* p) {
  if (V4) return __ldg(reinterpret_cast<const float4*>(p));
  const float2 a = __ldg(p), b = __ldg(p + 1);
  return make_float4(a.x, a.y, b.x, b.y);
}
// four floats: one 128-bit store, or four 32-bit stores (a float32 Stokes array may be aligned
// to 4 bytes only)
template <bool V4>
__device__ __forceinline__ void st_pair(float* p, float4 v) {
  if (V4) {
    *reinterpret_cast<float4*>(p) = v;
  } else {
    p[0] = v.x;
    p[1] = v.y;
    p[2] = v.z;
    p[3] = v.w;
  }
}

// pol-pair kernels below take the 128-bit path only for 16-byte aligned arrays (the C ABI promises
// complex64 alignment, 8 bytes, and nothing more)
static inline bool aligned16(const void* a, const void* b) {
  return (((uintptr_t)a | (uintptr_t)b) & 15) == 0;
}

// power detection with optional time sum.  in (rows*M, CP) complex64.
//   stokes == 0: out (rows, CP)   = sum_m re^2+im^2
//   stokes == 1: out (rows, CP/2) = sum_m |A|^2+|B|^2   (pol pairs are adjacent)
template <bool V4>
__global__ void __launch_bounds__(256) detect_kernel(const float2* __restrict__ in,
                                                     float* __restrict__ out, long long rows,
                                                     long long CP, int stokes, long long M) {
  const long long E = stokes ? CP / 2 : CP;
  const long long total = rows * E;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long j = i / E, e = i - j * E;
    float acc = 0.f;
    if (stokes) {
      for (long long m = 0; m < M; ++m) {
        const float4 v = ld_pair<V4>(in + (j * M + m) * CP + 2 * e);
        // (XX) + (YY), each as re*re + im*im like the reference
        acc += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
      }
    } else {
      const float2* src = in + (j * M) * CP + e;
      for (long long m = 0; m < M; ++m) {
        const float2 v = __ldg(src + m * CP);
        acc += v.x * v.x + v.y * v.y;
      }
    }
    out[i] = acc;
  }
}

static inline cudaError_t launch_detect(const float2* in, float* out, long long rows, long long CP,
                                        bool stokes, long long M, cudaStream_t st) {
  if (rows <= 0) return cudaSuccess;
  const long long total = rows * (stokes ? CP / 2 : CP);
  long long blocks = (total + 255) / 256;
  if (blocks > 148ll * 32) blocks = 148ll * 32;
  // the 128-bit Stokes loads read pol pairs at even complex offsets: a 16-byte aligned base suffices
  if ((((uintptr_t)in) & 15) == 0)
    detect_kernel<true><<<(unsigned)blocks, 256, 0, st>>>(in, out, rows, CP, stokes ? 1 : 0, M);
  else
    detect_kernel<false><<<(unsigned)blocks, 256, 0, st>>>(in, out, rows, CP, stokes ? 1 : 0, M);
  return cudaGetLastError();
}

// detection with time AND frequency summing ("scrunching"): one warp per output element.
//   out[j, c', (p)] = sum_{m<M} sum_{f<F} |in[j*M+m, c'*F+f, p]|^2   (Stokes: also summed over p)
// Used after channelize, where 2^16 fine channels per coarse channel are binned down (cfg 4).
__global__ void __launch_bounds__(256) detect_scrunch_kernel(const float2* __restrict__ in,
                                                             float* __restrict__ out,
                                                             long long rows, long long Cout,
                                                             int P, int stokes, long long M,
                                                             long long F) {
  const int lane = threadIdx.x & 31;
  const long long Pq = stokes ? 1 : P;
  const long long total = rows * Cout * Pq;
  const long long CP = Cout * F * P;   // complex elements per input row
  const long long wstep = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long o = blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5); o < total;
       o += wstep) {
    const long long j = o / (Cout * Pq), r = o - j * Cout * Pq;
    const long long c = r / Pq, pp = r - c * Pq;
    float acc = 0.f;
    for (long long m = 0; m < M; ++m) {
      const float2* row = in + (j * M + m) * CP + c * F * P;
      if (stokes) {
        for (long long i = lane; i < F * P; i += 32) {
          const float2 v = __ldg(row + i);
          acc += v.x * v.x + v.y * v.y;
        }
      } else {
        for (long long f = lane; f < F; f += 32) {
          const float2 v = __ldg(row + f * P + pp);
          acc += v.x * v.x + v.y * v.y;
        }
      }
    }
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
    if (lane == 0) out[o] = acc;
  }
}

// Fast path: P in {1, 2}, F*P a multiple of 64 complex values, Cout a multiple of CELLS.  A warp
// owns CELLS adjacent output cells of one output row (CELLS*F*P*8 contiguous bytes per input
// row) and keeps CELLS*SWEEPS 128-bit loads in flight per lane before the shuffle reduction.
template <int P, int CELLS>
__global__ void __launch_bounds__(256) detect_scrunch_wide(const float4* __restrict__ in,
                                                           float* __restrict__ out,
                                                           long long rows, long long Cout,
                                                           int stokes, long long M, long long F) {
  const int lane = threadIdx.x & 31;
  const long long cells4 = F * P / 2;                 // float4 per cell per input row
  const long long row4 = Cout * cells4;               // float4 per input row
  const long long groups = rows * (Cout / CELLS);
  const long long wstep = (long long)gridDim.x * (blockDim.x >> 5);
  for (long long g = blockIdx.x * (long long)(blockDim.x >> 5) + (threadIdx.x >> 5); g < groups;
       g += wstep) {
    const long long j = g / (Cout / CELLS), c0 = (g - j * (Cout / CELLS)) * CELLS;
    float a0[CELLS], a1[CELLS];
#pragma unroll
    for (int q = 0; q < CELLS; ++q) a0[q] = a1[q] = 0.f;
    for (long long m = 0; m < M; ++m) {
      const float4* base = in + (j * M + m) * row4 + c0 * cells4 + lane;
      for (long long i = 0; i < cells4; i += 32) {
        float4 v[CELLS];
#pragma unroll
        for (int q = 0; q < CELLS; ++q) v[q] = __ldcs(base + q * cells4 + i);
#pragma unroll
        for (int q = 0; q < CELLS; ++q) {
          a0[q] += v[q].x * v[q].x + v[q].y * v[q].y;
          a1[q] += v[q].z * v[q].z + v[q].w * v[q].w;
        }
      }
    }
#pragma unroll
    for (int q = 0; q < CELLS; ++q) {
      float x = a0[q], y = a1[q];
      if (P == 1 || stokes) { x += y; y = 0.f; }
#pragma unroll
      for (int s = 16; s > 0; s >>= 1) {
        x += __shfl_xor_sync(0xffffffffu, x, s);
        if (P == 2 && !stokes) y += __shfl_xor_sync(0xffffffffu, y, s);
      }
      if (lane == 0) {
        if (P == 2 && !stokes) {
          out[(j * Cout + c0 + q) * 2] = x;
          out[(j * Cout + c0 + q) * 2 + 1] = y;
        } else {
          out[j * Cout + c0 + q] = x;
        }
      }
    }
  }
}

static inline cudaError_t launch_detect_scrunch(const float2* in, float* out, long long rows,
                                                long long Cout, int P, bool stokes, long long M,
                                                long long F, cudaStream_t st) {
  const long long total = rows * Cout * (stokes ? 1 : P);
  if (total <= 0) return cudaSuccess;
  constexpr int CELLS = 8;
  if ((P == 1 || P == 2) && (F * P) % 64 == 0 && Cout % CELLS == 0 &&
      (((uintptr_t)in) & 15) == 0) {
    long long groups = rows * (Cout / CELLS);
    long long blocks = (groups + 7) / 8;
    if (blocks > 148ll * 8) blocks = 148ll * 8;
    if (P == 1)
      detect_scrunch_wide<1, CELLS><<<(unsigned)blocks, 256, 0, st>>>(
          reinterpret_cast<const float4*>(in), out, rows, Cout, stokes ? 1 : 0, M, F);
    else
      detect_scrunch_wide<2, CELLS><<<(unsigned)blocks, 256, 0, st>>>(
          reinterpret_cast<const float4*>(in), out, rows, Cout, stokes ? 1 : 0, M, F);
    return cudaGetLastError();
  }
  long long blocks = (total + 7) / 8;
  if (blocks > 148ll * 16) blocks = 148ll * 16;
  detect_scrunch_kernel<<<(unsigned)blocks, 256, 0, st>>>(in, out, rows, Cout, P, stokes ? 1 : 0,
                                                         M, F);
  return cudaGetLastError();
}

// incoherent dedispersion (transforms/dedispersion.py:136-177): per-channel integer roll + crop,
//   out[n, c, :] = in[n + delay[c], c, :]      n < rows_out
// a pure gather on 4-byte words: `words` words per (row, channel) cell, `C` cells per row.
__global__ void __launch_bounds__(256) shift_channels_kernel(const unsigned* __restrict__ in,
                                                             unsigned* __restrict__ out,
                                                             long long rows_out, long long C,
                                                             long long words,
                                                             const long long* __restrict__ delay) {
  const long long rw = C * words;           // words per row
  const long long total = rows_out * rw;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long n = i / rw, r = i - n * rw;
    const long long c = r / words;
    out[i] = __ldg(in + (n + __ldg(delay + c)) * rw + r);
  }
}

// mixing with a complex sinusoid per column (transforms.py:346 freq_shift):
//   out[n, col] = in[n, col] * exp(+2 pi i ft[col] n),  ft in cycles per sample, phase in FP64
__global__ void __launch_bounds__(256) mix_kernel(const float2* __restrict__ in,
                                                  float2* __restrict__ out, long long nsamp,
                                                  long long ncols,
                                                  const double* __restrict__ ft) {
  const long long total = nsamp * ncols;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long n = i / ncols, col = i - n * ncols;
    const double ph = __ldg(ft + col) * (double)n;
    const double fr = ph - rint(ph);
    float s, c;
    sincospif(2.0f * (float)fr, &s, &c);
    const float2 v = __ldg(in + i);
    out[i] = make_float2(v.x * c - v.y * s, v.x * s + v.y * c);
  }
}

// last step of real_to_complex (utils.py:56-61): multiply by exp(-i pi n / 2) and keep every
// second sample; for n = 2m the factor is (-1)^m exactly.   out[m, :] = (-1)^m in[2m, :]
__global__ void __launch_bounds__(256) decimate2_kernel(const float2* __restrict__ in,
                                                        float2* __restrict__ out,
                                                        long long rows_out, long long ncols) {
  const long long total = rows_out * ncols;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long m = i / ncols, col = i - m * ncols;
    const float2 v = __ldg(in + 2 * m * ncols + col);
    out[i] = (m & 1) ? make_float2(-v.x, -v.y) : v;
  }
}

// full Stokes [I, Q, U, V] from (A, B) pol pairs (core.py:937-966, PSR/IEEE convention)
//   linear:   I=AA+BB  Q=AA-BB  U=2Re(A*B)  V=2Im(A*B)
//   circular: I=AA+BB  Q=2Re(A*B)  U=2Im(A*B)  V=AA-BB          (A*B = conj(A) B)
template <bool V4>
__global__ void __launch_bounds__(256) stokes_kernel(const float2* __restrict__ in,
                                                     float* __restrict__ out, long long n,
                                                     int circular) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    const float4 v = ld_pair<V4>(in + 2 * i);  // (Are, Aim, Bre, Bim)
    const float aa = v.x * v.x + v.y * v.y;
    const float bb = v.z * v.z + v.w * v.w;
    const float re = v.x * v.z + v.y * v.w;   // Re(conj(A) B)
    const float im = v.x * v.w - v.y * v.z;   // Im(conj(A) B)
    st_pair<V4>(out + 4 * i, circular ? make_float4(aa + bb, 2.f * re, 2.f * im, aa - bb)
                                      : make_float4(aa + bb, aa - bb, 2.f * re, 2.f * im));
  }
}

// basis change (core.py:882-928): to_circular: [X - iY, X + iY]/sqrt2 ; to_linear: [L + R, i(L - R)]/sqrt2
template <bool V4>
__global__ void __launch_bounds__(256) pol_basis_kernel(const float2* __restrict__ in,
                                                        float2* __restrict__ out, long long n,
                                                        int to_circular) {
  const float h = 0.70710678118654752440f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    const float4 v = ld_pair<V4>(in + 2 * i);
    float4 o;
    if (to_circular) {   // L = X - iY = (Xre + Yim, Xim - Yre); R = X + iY = (Xre - Yim, Xim + Yre)
      o = make_float4((v.x + v.w) * h, (v.y - v.z) * h, (v.x - v.w) * h, (v.y + v.z) * h);
    } else {             // X = L + R ; Y = i (L - R) = (-(Lim - Rim), Lre - Rre)
      o = make_float4((v.x + v.z) * h, (v.y + v.w) * h, -(v.y - v.w) * h, (v.x - v.z) * h);
    }
    st_pair<V4>(reinterpret_cast<float*>(out + 2 * i), o);
  }
}

template <typename K, typename... A>
static inline cudaError_t launch_1d(K kern, long long n, cudaStream_t st, A... args) {
  if (n <= 0) return cudaSuccess;
  long long blocks = (n + 255) / 256;
  if (blocks > 148ll * 32) blocks = 148ll * 32;
  kern<<<(unsigned)blocks, 256, 0, st>>>(args...);
  return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------
// fold
// ------------------------------------------------------------------------------------------
struct FoldArgs {
  const float* in;
  float* profile;
  unsigned long long* counts;
  int* bins_out;
  double coef[kFoldMaxCoef];
  int ncoef;
  double sample_rate;
  long long n0;
  int nbin;
  long long nsamp, row_elems;
  double rcp_rate;   // RN(1 / sample_rate), see fold_time
  int fast_div;
};

// t = RN(x / sample_rate), bit-equal to numpy's float64 division, without the division sequence:
// with y = RN(1/b) from the host, q = RN(x y) is within one ulp of x/b, r = x - q b is exact in an
// FMA, and q' = RN(q + r y) is the correctly rounded quotient (Markstein's theorem; it needs y
// correctly rounded, q faithful and no underflow/overflow, which fold_args_finish guarantees by
// bounding |x| < 2^53 and 2^-60 < b < 2^200).  Three instructions instead of ~25; the phase of
// every sample goes through here, and at 1-4 floats per sample the fold is instruction-bound.
template <bool ALWAYS_FAST = false>
__device__ __forceinline__ double fold_time(const FoldArgs& a, double x) {
  if (!ALWAYS_FAST && !a.fast_div) return __ddiv_rn(x, a.sample_rate);
  const double q = __dmul_rn(x, a.rcp_rate);
  const double r = __fma_rn(-q, a.sample_rate, x);
  return __fma_rn(r, a.rcp_rate, q);
}

static inline void fold_args_finish(FoldArgs& a) {
  a.rcp_rate = 1.0 / a.sample_rate;
  const long long lim = 1ll << 52;
  a.fast_div = a.sample_rate > 8.7e-19 && a.sample_rate < 1.6e60 && a.n0 > -lim && a.n0 < lim &&
               a.nsamp < lim;
}

// bit-exact restatement of numpy.polynomial.polynomial.polyval + floor binning (oracle fold_bins)
// for the sample whose index n0 + n is x (an integer, exactly representable).  NC > 0: the number
// of coefficients is known at compile time (the per-sample kernels are instantiated for 1..4, so
// that the Horner chain is straight-line code on constant-bank operands), NC = 0: a.ncoef.
template <int NC = 0, bool ALWAYS_FAST = false>
__device__ __forceinline__ int fold_bin_at(const FoldArgs& a, double x) {
  const double t = fold_time<ALWAYS_FAST>(a, x);
  double c0;
  if constexpr (NC > 0) {
    c0 = a.coef[NC - 1];
#pragma unroll
    for (int i = NC - 2; i >= 0; --i) c0 = __dadd_rn(a.coef[i], __dmul_rn(c0, t));
  } else {
    c0 = a.coef[a.ncoef - 1];
    for (int i = a.ncoef - 2; i >= 0; --i) c0 = __dadd_rn(a.coef[i], __dmul_rn(c0, t));
  }
  const double fr = __dsub_rn(c0, floor(c0));
  // fr in [0, 1): floor(fr*nbin) fits an int; fr*nbin can round up to nbin (-> bin 0, like the
  // oracle's `% nbin`); a phase that is not finite (overflowing polynomial) gives NaN -> 0 here
  // and must not index outside the histogram either
  int b = __double2int_rd(__dmul_rn(fr, (double)a.nbin));
  b = b == a.nbin ? 0 : b;
  if ((unsigned)b >= (unsigned)a.nbin) b = 0;
  return b;
}
__device__ __forceinline__ int fold_bin(const FoldArgs& a, long long n) {
  return fold_bin_at<0>(a, (double)(a.n0 + n));
}

// Device-side PhasePredictor.__call__ (pulsar/predictor.py:121-147) for one polyco entry: the
// phase polynomial at dt seconds from the entry's tmid, evaluated with numpy's Horner order in FP64
// without FMA contraction (bit-equal to Polynomial.__call__), split as pulsar/phase.py:28-78 does
// into integer cycles (reference phase + nearest integer) and a fraction in [-0.5, 0.5].
// dt is either given per element or generated as dt0 + (n0 + i) / sample_rate.
struct PredictArgs {
  const double* dt;
  double dt0, sample_rate;
  long long n0, n;
  double coef[kFoldMaxCoef];
  int ncoef;
  long long rphase;
  long long* ph_int;
  double* ph_frac;
};

__global__ void __launch_bounds__(256) phase_predict_kernel(const PredictArgs a) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < a.n;
       i += (long long)gridDim.x * blockDim.x) {
    const double t = a.dt ? a.dt[i]
                          : __dadd_rn(a.dt0, __ddiv_rn((double)(a.n0 + i), a.sample_rate));
    double c0 = a.coef[a.ncoef - 1];
    for (int j = a.ncoef - 2; j >= 0; --j) c0 = __dadd_rn(a.coef[j], __dmul_rn(c0, t));
    const double whole = rint(c0);
    a.ph_int[i] = a.rphase + (long long)whole;
    a.ph_frac[i] = __dsub_rn(c0, whole);
  }
}

static inline cudaError_t launch_phase_predict(const PredictArgs& a, cudaStream_t st) {
  const long long blocks = std::min<long long>((a.n + 255) / 256, 148 * 8);
  phase_predict_kernel<<<(unsigned)blocks, 256, 0, st>>>(a);
  return cudaGetLastError();
}

// phase bin of every sample (and the counts) without touching any data: the fold behind a fused
// channelizer epilogue (pbk_stft_fold_exec_device) adds its sums to the bin's row itself
__global__ void __launch_bounds__(256) fold_bins_kernel(const FoldArgs a, int* __restrict__ bins) {
  for (long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x; n < a.nsamp;
       n += (long long)gridDim.x * blockDim.x) {
    const int b = fold_bin(a, n);
    bins[n] = b;
    atomicAdd(a.counts + b, 1ull);
  }
}

// ---- wide rows (row_elems >= 32): one CTA owns SPAN consecutive samples x up to 256 elements.
// Bins of a chunk of 64 samples are computed once into shared memory; every thread walks its
// element down the chunk (coalesced row segments, 8 loads in flight) and keeps the running sum of
// the current bin in a register, so a global float atomic is issued only when the bin changes
// (every ~200 samples for a slow pulsar) instead of once per sample.  Counts go through a
// per-CTA shared-memory histogram that is flushed once.
constexpr int kFoldChunk = 64;

__global__ void __launch_bounds__(256) fold_wide_kernel(const __grid_constant__ FoldArgs a,
                                                        int span, int smem_counts) {
  extern __shared__ int fsm[];
  int* sbin = fsm;                  // [2][kFoldChunk]
  int* scnt = fsm + 2 * kFoldChunk; // [nbin] (only CTAs with blockIdx.y == 0 use it)
  const long long nb = (long long)blockIdx.x * span;
  const int nrows = (int)min((long long)span, a.nsamp - nb);
  const bool counting = blockIdx.y == 0;
  if (counting && smem_counts)
    for (int i = threadIdx.x; i < a.nbin; i += blockDim.x) scnt[i] = 0;
  const long long e = (long long)blockIdx.y * blockDim.x + threadIdx.x;
  const bool live = e < a.row_elems;
  const float* src = a.in + nb * a.row_elems + (live ? e : 0);
  int cur = -1;
  float acc = 0.f;
  __syncthreads();
  for (int c0 = 0, buf = 0; c0 < nrows; c0 += kFoldChunk, buf ^= 1) {
    const int nr = min(kFoldChunk, nrows - c0);
    int* sb = sbin + buf * kFoldChunk;
    for (int t = threadIdx.x; t < nr; t += blockDim.x) {
      const int b = fold_bin(a, nb + c0 + t);
      sb[t] = b;
      if (counting) {
        if (a.bins_out) a.bins_out[nb + c0 + t] = b;
        if (smem_counts) atomicAdd(scnt + b, 1);
        else atomicAdd(a.counts + b, 1ull);     // histogram too large for shared memory
      }
    }
    __syncthreads();   // one barrier per chunk: the bins are double-buffered
    if (live) {
      const float* p = src + (long long)c0 * a.row_elems;
      int r = 0;
      for (; r + 8 <= nr; r += 8) {
        float v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = __ldg(p + (long long)(r + i) * a.row_elems);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int b = sb[r + i];
          if (b != cur) {
            if (cur >= 0) atomicAdd(a.profile + (long long)cur * a.row_elems + e, acc);
            acc = 0.f;
            cur = b;
          }
          acc += v[i];
        }
      }
      for (; r < nr; ++r) {
        const int b = sb[r];
        if (b != cur) {
          if (cur >= 0) atomicAdd(a.profile + (long long)cur * a.row_elems + e, acc);
          acc = 0.f;
          cur = b;
        }
        acc += __ldg(p + (long long)r * a.row_elems);
      }
    }
  }
  if (live && cur >= 0) atomicAdd(a.profile + (long long)cur * a.row_elems + e, acc);
  __syncthreads();
  if (counting && smem_counts)
    for (int i = threadIdx.x; i < a.nbin; i += blockDim.x)
      if (scnt[i]) atomicAdd(a.counts + i, (unsigned long long)scnt[i]);
}

// ---- narrow rows (row_elems <= 32 and nbin * row_elems floats fit in shared memory): per-CTA
// shared-memory histogram.  A CTA owns SPAN samples, reads them fully coalesced (consecutive
// floats = several samples x all elements), pre-reduces a warp in registers when all its samples
// share one bin (the common case) and adds into the histogram with shared-memory atomics; the
// histogram is flushed to the global profile once per CTA.
constexpr int kFoldNarrowRows = 256;   // samples per chunk (one bin computed per thread)

__global__ void __launch_bounds__(256) fold_narrow_kernel(const __grid_constant__ FoldArgs a,
                                                          int span) {
  extern __shared__ int fsm[];
  const int E = (int)a.row_elems;
  float* hist = reinterpret_cast<float*>(fsm);              // [nbin][E]
  int* scnt = fsm + (size_t)a.nbin * E;                     // [nbin]
  int* sbin = scnt + a.nbin;                                // [kFoldNarrowRows]
  for (int i = threadIdx.x; i < a.nbin * E; i += blockDim.x) hist[i] = 0.f;
  for (int i = threadIdx.x; i < a.nbin; i += blockDim.x) scnt[i] = 0;
  const long long nb = (long long)blockIdx.x * span;
  const int nrows = (int)min((long long)span, a.nsamp - nb);
  const bool pow2 = (32 % E) == 0;      // a warp then holds whole samples: 32/E of them
  const int lane = threadIdx.x & 31;
  __syncthreads();
  for (int c0 = 0; c0 < nrows; c0 += kFoldNarrowRows) {
    const int nr = min(kFoldNarrowRows, nrows - c0);
    if (threadIdx.x < nr) {
      const int b = fold_bin(a, nb + c0 + threadIdx.x);
      sbin[threadIdx.x] = b;
      if (a.bins_out) a.bins_out[nb + c0 + threadIdx.x] = b;
      atomicAdd(scnt + b, 1);
    }
    __syncthreads();
    const float* p = a.in + (nb + c0) * (long long)E;
    const int total = nr * E;
    for (int i0 = 0; i0 < total; i0 += blockDim.x) {       // uniform trip count per warp
      const int i = i0 + threadIdx.x;
      const bool ok = i < total;
      const int r = ok ? i / E : 0, el = ok ? i - r * E : 0;
      float v = ok ? __ldg(p + i) : 0.f;
      const int b = ok ? sbin[r] : -1;
      const int b0 = __shfl_sync(0xffffffffu, b, 0);
      if (pow2 && __all_sync(0xffffffffu, b == b0)) {
        for (int s = E; s < 32; s <<= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
        if (lane < E && b0 >= 0) atomicAdd(hist + b0 * E + el, v);
      } else if (ok) {
        atomicAdd(hist + b * E + el, v);
      }
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < a.nbin * E; i += blockDim.x)
    if (hist[i] != 0.f) atomicAdd(a.profile + i, hist[i]);
  for (int i = threadIdx.x; i < a.nbin; i += blockDim.x)
    if (scnt[i]) atomicAdd(a.counts + i, (unsigned long long)scnt[i]);
}

// ---- rows of 1 to 8, 16 or 32 floats (a single channel's intensity, one or two pols, Stokes,
// a few channels): one thread per sample.  The thread reads its whole row with the widest vector loads
// the row length allows and computes its own bin, four samples per thread in flight so that the
// FP64 Horner chains overlap; a warp whose 32 consecutive samples share one bin (the rule when a
// bin is wider than 32 samples) adds them with shuffles and issues E shared-memory atomics, any
// other warp adds per thread.  No barrier inside the span.
__host__ __device__ constexpr int fold_pow2_ceil(int e) {
  return e <= 1 ? 1 : e <= 2 ? 2 : e <= 4 ? 4 : e <= 8 ? 8 : e <= 16 ? 16 : 32;
}
// bytes the rows must be aligned to for fold_row_load
__host__ __device__ constexpr int fold_row_align(int e) { return e % 4 == 0 ? 16 : e % 2 == 0 ? 8 : 4; }

template <int E>
__device__ __forceinline__ void fold_row_load(const float* __restrict__ p, float* x) {
  if constexpr (E % 4 == 0) {
#pragma unroll
    for (int i = 0; i < E / 4; ++i) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(p) + i);
      x[4 * i] = v.x; x[4 * i + 1] = v.y; x[4 * i + 2] = v.z; x[4 * i + 3] = v.w;
    }
  } else if constexpr (E % 2 == 0) {
#pragma unroll
    for (int i = 0; i < E / 2; ++i) {
      const float2 v = __ldg(reinterpret_cast<const float2*>(p) + i);
      x[2 * i] = v.x; x[2 * i + 1] = v.y;
    }
  } else {
#pragma unroll
    for (int i = 0; i < E; ++i) x[i] = __ldg(p + i);
  }
}

// samples in flight per thread (rows of 16 / 32 floats: fewer, the rows fill the registers)
__host__ __device__ constexpr int fold_vec_unroll(int ep) { return ep <= 8 ? 4 : ep == 16 ? 2 : 1; }

// sum over the 32 lanes of EP (a power of two) values per lane: lane el (< EP) ends up with the
// total of element el.  Halving exchange: while a lane holds more than one element it keeps the
// half selected by one bit of its lane number and hands the other half to the partner across
// that bit, then plain butterflies over the remaining bits -- EP - 1 + (5 - log2 EP) shuffles
// instead of 5 EP.  x is overwritten.
template <int EP>
__device__ __forceinline__ float fold_warp_sum(float* x, int lane) {
#pragma unroll
  for (int h = EP / 2; h >= 1; h >>= 1) {
    const bool up = lane & h;                       // these lanes collect elements [h, 2h)
#pragma unroll
    for (int i = 0; i < h; ++i) {
      const float keep = up ? x[i + h] : x[i], give = up ? x[i] : x[i + h];
      x[i] = keep + __shfl_xor_sync(0xffffffffu, give, h);
    }
  }
  float s = x[0];
#pragma unroll
  for (int d = 16; d >= EP; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
  return s;                                         // lane l holds element l & (EP - 1)
}

template <int E, int NC>
__global__ void __launch_bounds__(256) fold_vec_kernel(const __grid_constant__ FoldArgs a,
                                                       int span) {
  constexpr int EP = fold_pow2_ceil(E);
  constexpr int kFoldVecUnroll = fold_vec_unroll(EP);
  extern __shared__ int fsm[];
  float* hist = reinterpret_cast<float*>(fsm);              // [nbin][E]
  int* scnt = fsm + (size_t)a.nbin * E;                     // [nbin]
  for (int i = threadIdx.x; i < a.nbin * E; i += blockDim.x) hist[i] = 0.f;
  for (int i = threadIdx.x; i < a.nbin; i += blockDim.x) scnt[i] = 0;
  const long long nb = (long long)blockIdx.x * span;
  const int nrows = (int)min((long long)span, a.nsamp - nb);
  const float* src = a.in + nb * E;
  const double base = (double)(a.n0 + nb);      // exact, and so is base + r (integers < 2^53)
  const int lane = threadIdx.x & 31;
  __syncthreads();
  for (int r0 = 0; r0 < nrows; r0 += 256 * kFoldVecUnroll) {   // uniform trip count per CTA
    float v[kFoldVecUnroll][EP];
    int b[kFoldVecUnroll];
#pragma unroll
    for (int u = 0; u < kFoldVecUnroll; ++u) {
      const int r = r0 + u * 256 + (int)threadIdx.x;
#pragma unroll
      for (int el = 0; el < EP; ++el) v[u][el] = 0.f;
      if (r < nrows) fold_row_load<E>(src + (long long)r * E, v[u]);
    }
#pragma unroll
    for (int u = 0; u < kFoldVecUnroll; ++u) {
      const int r = r0 + u * 256 + (int)threadIdx.x;
      b[u] = r < nrows ? fold_bin_at<NC, true>(a, __dadd_rn(base, (double)r)) : -1;
      if (r < nrows && a.bins_out) a.bins_out[nb + r] = b[u];
    }
#pragma unroll
    for (int u = 0; u < kFoldVecUnroll; ++u) {
      // up to three rounds of "the lanes that share the first pending lane's bin add up with
      // shuffles": one round when the warp's 32 samples share a bin, two when a bin boundary
      // falls inside the warp; small groups and what is left after three rounds (bins narrower
      // than ~10 samples) are added per thread, where few lanes collide on one address
      const float* x = v[u];
      unsigned todo = __ballot_sync(0xffffffffu, b[u] >= 0), rest = 0u;
#pragma unroll 1
      for (int round = 0; round < 3 && todo; ++round) {
        const int bb = __shfl_sync(0xffffffffu, b[u], __ffs(todo) - 1);
        const bool mine = b[u] == bb;
        const unsigned m = __ballot_sync(0xffffffffu, mine);
        todo &= ~m;
        if (__popc(m) < 6) {            // few lanes in this bin: their atomics below hardly collide
          rest |= m;
          continue;
        }
        float y[EP];
#pragma unroll
        for (int el = 0; el < EP; ++el) y[el] = mine ? x[el] : 0.f;
        const float s = fold_warp_sum<EP>(y, lane);
        if (lane < E) atomicAdd(hist + bb * E + lane, s);
        if (lane == 0) atomicAdd(scnt + bb, __popc(m));
      }
      if (((todo | rest) >> lane) & 1u) {
#pragma unroll
        for (int el = 0; el < E; ++el) atomicAdd(hist + b[u] * E + el, x[el]);
        atomicAdd(scnt + b[u], 1);
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < a.nbin * E; i += blockDim.x)
    if (hist[i] != 0.f) atomicAdd(a.profile + i, hist[i]);
  for (int i = threadIdx.x; i < a.nbin; i += blockDim.x)
    if (scnt[i]) atomicAdd(a.counts + i, (unsigned long long)scnt[i]);
}

template <int E, int NC>
static inline cudaError_t launch_fold_vec_nc(const FoldArgs& a, size_t smem, int span,
                                             cudaStream_t st) {
  static bool attr_done[16] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 16 && !attr_done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(fold_vec_kernel<E, NC>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
    if (e != cudaSuccess) return e;
    attr_done[dev] = true;
  }
  const long long gx = (a.nsamp + span - 1) / span;
  fold_vec_kernel<E, NC><<<(unsigned)gx, 256, smem, st>>>(a, span);
  return cudaGetLastError();
}

template <int E>
static inline cudaError_t launch_fold_vec(const FoldArgs& a, size_t smem, int span,
                                          cudaStream_t st) {
  switch (a.ncoef) {
    case 1: return launch_fold_vec_nc<E, 1>(a, smem, span, st);
    case 2: return launch_fold_vec_nc<E, 2>(a, smem, span, st);
    case 3: return launch_fold_vec_nc<E, 3>(a, smem, span, st);
    case 4: return launch_fold_vec_nc<E, 4>(a, smem, span, st);
    default: return launch_fold_vec_nc<E, 0>(a, smem, span, st);
  }
}

static inline int fold_pick_span(long long nsamp, long long ctas_per_span, int lo, int hi) {
  // enough CTAs to fill the 148 SMs several times over, long enough spans to amortise atomics
  long long span = hi;
  while (span > lo && (nsamp + span - 1) / span * ctas_per_span < 148ll * 8) span >>= 1;
  return (int)span;
}

static inline cudaError_t launch_fold(const FoldArgs& a, cudaStream_t st) {
  if (a.nsamp <= 0) return cudaSuccess;
  const size_t narrow_smem = ((size_t)a.nbin * a.row_elems + a.nbin + kFoldNarrowRows) * 4;
  if (a.row_elems <= 32 && narrow_smem <= 160 * 1024) {
    static bool attr_done[16] = {};
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 16 && !attr_done[dev]) {
      cudaError_t e = cudaFuncSetAttribute(fold_narrow_kernel,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
      if (e != cudaSuccess) return e;
      attr_done[dev] = true;
    }
    // a span must be long against nbin so that the flush is amortised
    const int span = fold_pick_span(a.nsamp, 1, 4096, 65536);
    const size_t vec_smem = ((size_t)a.nbin * a.row_elems + a.nbin) * 4;
    // (sample rates outside fold_args_finish's range keep the division of the scalar kernel)
    const uintptr_t addr = reinterpret_cast<uintptr_t>(a.in);
    if (a.fast_div)
      switch (a.row_elems) {
#define PBK_FOLD_VEC_CASE(E) \
        case E: if (addr % fold_row_align(E) == 0) return launch_fold_vec<E>(a, vec_smem, span, st); \
                break;
        PBK_FOLD_VEC_CASE(1) PBK_FOLD_VEC_CASE(2) PBK_FOLD_VEC_CASE(3) PBK_FOLD_VEC_CASE(4)
        PBK_FOLD_VEC_CASE(5) PBK_FOLD_VEC_CASE(6) PBK_FOLD_VEC_CASE(7) PBK_FOLD_VEC_CASE(8)
        PBK_FOLD_VEC_CASE(16) PBK_FOLD_VEC_CASE(32)
#undef PBK_FOLD_VEC_CASE
        default: break;
      }
    const long long gx = (a.nsamp + span - 1) / span;
    fold_narrow_kernel<<<(unsigned)gx, 256, narrow_smem, st>>>(a, span);
    return cudaGetLastError();
  }
  const int threads = a.row_elems >= 256 ? 256 : (int)((a.row_elems + 31) / 32 * 32);
  const long long gy = (a.row_elems + threads - 1) / threads;
  if (gy > 65535) return cudaErrorInvalidValue;
  const int smem_counts = a.nbin <= 11000;                // else count with global atomics
  const size_t smem = (2 * kFoldChunk + (smem_counts ? (size_t)a.nbin : 0)) * 4;
  const int span = fold_pick_span(a.nsamp, gy, 256, 4096);
  dim3 grid((unsigned)((a.nsamp + span - 1) / span), (unsigned)gy);
  fold_wide_kernel<<<grid, threads, smem, st>>>(a, span, smem_counts);
  return cudaGetLastError();
}

}  // namespace pbk
