// pbk_incoh.cuh -- incoherent dedispersion at many trial DMs, summed over frequency (DM x time
// plane): out[k, j, p] = sum_{c < C} in[j + e[k, c], c, p], channels added in ascending order in
// float32 (deterministic: no atomics, one thread owns each output element).
//
// Tiling (DESIGN.md 5.4e).  The plan sorts the trials by sweep and groups them into blocks of KD.
// One CTA computes kFlat output floats (TT = kFlat / P rows x P) of each of the KD trials of one
// block.  It walks the channels in chunks of CC adjacent channels; for each chunk it stages the
// rectangle of input rows that any of its KD trials reads, [j0 + lo, j0 + lo + TT + ext) x CC x P,
// into shared memory (coalesced rows of CC * P floats, stored channel-major), then every warp adds
// the chunk's channels to its accumulators: lanes read consecutive shared words (conflict-free),
// one shared read per add.  Load / add overlap comes from several resident CTAs per SM.
#pragma once

#include <cuda_runtime.h>

namespace pbk_incoh {

constexpr int kThreads = 256;                // 8 warps
constexpr int kWarps = kThreads / 32;
constexpr int kFlat = 512;                   // output floats (rows x P) per trial per CTA
constexpr int kMaxP = 256;                   // TT = kFlat / P >= 2 rows

struct Args {
  const float* in;
  float* out;
  long long row_elems;   // C * P: floats per input row
  int C, P, rows;        // channels, floats per cell, output rows per trial
  int TT;                // output rows per CTA tile (kFlat / P)
  int CC, nq;            // channels per chunk, chunks
  int stride;            // shared floats per staged channel (>= ext_max * P + kFlat)
  int nb;                // trial blocks
  const int* perm;       // [nb * KD] caller's trial index of each sorted slot, -1 = padding
  const int* off;        // [nb * KD * C] e[k, c] - lo[b, q(c)]
  const int* lo;         // [nb * nq] least delay of the block over the chunk
  const int* ext;        // [nb * nq] greatest delay minus lo
};

template <int KD>
__global__ void __launch_bounds__(kThreads, 2) incoh_trials_kernel(Args a) {
  extern __shared__ float s[];
  constexpr int NWT = kWarps / KD;            // warps per trial
  constexpr int R = kFlat / (NWT * 32);       // accumulators per thread
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int kslot = warp / NWT, wi = warp % NWT;
  // trial blocks vary fastest, so the CTAs resident at one time share their input rows in L2
  const int b = (int)(blockIdx.x % (unsigned)a.nb);
  const int j0 = (int)(blockIdx.x / (unsigned)a.nb) * a.TT;
  const int nflat = min(a.TT, a.rows - j0) * a.P;
  const int nrow = min(a.TT, a.rows - j0);
  const int k = a.perm[b * KD + kslot];
  const int* offk = a.off + (long long)(b * KD + kslot) * a.C;

  float acc[R];
#pragma unroll
  for (int m = 0; m < R; ++m) acc[m] = 0.f;

  for (int q = 0; q < a.nq; ++q) {
    const int c0 = q * a.CC;
    const int ncc = min(a.CC, a.C - c0);
    const int wq = ncc * a.P;                  // floats of one staged row (<= kThreads)
    const int lo = a.lo[b * a.nq + q];
    const int nst = nrow + a.ext[b * a.nq + q];
    const int rstep = kThreads / wq;
    const int r0 = tid / wq;
    if (r0 < rstep) {
      const int col = tid - r0 * wq;
      const int cc = col / a.P, p = col - cc * a.P;
      float* dst = s + cc * a.stride + p;
      const float* src = a.in + (long long)(j0 + lo) * a.row_elems + (long long)c0 * a.P + col;
      int r = r0;
      for (; r + 3 * rstep < nst; r += 4 * rstep) {
        const float v0 = __ldg(src + (long long)r * a.row_elems);
        const float v1 = __ldg(src + (long long)(r + rstep) * a.row_elems);
        const float v2 = __ldg(src + (long long)(r + 2 * rstep) * a.row_elems);
        const float v3 = __ldg(src + (long long)(r + 3 * rstep) * a.row_elems);
        dst[r * a.P] = v0;
        dst[(r + rstep) * a.P] = v1;
        dst[(r + 2 * rstep) * a.P] = v2;
        dst[(r + 3 * rstep) * a.P] = v3;
      }
      for (; r < nst; r += rstep) dst[r * a.P] = __ldg(src + (long long)r * a.row_elems);
    }
    __syncthreads();
    if (k >= 0) {
      for (int cc = 0; cc < ncc; ++cc) {
        const float* sp = s + cc * a.stride + offk[c0 + cc] * a.P + wi * 32 + lane;
#pragma unroll
        for (int m = 0; m < R; ++m) acc[m] += sp[m * NWT * 32];
      }
    }
    __syncthreads();
  }
  if (k < 0) return;
  float* o = a.out + ((long long)k * a.rows + j0) * a.P;
#pragma unroll
  for (int m = 0; m < R; ++m) {
    const int i = wi * 32 + lane + m * NWT * 32;
    if (i < nflat) o[i] = acc[m];
  }
}

inline const void* kernel_of(int KD) {
  switch (KD) {
    case 8: return (const void*)incoh_trials_kernel<8>;
    case 4: return (const void*)incoh_trials_kernel<4>;
    case 2: return (const void*)incoh_trials_kernel<2>;
    default: return (const void*)incoh_trials_kernel<1>;
  }
}

inline cudaError_t launch(int KD, const Args& a, unsigned grid, size_t smem, cudaStream_t st) {
  switch (KD) {
    case 8: incoh_trials_kernel<8><<<grid, kThreads, smem, st>>>(a); break;
    case 4: incoh_trials_kernel<4><<<grid, kThreads, smem, st>>>(a); break;
    case 2: incoh_trials_kernel<2><<<grid, kThreads, smem, st>>>(a); break;
    default: incoh_trials_kernel<1><<<grid, kThreads, smem, st>>>(a); break;
  }
  return cudaGetLastError();
}

}  // namespace pbk_incoh
