// pbk_fast.cuh -- second-generation tile-FFT pass kernel: everything about the tile is a
// compile-time constant (radix list, lane pairs per tile, thread count), CTAs are persistent
// (grid = resident CTAs, each loops over tiles), stage twiddles live in shared memory, and the
// inter-level twiddle W_M^(nrest*k) is factored into a per-task root times a per-tile table so a
// task needs one sincospif instead of seven.
//
// These kernels are specialised at compile time to the coherent-dedispersion passes: FWD =
// forward level with its level twiddle (complex64, int8 or pair-planar scratch input), MID =
// fft * generated chirp * ifft, INV = inverse level + epilogue (kind and crop handling are template
// parameters).  Run-time switches around code that touches the 64-register data array make the
// compiler copy the whole array at every merge point, so there are none.  The scratch array
// between passes is pair-planar ({re0,re1,im0,im1} per lane pair = the packed register layout),
// the per-tile address record is computed by one thread and broadcast through shared memory, and
// the chirp is evaluated in FP64 without a division (see fast_chirp).
// Preconditions checked by the host (pbk_api.cu: setup_fast): uniform lane pairs (I and P even,
// pair adjacent and 16-byte aligned in both maps), a tile never straddles a row (I % W == 0,
// W % P == 0), no fftshift bookkeeping, forward sign, unit scale, generated chirp with
// |f - fc| <= fc/16.  Everything else runs on the generic kernel in pbk_fft.cuh, which is the
// same algorithm with runtime tile parameters.
#pragma once
#include <type_traits>

#include "pbk_fft.cuh"

namespace pbk {

constexpr int ilog2c(int v) { return v <= 1 ? 0 : 1 + ilog2c(v >> 1); }

template <int R0_, int R1_, int R2_, int R3_, int LOG2PW_, int NT_, int MINB_>
struct FastCfg {
  static constexpr int NS = (R0_ > 1) + (R1_ > 1) + (R2_ > 1) + (R3_ > 1);
  static constexpr int L = R0_ * R1_ * R2_ * R3_;
  static constexpr int LOG2L = ilog2c(L);
  static constexpr int LOG2PW = LOG2PW_;
  static constexpr int PW = 1 << LOG2PW_;
  static constexpr int W = 2 * PW;
  static constexpr int NT = NT_;
  static constexpr int MINB = MINB_;
  __host__ __device__ static constexpr int radix(int j) {
    return j == 0 ? R0_ : j == 1 ? R1_ : j == 2 ? R2_ : R3_;
  }
  __host__ __device__ static constexpr int stride(int j) {  // S_j = L / (R_0 .. R_j)
    int s = L;
    for (int i = 0; i <= j; ++i) s /= radix(i);
    return s;
  }
  static constexpr int RL = radix(NS - 1);       // radix of the last (stride-1) stage
  static constexpr int LOG2RL = ilog2c(RL);
  static constexpr int KS = L / RL;              // k spacing between last-stage registers
  static constexpr int PPB = (8 >> LOG2PW_) > 1 ? (8 >> LOG2PW_) : 1;  // points per 128 bytes
  __host__ __device__ static constexpr int tw_off(int j) {  // float2 offset of stage j's table
    int o = 0;
    for (int i = 0; i < j; ++i) o += (radix(i) - 1) * stride(i);
    return o;
  }
  static constexpr int TW_TOTAL = tw_off(NS - 1) > 0 ? tw_off(NS - 1) : 1;
  static constexpr size_t TILE_BYTES = (size_t)L * PW * sizeof(float4);
  // tile | stage tables (padded to 16 B) | level-twiddle tables G (one of RL float4 per row of
  // lanes in the tile: up to W/2 rows when the array has only 2 lanes per row) | TileInfo
  static constexpr int TW_PAD = (TW_TOTAL + 1) & ~1;
  static constexpr int G_ROWS = W / 2;
  static constexpr size_t SMEM_BASE = TILE_BYTES + (size_t)TW_PAD * sizeof(float2) + 64;
  __host__ __device__ static constexpr size_t smem_bytes(bool narrow) {
    return SMEM_BASE + (size_t)RL * (narrow ? G_ROWS : 1) * sizeof(float4);
  }
  static constexpr size_t SMEM_BYTES = smem_bytes(true);
};

// host-side builder of the stage tables in the layout the kernel expects:
// stage j, [m-1][q] -> exp(-2 pi i q m / (R_j S_j)), m = 1..R_j-1, q < S_j
template <class C>
static inline void fast_build_tables(float2* dst) {
  for (int j = 0; j + 1 < C::NS; ++j) {
    const int R = C::radix(j), S = C::stride(j);
    const long long M = (long long)R * S;
    float2* t = dst + C::tw_off(j);
    for (int m = 1; m < R; ++m)
      for (int q = 0; q < S; ++q) {
        const long long e = ((long long)q * m) % M;
        const double ang = -2.0 * 3.14159265358979323846 * (double)e / (double)M;
        t[(m - 1) * S + q] = make_float2((float)cos(ang), (float)sin(ang));
      }
  }
}

// ------------------------------------------------------------------------------------------
// shared-memory addressing (float4 index) with the XOR swizzle on the low point bits
// ------------------------------------------------------------------------------------------
template <class C, int S>
__device__ __forceinline__ int phys_pt(int base, int i) {
  if constexpr (C::PPB == 1) {
    return base + i * S;
  } else if constexpr (S % (C::RL * C::PPB) == 0) {
    const int sw = (base >> C::LOG2RL) & (C::PPB - 1);
    return (base ^ sw) + i * S;
  } else {
    static_assert(S >= C::RL, "non-final stage strides are multiples of the last radix");
    const int sw = ((base >> C::LOG2RL) + i * (S / C::RL)) & (C::PPB - 1);
    return (base + i * S) ^ sw;
  }
}

__device__ __forceinline__ c2 lds_c2(const float4* s, int idx) {
  const float4 t = s[idx];
  c2 v;
  v.re = make_float2(t.x, t.y);
  v.im = make_float2(t.z, t.w);
  return v;
}
__device__ __forceinline__ void sts_c2(float4* s, int idx, c2 v) {
  s[idx] = make_float4(v.re.x, v.re.y, v.im.x, v.im.y);
}

template <int R, int S, bool CONJ>
__device__ __forceinline__ void stage_twiddle(c2* v, const float2* tw, int q) {
#pragma unroll
  for (int m = 1; m < R; ++m) {
    const float2 w = tw[(m - 1) * S + q];
    v[m] = cmul(v[m], p_bc(w.x), p_bc(CONJ ? -w.y : w.y));
  }
}

// digit reversal: last-stage block index -> low part of the tile-level frequency index
template <class C>
__device__ __forceinline__ int klo_of(int b) {
  if constexpr (C::NS <= 1) {
    return 0;
  } else if constexpr (C::NS == 2) {
    return b;
  } else if constexpr (C::NS == 3) {
    return (b / C::radix(1)) + C::radix(0) * (b % C::radix(1));
  } else {
    const int m2 = b % C::radix(2);
    const int t = b / C::radix(2);
    const int m1 = t % C::radix(1);
    const int m0 = t / C::radix(1);
    return m0 + C::radix(0) * (m1 + C::radix(1) * m2);
  }
}

// per-tile context (uniform across the CTA) and per-thread lane-pair pointers
struct FastTile {
  const char* gin;    // byte pointer to this thread's lane pair at row 0 of the tile (input)
  char* gout;         // same for the output map (already shifted by the crop for final passes)
  unsigned nrest;     // inner time offset shared by the whole tile
  unsigned klow;      // low part of the full frequency index (MID chirp)
  int chan;           // channel of this thread's pair
  unsigned row_lo, row_cnt;   // final passes: rows [row_lo, row_lo+row_cnt) survive the crop
};

constexpr int EPI_SCRATCH = 3;   // not a final pass: pair-planar complex64 to the scratch array
// how a pass reads its input: user complex64 (re,im interleaved), user int8 pairs, or the scratch
// array, where each 16-byte lane pair is stored as {re0, re1, im0, im1} ("pair-planar") so that a
// 128-bit access is exactly the packed register layout of c2 and needs no shuffling
enum { LK_C64 = 0, LK_I8 = 1, LK_PLANAR = 2,
       LK_TRANSP = 3 /* user complex64 where every lane pair owns a contiguous run of rows
                        (ISTFT input): transposed through shared memory */,
       LK_U4 = 4 /* packed 4+4-bit complex: two bytes per lane pair */,
       LK_U2 = 5 /* packed 2+2-bit complex: one byte per lane pair */,
       LK_TRANSP_PLANAR = 6 /* scratch (pair-planar) where every lane pair owns a contiguous run of
                               rows: the last level of an array with ONE lane pair per row */ };
// bits per complex input element
__host__ __device__ constexpr int lk_bits(int lk) {
  return lk == LK_I8 ? 16 : lk == LK_U4 ? 8 : lk == LK_U2 ? 4 : 64;
}

// everything about a tile that is uniform across the CTA; computed by one thread (the address
// arithmetic has 64-bit divisions) and broadcast through shared memory
struct TileInfo {
  long long bi, bo;     // byte offsets of lane pair 0, row 0 in the input / output array
  unsigned nrest, klow; // of lane 0
  unsigned kprev;       // of lane 0 (MID tiles narrower than W lanes span several of them)
  int chan0;
  unsigned row_lo, row_cnt;   // crop row range of lane 0 (all lanes when the tile is one row)
};

template <class C, int EPI>
__device__ __forceinline__ void fast_tile_info(const PassArgs& p, long long tile, TileInfo& ti,
                                               int in_elem_bits, int out_elem_bytes) {
  const long long q0 = tile * C::W;              // first lane of the tile
  const long long o = q0 / p.RI;
  const long long r0 = q0 - o * p.RI;
  const long long nrest = r0 / p.I;
  const int col0 = (int)(r0 - nrest * p.I);      // multiple of W (hence of P), or 0 when I < W
  const long long o_orig = o >> p.log2Kprev;
  const long long kprev = o & ((1ll << p.log2Kprev) - 1);
  const long long klow = (kprev >> p.kl_sa) + ((kprev & p.kl_mb) << p.kl_sb);
  // (lane pairs start at even elements, so packed sub-byte inputs land on whole bytes)
  ti.bi = (map_base(p.min, o_orig, kprev, klow, nrest, col0, p.P) * in_elem_bits) >> 3;
  long long bo = map_base(p.mout, o_orig, kprev, klow, nrest, col0, p.P) * out_elem_bytes;
  ti.nrest = (unsigned)nrest;
  ti.klow = (unsigned)klow;
  ti.kprev = (unsigned)kprev;
  ti.chan0 = col0 / p.P;
  ti.row_lo = 0;
  ti.row_cnt = C::L;
  if (EPI != EPI_SCRATCH) {
    // time index of tile row r is r*n_mul + nrest (n_mul = 2^log2nmul); keep crop_start <= n <
    // crop_stop  <=>  r in [ceil((start-nrest)/n_mul), ceil((stop-nrest)/n_mul))
    const long long add = (1ll << p.log2nmul) - 1;
    long long lo = (p.crop_start - nrest + add) >> p.log2nmul;
    long long hi = (p.crop_stop - nrest + add) >> p.log2nmul;
    lo = lo < 0 ? 0 : lo;
    hi = hi > C::L ? C::L : hi;
    ti.row_lo = (unsigned)lo;
    ti.row_cnt = hi > lo ? (unsigned)(hi - lo) : 0u;
    bo -= p.crop_start * p.mout.a_n * out_elem_bytes;
  }
  ti.bo = bo;
}

// Every element is touched once per pass.  Evict-first hints (ld.global.cs / st.global.cs) were
// measured SLOWER than plain L2-cached accesses on B200 (cfg2: 7.58 vs 7.42 ms), so the default is
// ld.global.cg + plain stores; PBK_STREAM_HINTS restores the hints for experiments.
#ifdef PBK_STREAM_HINTS
#define PBK_STCS(ptr, val) __stcs((ptr), (val))
__device__ __forceinline__ float4 ldg_stream_f4(const void* ptr) {
  return __ldcs(reinterpret_cast<const float4*>(ptr));
}
#else
#define PBK_STCS(ptr, val) (*(ptr) = (val))
__device__ __forceinline__ float4 ldg_stream_f4(const void* ptr) {
  return __ldcg(reinterpret_cast<const float4*>(ptr));
}
#endif

template <int LOADK>
__device__ __forceinline__ c2 fast_load(const FastTile& T, unsigned row, unsigned rowbytes) {
  const char* a = T.gin + (unsigned long long)row * rowbytes;
  c2 v;
  if (LOADK == LK_PLANAR) {
    const float4 t = ldg_stream_f4(a);
    v.re = make_float2(t.x, t.y);
    v.im = make_float2(t.z, t.w);
  } else if (LOADK == LK_C64) {
    const float4 t = ldg_stream_f4(a);
    v.re = make_float2(t.x, t.z);
    v.im = make_float2(t.y, t.w);
  } else if (LOADK == LK_U4) {
    const unsigned t = __ldcs(reinterpret_cast<const unsigned short*>(a));
    v.re = make_float2(dec4(t), dec4(t >> 8));
    v.im = make_float2(dec4(t >> 4), dec4(t >> 12));
  } else if (LOADK == LK_U2) {
    const unsigned t = __ldcs(reinterpret_cast<const unsigned char*>(a));
    v.re = make_float2(dec2(t & 3u), dec2((t >> 4) & 3u));
    v.im = make_float2(dec2((t >> 2) & 3u), dec2((t >> 6) & 3u));
  } else {
    const char4 t = __ldcs(reinterpret_cast<const char4*>(a));
    v.re = make_float2((float)t.x, (float)t.z);
    v.im = make_float2((float)t.y, (float)t.w);
  }
  return v;
}

// scratch store: pair-planar {re0, re1, im0, im1}
__device__ __forceinline__ void fast_store_c64(const FastTile& T, unsigned row, unsigned rowbytes,
                                               c2 v) {
  PBK_STCS(reinterpret_cast<float4*>(T.gout + (unsigned long long)row * rowbytes),
           make_float4(v.re.x, v.re.y, v.im.x, v.im.y));
}

// store of an inverse pass: scratch (streaming complex64) or the final epilogue -- crop on the
// time index (hoisted to a row range per tile), then c64 / per-pol intensity / Stokes I
template <int EPI>
__device__ __forceinline__ void fast_store_out(const FastTile& T, unsigned row,
                                               unsigned rowbytes, c2 v) {
  char* a = T.gout + (unsigned long long)row * rowbytes;
  if (EPI == EPI_SCRATCH) {
    PBK_STCS(reinterpret_cast<float4*>(a), make_float4(v.re.x, v.re.y, v.im.x, v.im.y));
    return;
  }
  if (row - T.row_lo >= T.row_cnt) return;
  if (EPI == EPI_C64) {
    *reinterpret_cast<float4*>(a) = make_float4(v.re.x, v.im.x, v.re.y, v.im.y);
  } else {
    const float2 pw = p_fma(v.re, v.re, p_mul(v.im, v.im));
    if (EPI == EPI_INTENSITY) *reinterpret_cast<float2*>(a) = pw;
    else *reinterpret_cast<float*>(a) = pw.x + pw.y;
  }
}

// level twiddle for the R registers of a last-stage group: W_M^(nrest*(klo + KS*m))
//   = E * G[m],  E = W_M^(nrest*klo) (one exact root per task), G[m] = W_M^(nrest*KS*m) (per tile,
//   kept in shared memory as {G.x, G.y, G.y, G.x} so that E*G[m] is two packed instructions)
// (GS = float4 stride between consecutive m: 1 for the one table of a wide tile; narrow tiles keep
// a table per lane row stored m-major, [m][row], so that the threads of a quarter-warp -- eight
// different lane rows -- read eight consecutive 16-byte entries instead of one bank group 8 times)
template <int R, bool CONJ, int GS = 1>
__device__ __forceinline__ void level_twiddle(const PassArgs& p, c2* v, unsigned nrest,
                                              unsigned klo, const float4* G4) {
  const float2 E = unit_root((unsigned long long)nrest * klo, p.log2M);
  const float2 ex = p_bc(E.x), ey = make_float2(-E.y, E.y);
#pragma unroll
  for (int m = 0; m < R; ++m) {
    float2 w = E;
    if (m > 0) {
      const float4 g = G4[m * GS];
      w = p_fma(make_float2(g.x, g.y), ex, p_mul(make_float2(g.z, g.w), ey));
    }
    v[m] = cmul(v[m], p_bc(w.x), p_bc(CONJ ? -w.y : w.y));
  }
}

// chirp for the R registers of a last-stage group (uniform pair: one value serves both lanes).
// Only the generated chirp runs here; an explicit chirp array goes through the generic kernel.
// Reference: dedispersion.py:19-23, H = exp(-2 pi i phi), phi = D f (1/fr - 1/f)^2 cycles with
// f = f_chan + fftfreq[k].
//  * Register m holds full frequency index k_m = k_0 + m*N/R with k_0 < N/R, so the fftfreq wrap
//    (k >= N/2 -> k - N, dedispersion.py:20) is "m >= R/2" at compile time and the signed index
//    is ks = k_0 + N*c_m, c_m = m/R - [m >= R/2]: one exact FP64 fma, no integer work.
//  * With delta = ks*df (offset from the channel centre fc) the cancellation-free form is
//        phi = (D/fc) * a^2 / (1 + x),   a = (fc - fr)/fr + delta/fr,   x = delta/fc,
//    and 1/(1+x) comes from the cubic 1 - x + x^2 - x^3 refined by two Newton steps (error x^16;
//    the host only selects this kernel when |x| <= 1/16), so there is no FP64 division.
//    cc = {(fc-fr)/fr, df/fc, D/fc} per channel, p.bd = df/fr.
//  * phi is reduced exactly (phi - rint(phi), |.| <= 1/2 cycle) before the FP32 sine/cosine.
// FP64 phase of one channel at signed bin ks (see the comment above), reduced to [-0.5, 0.5]
__device__ __forceinline__ float2 fast_chirp_value(const PassArgs& p, const double* cc, double ks) {
  const double a = fma(ks, p.bd, cc[0]);
  const double x = ks * cc[1];
  const double u = 1.0 + x;
  double r = fma(x, fma(x, 1.0 - x, -1.0), 1.0);
  r = fma(r, fma(-u, r, 1.0), r);
  r = fma(r, fma(-u, r, 1.0), r);
  const double phi = (a * a) * (r * cc[2]);             // cycles
  const double fr = phi - rint(phi);                    // exact reduction to [-0.5, 0.5]
  float sn, cs;
#ifdef PBK_ACCURATE_SINCOS
  sincospif(2.0f * (float)fr, &sn, &cs);
#else
  __sincosf(6.283185307179586f * (float)fr, &sn, &cs);   // MUFU, |error| < 5e-7 on |x| <= pi
#endif
  return make_float2(cs * p.scale, -sn * p.scale);
}

// TWOCH: single-polarisation data (P = 1) -- the two lanes of a pair are two adjacent channels,
// each with its own chirp; otherwise the pair is the two pols of one channel and shares it.
// Batch index (blockIdx.y) of a batched launch: the trial of a trial plan, or the overlap-save
// block of pbk_dedisp_exec_blocks_device.  Read where it is used, so that the compiler does not
// keep it (and the offsets built from it) live across the tile loop.
__device__ __forceinline__ long long trial_y() {
  unsigned y;
  asm volatile("mov.u32 %0, %%ctaid.y;" : "=r"(y));
  return (long long)y;
}

template <int R, class C, bool TWOCH>
__device__ __forceinline__ void fast_chirp(const PassArgs& p, const FastTile& T, c2* v, int klo) {
  const double k0 = (double)((long long)T.klow + ((long long)klo << p.log2Kmul));
  const double Nd = (double)p.N;
  double cc0[3], cc1[3];
  const double* cc = p.chan_const + trial_y() * p.trial_cc + 3 * T.chan;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    cc0[i] = cc[i];
    cc1[i] = TWOCH ? cc[3 + i] : 0.0;
  }
  if (TWOCH && p.split) {
    // ONE column of length 2N whose even / odd samples are the two lanes (radix-2 decimation in
    // time done by the memory layout: row j of the (N, 2) view holds x[2j], x[2j+1]).  Register m
    // holds E[k], O[k] of the two half-length transforms at the natural index k = k0 + m N/R:
    //   X[k] = E + w O,  X[k+N] = E - w O,  w = exp(-i pi k / N)      (full-length spectrum)
    //   Y[k] = X[k] H(k),  Y[k+N] = X[k+N] H(k - N)                   (fftfreq: k+N >= 2N/2)
    //   E' = (Y[k] + Y[k+N]) / 2,  O' = conj(w) (Y[k] - Y[k+N]) / 2   (the 1/2 is in p.scale)
    const long long k0i = (long long)T.klow + ((long long)klo << p.log2Kmul);
    const int log2N2 = 64 - __clzll((unsigned long long)p.N);          // log2(2N)
#pragma unroll
    for (int m = 0; m < R; ++m) {
      const double kn = fma((double)m / R, Nd, k0);
      const float2 h0 = fast_chirp_value(p, cc0, kn);
      const float2 h1 = fast_chirp_value(p, cc0, kn - Nd);
      const float2 w = unit_root((unsigned long long)(k0i + m * (p.N / R)), log2N2);
      const float er = v[m].re.x, ei = v[m].im.x, orr = v[m].re.y, oi = v[m].im.y;
      const float tr = w.x * orr - w.y * oi, ti = w.x * oi + w.y * orr;
      const float x0r = er + tr, x0i = ei + ti, x1r = er - tr, x1i = ei - ti;
      const float y0r = x0r * h0.x - x0i * h0.y, y0i = x0r * h0.y + x0i * h0.x;
      const float y1r = x1r * h1.x - x1i * h1.y, y1i = x1r * h1.y + x1i * h1.x;
      const float dr = y0r - y1r, di = y0i - y1i;
      v[m].re = make_float2(y0r + y1r, w.x * dr + w.y * di);
      v[m].im = make_float2(y0i + y1i, w.x * di - w.y * dr);
    }
    return;
  }
#pragma unroll
  for (int m = 0; m < R; ++m) {
    const double cm = (double)m / R - (m >= R / 2 ? 1.0 : 0.0);
    const double ks = fma(cm, Nd, k0);
    const float2 h0 = fast_chirp_value(p, cc0, ks);
    if (TWOCH) {
      const float2 h1 = fast_chirp_value(p, cc1, ks);
      v[m] = cmul(v[m], make_float2(h0.x, h1.x), make_float2(h0.y, h1.y));
    } else {
      v[m] = cmul(v[m], p_bc(h0.x), p_bc(h0.y));
    }
  }
}

// ------------------------------------------------------------------------------------------
// stages
// ------------------------------------------------------------------------------------------
// first forward stage: global -> registers -> smem (DIF, stage table 0)
template <class C, int LOADK, bool SIGNINV = false>
__device__ __forceinline__ void fwd_first(const FastTile& T, float4* tile, const float2* tws,
                                          int tid, unsigned rowbytes_in) {
  constexpr int R = C::radix(0), S = C::stride(0);
  constexpr int TASKS = S * C::PW;
  constexpr int ITERS = (TASKS + C::NT - 1) / C::NT;
  const int pr = tid & (C::PW - 1);
#pragma unroll
  for (int it = 0; it < ITERS; ++it) {
    const int tau = tid + it * C::NT;
    if (TASKS % C::NT != 0 && tau >= TASKS) break;
    const int b = tau >> C::LOG2PW;
    c2 v[R];
#pragma unroll
    for (int i = 0; i < R; ++i) v[i] = fast_load<LOADK>(T, (unsigned)(b + i * S), rowbytes_in);
    Butterfly<R, SIGNINV>::run(v);
    stage_twiddle<R, S, SIGNINV>(v, tws + C::tw_off(0), b);
#pragma unroll
    for (int i = 0; i < R; ++i) sts_c2(tile, (phys_pt<C, S>(b, i) << C::LOG2PW) + pr, v[i]);
  }
}

// first stage of a tile whose lane pairs each own a CONTIGUOUS run of L rows in global memory
// while the pairs are far apart (ISTFT input, misc.py:81-86): the tile is copied in with
// consecutive threads on consecutive rows, transposed through shared memory, then the stage runs
// from there.  `fxor` is the ifftshift (row index xor) of the reference's np.fft.ifftshift.
// PLANAR: the input is the pair-planar scratch array and pair q of the tile starts pair_bytes * q
// after pair 0 (lane rows of the last level, see LK_TRANSP_PLANAR)
template <class C, bool SIGNINV, bool PLANAR = false>
__device__ __forceinline__ void fwd_first_transposed(const PassArgs& p, const char* gin_tile,
                                                     float4* tile, const float2* tws, int tid,
                                                     unsigned rowbytes_in,
                                                     long long pair_bytes = 0) {
  constexpr int R = C::radix(0), S = C::stride(0);
  constexpr int TASKS = S * C::PW;
  static_assert(TASKS % C::NT == 0, "whole first-stage tasks per thread");
  constexpr int ITERS = TASKS / C::NT;
  const int pr = tid & (C::PW - 1);
  // all of a thread's loads are issued before the first store to shared memory (16 x 16 bytes in
  // flight per thread: the pass only reads, and with a load -> store -> load chain ncu showed it
  // waiting on the long scoreboard 3.8 warp-cycles per issue at 34 % of DRAM peak)
  static_assert((C::PW * C::L) % C::NT == 0, "whole copy rounds per thread");
  constexpr int NLD = C::PW * C::L / C::NT;
  constexpr int BATCH = NLD < 16 ? NLD : 16;
  static_assert(NLD % BATCH == 0, "whole batches");
#pragma unroll 1
  for (int u0 = 0; u0 < NLD; u0 += BATCH) {
    float4 stage[BATCH];
#pragma unroll
    for (int u = 0; u < BATCH; ++u) {
      const int j = tid + (u0 + u) * C::NT;
      const int pair = j >> C::LOG2L, kk = j & (C::L - 1);
      const int cp = 2 * pair;
      const long long po = PLANAR ? pair * pair_bytes
                                  : ((long long)(cp / p.P) * p.min.a_c + (cp % p.P) * p.min.a_p) * 8;
      stage[u] = __ldcg(reinterpret_cast<const float4*>(gin_tile + po +
                                                        (unsigned long long)kk * rowbytes_in));
    }
#pragma unroll
    for (int u = 0; u < BATCH; ++u) {
      const int j = tid + (u0 + u) * C::NT;
      const int pair = j >> C::LOG2L, kk = j & (C::L - 1);
      tile[pair * C::L + (kk ^ (pair & 7))] = stage[u];
    }
  }
  __syncthreads();
  c2 v[ITERS][R];
#pragma unroll
  for (int it = 0; it < ITERS; ++it) {
    const int b = (tid + it * C::NT) >> C::LOG2PW;
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const int row = (b + i * S) ^ p.fxor;
      const float4 t = tile[pr * C::L + (row ^ (pr & 7))];
      if (PLANAR) {
        v[it][i].re = make_float2(t.x, t.y);
        v[it][i].im = make_float2(t.z, t.w);
      } else {
        v[it][i].re = make_float2(t.x, t.z);
        v[it][i].im = make_float2(t.y, t.w);
      }
    }
  }
  __syncthreads();   // every thread holds its inputs: the tile buffer can take the stage output
#pragma unroll
  for (int it = 0; it < ITERS; ++it) {
    const int b = (tid + it * C::NT) >> C::LOG2PW;
    Butterfly<R, SIGNINV>::run(v[it]);
    stage_twiddle<R, S, SIGNINV>(v[it], tws + C::tw_off(0), b);
#pragma unroll
    for (int i = 0; i < R; ++i) sts_c2(tile, (phys_pt<C, S>(b, i) << C::LOG2PW) + pr, v[it][i]);
  }
}

// generic middle stage smem -> smem
template <class C, int J, bool DIT, bool SIGNINV>
__device__ __forceinline__ void mid_stage(float4* tile, const float2* tws, int tid) {
  constexpr int R = C::radix(J), S = C::stride(J);
  constexpr int TASKS = (C::L / R) * C::PW;
  constexpr int ITERS = (TASKS + C::NT - 1) / C::NT;
  const int pr = tid & (C::PW - 1);
#pragma unroll
  for (int it = 0; it < ITERS; ++it) {
    const int tau = tid + it * C::NT;
    if (TASKS % C::NT != 0 && tau >= TASKS) break;
    const int b = tau >> C::LOG2PW;
    const int q = b & (S - 1);
    const int base = (b / S) * (R * S) + q;
    c2 v[R];
#pragma unroll
    for (int i = 0; i < R; ++i) v[i] = lds_c2(tile, (phys_pt<C, S>(base, i) << C::LOG2PW) + pr);
    if (DIT) {
      stage_twiddle<R, S, true>(v, tws + C::tw_off(J), q);
      Butterfly<R, true>::run(v);
    } else {
      Butterfly<R, SIGNINV>::run(v);
      stage_twiddle<R, S, SIGNINV>(v, tws + C::tw_off(J), q);
    }
#pragma unroll
    for (int i = 0; i < R; ++i) sts_c2(tile, (phys_pt<C, S>(base, i) << C::LOG2PW) + pr, v[i]);
  }
}

// barrier of the threads that share a tile: the whole CTA here, a named barrier of one thread
// group in the TMA-pipelined kernel (pbk_tma.cuh)
struct CtaSync {
  __device__ __forceinline__ void operator()() const { __syncthreads(); }
};

template <class C, bool DIT, bool SIGNINV, class Sync = CtaSync>
__device__ __forceinline__ void mid_stages(float4* tile, const float2* tws, int tid,
                                           Sync sync = Sync()) {
  // forward order 1..NS-2, inverse order NS-2..1
  if constexpr (!DIT) {
    if constexpr (C::NS > 2) { mid_stage<C, 1, false, SIGNINV>(tile, tws, tid); sync(); }
    if constexpr (C::NS > 3) { mid_stage<C, 2, false, SIGNINV>(tile, tws, tid); sync(); }
  } else {
    if constexpr (C::NS > 3) { mid_stage<C, 2, true, false>(tile, tws, tid); sync(); }
    if constexpr (C::NS > 2) { mid_stage<C, 1, true, false>(tile, tws, tid); sync(); }
  }
}

// index of last-stage register i of block b (float4 index)
template <class C>
__device__ __forceinline__ int last_idx(int b, int i, int pr) {
  const int sw = C::PPB > 1 ? (b & (C::PPB - 1)) : 0;
  return ((b * C::RL + (i ^ sw)) << C::LOG2PW) + pr;
}

// last inverse stage: smem -> registers -> epilogue (mirror of fwd_first)
template <class C, int EPI>
__device__ __forceinline__ void inv_last(const FastTile& T, float4* tile, const float2* tws,
                                         int tid, unsigned rowbytes_out) {
  constexpr int R = C::radix(0), S = C::stride(0);
  constexpr int TASKS = S * C::PW;
  constexpr int ITERS = (TASKS + C::NT - 1) / C::NT;
  const int pr = tid & (C::PW - 1);
#pragma unroll
  for (int it = 0; it < ITERS; ++it) {
    const int tau = tid + it * C::NT;
    if (TASKS % C::NT != 0 && tau >= TASKS) break;
    const int b = tau >> C::LOG2PW;
    c2 v[R];
#pragma unroll
    for (int i = 0; i < R; ++i) v[i] = lds_c2(tile, (phys_pt<C, S>(b, i) << C::LOG2PW) + pr);
    stage_twiddle<R, S, true>(v, tws + C::tw_off(0), b);
    Butterfly<R, true>::run(v);
#pragma unroll
    for (int i = 0; i < R; ++i) fast_store_out<EPI>(T, (unsigned)(b + i * S), rowbytes_out, v[i]);
  }
}

// last inverse stage of a TSUM pass: the detected power of every surviving row is added to the
// thread's running sums instead of being stored (one accumulator per tile row the thread owns;
// consecutive tiles of a TSUM CTA are consecutive time offsets of the same columns)
template <class C, int EPI>
struct TsumAcc {
  static constexpr int R = C::radix(0);
  static constexpr int ITERS = (C::stride(0) * C::PW + C::NT - 1) / C::NT;
  using acc_t = typename std::conditional<EPI == EPI_STOKES_I, float, float2>::type;
  acc_t a[ITERS][R];
  __device__ __forceinline__ void clear() {
#pragma unroll
    for (int it = 0; it < ITERS; ++it)
#pragma unroll
      for (int i = 0; i < R; ++i) {
        if constexpr (EPI == EPI_STOKES_I) a[it][i] = 0.f;
        else a[it][i] = make_float2(0.f, 0.f);
      }
  }
};

template <class C, int EPI>
__device__ __forceinline__ void inv_last_sum(const FastTile& T, float4* tile, const float2* tws,
                                             int tid, TsumAcc<C, EPI>& acc) {
  constexpr int R = C::radix(0), S = C::stride(0);
  constexpr int TASKS = S * C::PW;
  static_assert(TASKS % C::NT == 0, "whole last-stage tasks per thread");
  constexpr int ITERS = TASKS / C::NT;
  const int pr = tid & (C::PW - 1);
#pragma unroll
  for (int it = 0; it < ITERS; ++it) {
    const int b = (tid + it * C::NT) >> C::LOG2PW;
    c2 v[R];
#pragma unroll
    for (int i = 0; i < R; ++i) v[i] = lds_c2(tile, (phys_pt<C, S>(b, i) << C::LOG2PW) + pr);
    stage_twiddle<R, S, true>(v, tws + C::tw_off(0), b);
    Butterfly<R, true>::run(v);
#pragma unroll
    for (int i = 0; i < R; ++i) {
      if ((unsigned)(b + i * S) - T.row_lo >= T.row_cnt) continue;
      if constexpr (EPI == EPI_STOKES_I) {
        float s = acc.a[it][i];
        s = fmaf(v[i].re.x, v[i].re.x, s);
        s = fmaf(v[i].im.x, v[i].im.x, s);
        s = fmaf(v[i].re.y, v[i].re.y, s);
        s = fmaf(v[i].im.y, v[i].im.y, s);
        acc.a[it][i] = s;
      } else {
        acc.a[it][i] = p_fma(v[i].re, v[i].re, p_fma(v[i].im, v[i].im, acc.a[it][i]));
      }
    }
  }
}

// adds the running sums of a finished (or interrupted) group of 2^tsum_log2 time rows to the output.
// `colbase` points at this thread's column(s) in output row 0; tile row r at inner offset nrest is
// time n = (r << log2nmul) + nrest and lands in output row (n - crop_start) >> tsum_log2.  A group
// receives at most two contributions (a CTA's run of tiles is at least two groups long and run
// boundaries avoid the groups that straddle the wrap of the inner offset), so the float atomics
// give the same result in either order.  With p.tsum_bins (the fold) the row is tsum_bins[row] and
// a profile row collects the groups of every row in its phase bin in any order: reproducible to
// rounding, not bit for bit.  Only sums of rows inside the crop are non-zero, so the bin array is
// read for rows [0, out_rows) only.
__device__ __forceinline__ char* tsum_row(const PassArgs& p, char* colbase, long long n,
                                          long long out_row_bytes) {
  const long long row = (n - p.crop_start) >> p.tsum_log2;
  return colbase + (p.tsum_bins ? (long long)p.tsum_bins[row] : row) * out_row_bytes;
}

template <class C, int EPI>
__device__ __forceinline__ void tsum_flush(const PassArgs& p, TsumAcc<C, EPI>& acc, char* colbase,
                                           unsigned nrest, int tid, long long out_row_bytes) {
  constexpr int R = C::radix(0), S = C::stride(0);
#pragma unroll
  for (int it = 0; it < TsumAcc<C, EPI>::ITERS; ++it) {
    const int b = (tid + it * C::NT) >> C::LOG2PW;
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const long long n = ((long long)(b + i * S) << p.log2nmul) + nrest;
      if constexpr (EPI == EPI_STOKES_I) {
        if (acc.a[it][i] != 0.f)
          atomicAdd(reinterpret_cast<float*>(tsum_row(p, colbase, n, out_row_bytes)), acc.a[it][i]);
      } else {
        const float2 v = acc.a[it][i];
        if (v.x != 0.f || v.y != 0.f) {
          float* a = reinterpret_cast<float*>(tsum_row(p, colbase, n, out_row_bytes));
          if (v.x != 0.f) atomicAdd(a, v.x);
          if (v.y != 0.f) atomicAdd(a + 1, v.y);
        }
      }
    }
  }
  acc.clear();
}

// ------------------------------------------------------------------------------------------
// kernel
// ------------------------------------------------------------------------------------------
// TSUM (final INV pass with a detected output and a time sum, row R of SURVEY 8a): a CTA owns a
// CONTIGUOUS run of tiles ordered (column group, inner time offset), keeps the power sums of the
// current group of 2^tsum_log2 consecutive time rows in registers and adds them to the (zeroed)
// output when the group ends -- the full-resolution intensity array never exists.
template <int MODE, class C, int LOADK, int EPI, bool TWOCH = false, bool NARROW = false,
          bool SIGNINV = false, bool TSUM = false>
__global__ void __launch_bounds__(C::NT, C::MINB)
fast_pass_kernel(const __grid_constant__ PassArgs p, const float2* __restrict__ tables,
                 long long ntiles) {
  static_assert(C::NS >= 2, "fast kernel needs at least two stages");
  extern __shared__ float4 smem_dyn[];
  float4* tile = smem_dyn;
  float2* tws = reinterpret_cast<float2*>(tile + (size_t)C::L * C::PW);
  float4* G4 = reinterpret_cast<float4*>(tws + C::TW_PAD);
  TileInfo* sinfo = reinterpret_cast<TileInfo*>(G4 + C::RL * (NARROW ? C::G_ROWS : 1));
  const int tid = threadIdx.x;
  const int pr = tid & (C::PW - 1);

  constexpr int in_bits = lk_bits(LOADK);   // BITS per complex input element
  constexpr int out_eb = (EPI == EPI_INTENSITY || EPI == EPI_STOKES_I) ? 4 : 8;
  const unsigned rb_in = (unsigned)((p.min.a_row * in_bits) >> 3);
  const unsigned rb_out = (unsigned)(p.mout.a_row * out_eb);

  static_assert(!TSUM || (MODE == MODE_INV && !NARROW &&
                          (EPI == EPI_INTENSITY || EPI == EPI_STOKES_I)), "TSUM is a final INV pass");
  // iteration space: plain passes stride over tiles by the grid.  TSUM passes: q = tsum_q adjacent
  // CTAs share a contiguous run of (column-group block, inner time offset) and take one column
  // group of the block each, so that together they read whole rows (DRAM page locality)
  const int ncg = TSUM ? p.I / C::W : 1;
  const int tq = TSUM ? p.tsum_q : 1;
  const int cgq = TSUM ? (int)(blockIdx.x % tq) : 0;
  // FSUM (FWD-last pass with a detected, frequency-summed output): G = 2^fsum_g_log2 consecutive
  // tiles are the consecutive groups of first-level bins that land in the same output cells; a CTA
  // takes whole groups of G tiles (iteration i -> tile (blockIdx + (i / G) grid) G + i % G), keeps
  // the power sums in registers and stores them once per group: deterministic, no atomics.
  constexpr bool FSUM = MODE == MODE_FWD && (EPI == EPI_INTENSITY || EPI == EPI_STOKES_I);
  static_assert(!FSUM || NARROW, "the detected channelizer epilogue is built for few-lane arrays");
  const int fs_g = FSUM ? p.fsum_g_log2 : 0;
  auto fs_tile_at = [&](long long i) -> long long {
    return ((blockIdx.x + (i >> fs_g) * (long long)gridDim.x) << fs_g) + (i & ((1ll << fs_g) - 1));
  };
  const long long fs_groups = FSUM ? ntiles >> fs_g : 0;
  const long long fs_iters = FSUM && blockIdx.x < fs_groups
      ? ((fs_groups - blockIdx.x + gridDim.x - 1) / gridDim.x) << fs_g : 0;
  auto tile_at = [&](long long i) -> long long {
    if (FSUM) return fs_tile_at(i);
    if (!TSUM) return i;
    const long long cb = i >> p.log2nmul, nr = i & ((1ll << p.log2nmul) - 1);
    return nr * ncg + cb * tq + cgq;
  };
  const long long ts_total = TSUM ? ntiles / tq : 0;              // runs are split over grid / q
  const long long ts_r = TSUM ? blockIdx.x / tq : 0, ts_nr = TSUM ? gridDim.x / tq : 1;
  // Groups of summed rows start where (inner offset - crop_start) is a multiple of M.  When
  // crop_start is not, the first and last group of a walk over the inner offsets are the two
  // halves of groups that straddle the wrap; a run boundary inside them would give such a group
  // a third contribution, so it is moved to the edge of the partial group.
  const unsigned ts_off = TSUM ? (unsigned)(p.crop_start & ((1ll << p.tsum_log2) - 1)) : 0u;
  auto ts_snap = [&](long long u) -> long long {
    if (!TSUM || ts_off == 0) return u;
    const long long nr = u & ((1ll << p.log2nmul) - 1);
    const long long tail = (1ll << p.log2nmul) - ((1ll << p.tsum_log2) - ts_off);
    if (nr > 0 && nr < ts_off) return u - nr + ts_off;
    if (nr > tail) return u - nr + tail;
    return u;
  };
  long long t = TSUM ? ts_snap(ts_total * ts_r / ts_nr) : FSUM ? 0 : p.tile0 + blockIdx.x;
  const long long t_end = TSUM ? ts_snap(ts_total * (ts_r + 1) / ts_nr) : FSUM ? fs_iters : ntiles;
  const long long t_step = (TSUM || FSUM) ? 1 : gridDim.x;
  pdl_trigger();
  for (int i = tid; i < C::TW_TOTAL; i += C::NT) tws[i] = tables[i];
  // Batched launches offset each tile by the batch index (trial plans batch the MID and INV
  // passes, overlap-save blocks every pass).  In FWD kernels thread 0 adds the offsets to the tile
  // record: added to every thread's pointers, they spill 16 bytes in the 256-point FWD kernels at
  // the 128-register cap.  MID and INV kernels add them to the pointers (below), which spills less
  // there than the record does.
  auto tile_info = [&](long long tile) {
    fast_tile_info<C, EPI>(p, tile, *sinfo, in_bits, out_eb);
    if constexpr (MODE == MODE_FWD) {
      sinfo->bi += trial_y() * p.trial_in_bytes;
      sinfo->bo += trial_y() * p.trial_out_bytes;
    }
  };
  if (tid == 0 && t < t_end) tile_info(tile_at(t));
  __syncthreads();
  pdl_wait();   // the previous pass's output (and the array this pass overwrites) from here on

  // Per-thread part of the addresses.  A tile is W adjacent lanes; a lane is (row jr, column) of
  // the (.., I) array.  Normally (I a multiple of W) the tile sits inside one row (jr = 0, col0 a
  // multiple of P).  NARROW kernels serve arrays with few channels (I < W): the tile then spans
  // nrows = W / I consecutive rows -- consecutive inner time offsets for the strided levels,
  // consecutive kprev blocks for the MID level -- and everything row-dependent is per thread.
  const int nrows = NARROW ? C::W / p.I : 1;
  const int jr = NARROW ? (2 * pr) / p.I : 0;
  const int colt = NARROW ? (2 * pr) % p.I : 2 * pr;
  // FWDLAST: the last pass of a plain forward FFT / STFT (no inter-level twiddle; scaled,
  // optionally fftshift-ed, natural-order complex64 written to the user's array)
  constexpr bool FWDLAST = MODE == MODE_FWD && EPI != EPI_SCRATCH;
  constexpr bool LASTLEVEL = MODE == MODE_MID || FWDLAST;   // rows of lanes are kprev blocks
  const long long row_in = LASTLEVEL ? p.min.a_kp : p.min.a_n;
  const long long row_out = LASTLEVEL ? p.mout.a_kp : p.mout.a_n;
  const long long off_in =
      ((jr * row_in + (long long)(colt / p.P) * p.min.a_c + (colt % p.P) * p.min.a_p) * in_bits) >> 3;
  const long long off_out =
      (jr * row_out + (long long)(colt / p.P) * p.mout.a_c + (colt % p.P) * p.mout.a_p) * out_eb;
  const int chant = colt / p.P;
  constexpr int GS = NARROW ? C::G_ROWS : 1;   // level-twiddle tables: [m][lane row]
  const float4* G4t = G4 + jr;                 // this thread's lane row

  constexpr int RL = C::RL;
  constexpr int LTASKS = (C::L / RL) * C::PW;
  constexpr int LITERS = (LTASKS + C::NT - 1) / C::NT;

  float2 fs_acc[FSUM ? ((C::L / C::RL) * C::PW + C::NT - 1) / C::NT * C::RL : 1];
  TsumAcc<C, TSUM ? EPI : EPI_STOKES_I> tacc;
  char* ts_colbase = nullptr;   // TSUM: output columns and inner offset of the running sums
  unsigned ts_nrest = 0;
  const long long ts_rowbytes = p.mout.a_n * out_eb;
  if (TSUM) tacc.clear();

  for (; t < t_end; t += t_step) {
    FastTile T;
    unsigned nrest0;
    {
      const TileInfo ti = *sinfo;
      T.gin = reinterpret_cast<const char*>(p.in) + ti.bi + off_in;
      T.gout = reinterpret_cast<char*>(p.out) + ti.bo + off_out;
      if constexpr (MODE != MODE_FWD) {   // (FWD: in the tile record, see tile_info)
        T.gin += trial_y() * p.trial_in_bytes;
        T.gout += trial_y() * p.trial_out_bytes;
      }
      if constexpr (TSUM) {
        // ti.bo = (nrest - crop_start) rows + the column offset; keep the column part only
        char* colbase = T.gout - ((long long)ti.nrest - p.crop_start) * ts_rowbytes;
        if (ts_colbase != nullptr &&
            (colbase != ts_colbase || ((ti.nrest - ts_off) & ((1u << p.tsum_log2) - 1)) == 0))
          tsum_flush<C, EPI>(p, tacc, ts_colbase, ts_nrest, tid, ts_rowbytes);
        ts_colbase = colbase;
        ts_nrest = ti.nrest;
      }
      nrest0 = ti.nrest;
      T.nrest = ti.nrest + (LASTLEVEL ? 0 : jr);
      if (LASTLEVEL && NARROW) {
        const unsigned kprev = ti.kprev + jr;
        T.klow = (kprev >> p.kl_sa) + ((kprev & p.kl_mb) << p.kl_sb);
        if (FWDLAST)   // natural-order output: the low part of the frequency index is per lane row
          T.gout += ((long long)T.klow - (long long)ti.klow) * p.mout.a_kl * out_eb;
      } else {
        T.klow = ti.klow;
      }
      T.chan = ti.chan0 + chant;
      T.row_lo = ti.row_lo;
      T.row_cnt = ti.row_cnt;
      if (EPI != EPI_SCRATCH && NARROW && !FWDLAST) {   // the crop row range depends on the lane's row
        const long long add = (1ll << p.log2nmul) - 1;
        long long lo = (p.crop_start - (long long)T.nrest + add) >> p.log2nmul;
        long long hi = (p.crop_stop - (long long)T.nrest + add) >> p.log2nmul;
        lo = lo < 0 ? 0 : lo;
        hi = hi > C::L ? C::L : hi;
        T.row_lo = (unsigned)lo;
        T.row_cnt = hi > lo ? (unsigned)(hi - lo) : 0u;
      }
    }
    if (MODE != MODE_MID && !FWDLAST) {
      if (NARROW) {
        for (int i = tid; i < RL * nrows; i += C::NT) {
          const int j = i / RL, m = i - j * RL;
          const float2 g =
              unit_root((unsigned long long)(nrest0 + j) * (unsigned)(C::KS * m), p.log2M);
          G4[m * C::G_ROWS + j] = make_float4(g.x, g.y, g.y, g.x);
        }
      } else if (tid < RL) {
        const float2 g = unit_root((unsigned long long)nrest0 * (unsigned)(C::KS * tid), p.log2M);
        G4[tid] = make_float4(g.x, g.y, g.y, g.x);
      }
    }
    if (MODE == MODE_INV) __syncthreads();  // INV consumes G in its first phase
    // every thread has copied *sinfo by the first barrier of this tile; thread 0 then prepares
    // the next tile's record, which the end-of-tile barrier publishes
#define PBK_NEXT_TILE_INFO()                                                        \
  if (tid == 0 && t + t_step < t_end)                                               \
    tile_info(tile_at(t + t_step))
    if (MODE == MODE_INV) PBK_NEXT_TILE_INFO();

    if (MODE == MODE_FWD) {
      if constexpr (LOADK == LK_TRANSP)
        fwd_first_transposed<C, SIGNINV>(p, T.gin - off_in, tile, tws, tid, rb_in);
      else if constexpr (LOADK == LK_TRANSP_PLANAR)
        fwd_first_transposed<C, SIGNINV, true>(p, T.gin - off_in, tile, tws, tid, rb_in,
                                               row_in * 8);
      else
        fwd_first<C, LOADK, SIGNINV>(T, tile, tws, tid, rb_in);
      __syncthreads();
      PBK_NEXT_TILE_INFO();
      mid_stages<C, false, SIGNINV>(tile, tws, tid);
      if constexpr (!FWDLAST) {
#pragma unroll
        for (int it = 0; it < LITERS; ++it) {
          const int tau = tid + it * C::NT;
          if (LTASKS % C::NT != 0 && tau >= LTASKS) break;
          const int b = tau >> C::LOG2PW;
          c2 v[RL];
#pragma unroll
          for (int i = 0; i < RL; ++i) v[i] = lds_c2(tile, last_idx<C>(b, i, pr));
          Butterfly<RL, SIGNINV>::run(v);
          const int klo = klo_of<C>(b);
          level_twiddle<RL, SIGNINV, GS>(p, v, T.nrest, (unsigned)klo, G4t);
#pragma unroll
          for (int i = 0; i < RL; ++i) fast_store_c64(T, (unsigned)(klo + i * C::KS), rb_out, v[i]);
        }
      } else {
        // last pass of a forward FFT / STFT: no level twiddle; scale, fftshift (row xor) and
        // natural-order complex64 to the user's array
        static_assert(!FWDLAST || LTASKS % C::NT == 0, "whole last-stage tasks per thread");
        c2 v[LITERS][RL];
        int klo[LITERS];
        const float2 sc = p_bc(p.scale);
#pragma unroll
        for (int it = 0; it < LITERS; ++it) {
          const int b = (tid + it * C::NT) >> C::LOG2PW;
#pragma unroll
          for (int i = 0; i < RL; ++i) v[it][i] = lds_c2(tile, last_idx<C>(b, i, pr));
          Butterfly<RL, SIGNINV>::run(v[it]);
          klo[it] = klo_of<C>(b);
#pragma unroll
          for (int i = 0; i < RL; ++i) {
            v[it][i].re = p_mul(v[it][i].re, sc);
            v[it][i].im = p_mul(v[it][i].im, sc);
          }
        }
        if constexpr (FSUM) {
          // detected output: |z|^2 of every register, summed over the G tiles of a group (registers),
          // then over the lane rows of the tile (the 16 threads of a half-warp hold 16 adjacent
          // first-level bins), stored by one lane per row.  p.I == 2: the pair is (pol 0, pol 1)
          // of the one channel, or the (even, odd) samples of a single-pol column (fsum_split).
          static_assert(LITERS * RL <= 32, "power sums stay in registers");
          if ((t & ((1ll << fs_g) - 1)) == 0) {
#pragma unroll
            for (int q = 0; q < LITERS * RL; ++q) fs_acc[q] = make_float2(0.f, 0.f);
          }
#pragma unroll
          for (int it = 0; it < LITERS; ++it)
#pragma unroll
            for (int i = 0; i < RL; ++i) {
              c2 z = v[it][i];
              if (p.fsum_split) {
                // half-length spectra E (lane 0), O (lane 1) at bin k = klow + Kprev * row
                const unsigned long long k =
                    (unsigned long long)T.klow + ((unsigned long long)(klo[it] + i * C::KS) << p.log2Kmul);
                const float2 w = unit_root(k, p.fsum_log2n);      // exp(-2 pi i k / n), n = 2 * half
                const float tr = w.x * z.re.y - w.y * z.im.y, ti2 = w.x * z.im.y + w.y * z.re.y;
                z.re = make_float2(z.re.x + tr, z.re.x - tr);     // X[k], X[k + n/2]
                z.im = make_float2(z.im.x + ti2, z.im.x - ti2);
              }
              fs_acc[it * RL + i] = p_fma(z.re, z.re, p_fma(z.im, z.im, fs_acc[it * RL + i]));
            }
          if ((t & ((1ll << fs_g) - 1)) == (1ll << fs_g) - 1) {
            // lane rows of a tile: pr (nrows == PW when I == 2); reduce over them
            float* outf = reinterpret_cast<float*>(T.gout);       // this segment's output row
            const bool folded = p.fsum_bins != nullptr;
            if (folded) {   // row of the segment's phase bin in the profile; sums are added to it
              const long long rowf = p.fsum_cells * p.fsum_pq;
              const long long seg = (outf - reinterpret_cast<float*>(p.out)) / rowf;
              outf = reinterpret_cast<float*>(p.out) + (long long)p.fsum_bins[seg] * rowf;
            }
            const unsigned kp_cell = (unsigned)(T.klow >> p.fsum_log2);   // same for the whole group
#pragma unroll
            for (int it = 0; it < LITERS; ++it)
#pragma unroll
              for (int i = 0; i < RL; ++i) {
                float2 a = fs_acc[it * RL + i];
#pragma unroll
                for (int sft = 1; sft < C::PW; sft <<= 1) {
                  a.x += __shfl_xor_sync(0xffffffffu, a.x, sft);
                  a.y += __shfl_xor_sync(0xffffffffu, a.y, sft);
                }
                if ((i & (C::PW - 1)) == pr) {     // spread the stores over the lanes
                  const unsigned row = (unsigned)(klo[it] + i * C::KS);
                  if (p.fsum_split) {
                    // fftshift of the full length: bin k lands at k + n/2, bin k + n/2 at k
                    const unsigned cell = (row << p.fsum_row_shift) + kp_cell;
                    const unsigned half = 1u << (p.log2L + p.fsum_row_shift);   // (n/2) / F
                    if (folded) {
                      atomicAdd(outf + cell + half, a.x);
                      atomicAdd(outf + cell, a.y);
                    } else {
                      outf[cell + half] = a.x;
                      outf[cell] = a.y;
                    }
                  } else {
                    const unsigned cell = ((row ^ (unsigned)p.kxor) << p.fsum_row_shift) + kp_cell;
                    if (folded) {
                      if (p.fsum_pq == 2) {
                        atomicAdd(outf + 2 * cell, a.x);
                        atomicAdd(outf + 2 * cell + 1, a.y);
                      } else {
                        atomicAdd(outf + cell, a.x + a.y);
                      }
                    } else if (p.fsum_pq == 2) {
                      *reinterpret_cast<float2*>(outf + 2 * cell) = a;
                    } else {
                      outf[cell] = a.x + a.y;
                    }
                  }
                }
              }
          }
        } else if (NARROW && p.fsum_split) {
          // plain channelizer of ONE single-pol column run as its (even, odd) samples at half
          // length: the pair holds E[k], O[k] at bin k = klow + Kprev * row; X[k] = E + wO goes to
          // slot k + n/2 of the fftshift-ed segment, X[k + n/2] = E - wO to slot k (misc.py:48).
          // The 16 lane rows of a tile are adjacent klow: 128-byte runs per store instruction.
          float2* seg = reinterpret_cast<float2*>(T.gout);
          const unsigned long long halfn = 1ull << (p.fsum_log2n - 1);
#pragma unroll
          for (int it = 0; it < LITERS; ++it)
#pragma unroll
            for (int i = 0; i < RL; ++i) {
              const c2 z = v[it][i];
              const unsigned long long k =
                  (unsigned long long)T.klow + ((unsigned long long)(klo[it] + i * C::KS) << p.log2Kmul);
              const float2 w = unit_root(k, p.fsum_log2n);        // exp(-2 pi i k / n)
              const float tr = w.x * z.re.y - w.y * z.im.y, ti2 = w.x * z.im.y + w.y * z.re.y;
              seg[k + halfn] = make_float2(z.re.x + tr, z.im.x + ti2);
              seg[k] = make_float2(z.re.x - tr, z.im.x - ti2);
            }
        } else if (!p.out_transpose) {
          // output lanes are adjacent in memory: one natural-order 16-byte store per row
#pragma unroll
          for (int it = 0; it < LITERS; ++it)
#pragma unroll
            for (int i = 0; i < RL; ++i) {
              const unsigned row = (unsigned)(klo[it] + i * C::KS) ^ (unsigned)p.kxor;
              *reinterpret_cast<float4*>(T.gout + (unsigned long long)row * rb_out) =
                  make_float4(v[it][i].re.x, v[it][i].im.x, v[it][i].re.y, v[it][i].im.y);
            }
        } else {
          // STFT output (misc.py:50): every lane pair owns a CONTIGUOUS run of L rows and the
          // pairs are far apart, so the tile is transposed through shared memory and copied out
          // with consecutive threads on consecutive rows
          __syncthreads();                       // all last-stage reads of the tile are done
#pragma unroll
          for (int it = 0; it < LITERS; ++it)
#pragma unroll
            for (int i = 0; i < RL; ++i) {
              const int k = (klo[it] + i * C::KS) ^ p.kxor;
              tile[pr * C::L + (k ^ (pr & 7))] =
                  make_float4(v[it][i].re.x, v[it][i].im.x, v[it][i].re.y, v[it][i].im.y);
            }
          __syncthreads();
          char* gt = T.gout - off_out;           // tile base (lane pair 0)
          for (int j = tid; j < C::PW * C::L; j += C::NT) {
            const int pair = j >> C::LOG2L, kk = j & (C::L - 1);
            const int cp = 2 * pair;
            const long long po =
                ((long long)(cp / p.P) * p.mout.a_c + (cp % p.P) * p.mout.a_p) * out_eb;
            *reinterpret_cast<float4*>(gt + po + (unsigned long long)kk * rb_out) =
                tile[pair * C::L + (kk ^ (pair & 7))];
          }
        }
      }
    } else if (MODE == MODE_MID) {
      fwd_first<C, LOADK>(T, tile, tws, tid, rb_in);
      __syncthreads();
      PBK_NEXT_TILE_INFO();
      mid_stages<C, false, false>(tile, tws, tid);
#pragma unroll
      for (int it = 0; it < LITERS; ++it) {
        const int tau = tid + it * C::NT;
        if (LTASKS % C::NT != 0 && tau >= LTASKS) break;
        const int b = tau >> C::LOG2PW;
        c2 v[RL];
#pragma unroll
        for (int i = 0; i < RL; ++i) v[i] = lds_c2(tile, last_idx<C>(b, i, pr));
        Butterfly<RL, false>::run(v);
        fast_chirp<RL, C, TWOCH>(p, T, v, klo_of<C>(b));
        Butterfly<RL, true>::run(v);
#pragma unroll
        for (int i = 0; i < RL; ++i) sts_c2(tile, last_idx<C>(b, i, pr), v[i]);
      }
      __syncthreads();
      mid_stages<C, true, false>(tile, tws, tid);
      inv_last<C, EPI>(T, tile, tws, tid, rb_out);
    } else {  // MODE_INV
#pragma unroll
      for (int it = 0; it < LITERS; ++it) {
        const int tau = tid + it * C::NT;
        if (LTASKS % C::NT != 0 && tau >= LTASKS) break;
        const int b = tau >> C::LOG2PW;
        const int klo = klo_of<C>(b);
        c2 v[RL];
#pragma unroll
        for (int i = 0; i < RL; ++i) v[i] = fast_load<LK_PLANAR>(T, (unsigned)(klo + i * C::KS), rb_in);
        level_twiddle<RL, true, GS>(p, v, T.nrest, (unsigned)klo, G4t);
        Butterfly<RL, true>::run(v);
#pragma unroll
        for (int i = 0; i < RL; ++i) sts_c2(tile, last_idx<C>(b, i, pr), v[i]);
      }
      __syncthreads();
      mid_stages<C, true, false>(tile, tws, tid);
      if constexpr (TSUM) inv_last_sum<C, EPI>(T, tile, tws, tid, tacc);
      else inv_last<C, EPI>(T, tile, tws, tid, rb_out);
    }
    __syncthreads();  // tile buffer, G and the tile record are reused by the next tile
  }
  if constexpr (TSUM) {
    if (ts_colbase != nullptr) tsum_flush<C, EPI>(p, tacc, ts_colbase, ts_nrest, tid, ts_rowbytes);
  }
#undef PBK_NEXT_TILE_INFO
}

}  // namespace pbk
