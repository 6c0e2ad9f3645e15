// pbk_fft.cuh -- sm_100a tile-FFT pass kernels for the pulsarbat baseband hot path.
//
// What this replaces in the reference (paths under /root/reference/pulsarbat):
//   transforms/dedispersion.py:125   x = ifft(fft(z.data, axis=0) * chirp, axis=0)
//   transforms/dedispersion.py:19-23 _transfer_function (the chirp; here generated in registers)
//   fft.py:30-48                      pb.fft.fft / ifft (axis-0, batch-innermost c64 transforms)
//   contrib/misc.py:43-52, 81-91      stft / istft (segment FFT + fftshift + scale)
//   core.py:766-774, 944-948          re^2+im^2 and Stokes I (fused into the last inverse pass)
//
// Design (see DESIGN.md):
//  * A length-N transform (N = 2^n) along the slow axis of a (O, N, I) array is split into
//    m levels N = L1*L2*..*Lm.  Level l transforms the index with the largest remaining stride;
//    each CTA owns one tile = L points x W adjacent "lanes" (lanes = flattened (outer, inner)
//    index, adjacent lanes are adjacent in memory), so every global access is a W*8-byte chunk.
//  * Forward levels are decimation-in-frequency (butterfly, then twiddle), the inverse levels
//    are the mirrored decimation-in-time graph (conj twiddle, then butterfly).  Because the
//    graphs are mirrors, nothing is ever reordered: the last forward stage leaves 16 spectral
//    points in registers, the chirp is applied there, and the first inverse stage consumes the
//    same registers.  fft * H * ifft for a tile is ONE kernel (MODE_MID).
//  * Each thread owns a PAIR of adjacent lanes and keeps (re0,re1) and (im0,im1) in aligned
//    64-bit register pairs, so every add/mul/fma is a packed FADD2/FMUL2/FFMA2 (sm_100 needs
//    the packed forms to reach its FP32 rate); twiddles are shared by both lanes when the pair
//    is "uniform" (same inner time offset / same channel), which is the case for pol pairs.
//  * Stages are radix-16 (first stage radix 2/4/8/16 to absorb log2(L) mod 4); between stages
//    the tile lives in shared memory as float4 {re0,re1,im0,im1} with an XOR swizzle that makes
//    every LDS.128/STS.128 conflict-free for all strides.
//  * The chirp phase is evaluated in FP64 in cycles with the cancellation-free form
//    D*((f-fr)/fr)^2/f, reduced mod 1 exactly (phi - rint(phi)), then sincospif in FP32.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

namespace pbk {

enum { MODE_FWD = 0, MODE_MID = 1, MODE_INV = 2 };
enum { LOAD_C64 = 0, LOAD_I8X2 = 1, LOAD_PLANAR = 2, LOAD_F32 = 3 /* real input, im = 0 */,
       LOAD_TRANSP = 4 /* fast kernels only: complex64 input transposed through shared memory */,
       LOAD_U4X2 = 5 /* packed 4+4-bit complex */, LOAD_U2X2 = 6 /* packed 2+2-bit complex */,
       LOAD_TRANSP_PLANAR = 7 /* fast kernels only: scratch input transposed through shared memory */ };

// bits per complex input element of a load kind
__host__ __device__ constexpr int load_bits(int kind) {
  return kind == LOAD_I8X2 ? 16 : kind == LOAD_U4X2 ? 8 : kind == LOAD_U2X2 ? 4
         : kind == LOAD_F32 ? 32 : 64;
}
__host__ __device__ constexpr bool load_is_raw(int kind) {
  return kind == LOAD_I8X2 || kind == LOAD_U4X2 || kind == LOAD_U2X2;
}
enum { EPI_C64 = 0, EPI_INTENSITY = 1, EPI_STOKES_I = 2 };
enum { CHIRP_NONE = 0, CHIRP_COMPUTED = 1, CHIRP_ARRAY = 2, CHIRP_RAMP = 3 };

constexpr int kThreads = 256;
constexpr int kMaxStages = 4;

// Programmatic dependent launch between the passes of a plan: every pass kernel lets the next
// launch of the stream start as soon as all of its own CTAs are running (pdl_trigger, first
// instruction) and waits for the previous kernel of the stream to finish and flush its stores
// (pdl_wait) only after its prologue -- stage tables, tile records, everything that depends on
// constants alone -- so that launch latency, CTA ramp-up and prologue overlap the previous pass's
// tail.  EVERY CTA executes pdl_wait, work or not: a grid completes only after all of its CTAs
// have passed it, which keeps completion transitive along the chain of passes.  Both are no-ops
// for a launch without the attribute (PBK_PDL=0, or the profiler's serialised replay).
__device__ __forceinline__ void pdl_trigger() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

inline bool pdl_enabled() {
  static const bool on = [] {
    const char* e = getenv("PBK_PDL");
    return !(e && e[0] == '0');
  }();
  return on;
}
// launch of a pass kernel (one that executes pdl_wait in every CTA) with the programmatic
// stream-serialisation attribute
template <class... KArgs, class... Args>
inline cudaError_t pdl_launch(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem,
                              cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// element index = o_orig*a_o + kprev*a_kp + klow*a_kl + nrest*a_n + (col / P)*a_c + (col % P)*a_p
//                 + row * a_row
struct AddrMap {
  long long a_o, a_kp, a_kl, a_n, a_c, a_p, a_row;
};

struct PassArgs {
  const void* in;
  void* out;
  AddrMap min, mout;
  long long Q;        // number of lanes = O_level * RI
  long long RI;       // inner extent at this level (R * I)
  int I;              // innermost batch (nchan * npol)
  int P;              // npol (channel = col / P)
  int log2L;          // tile transform length
  int nstages;        // ceil(log2L / 4)
  int log2r1;         // radix of the first stage (others are 16)
  int log2pw;         // lane pairs per tile
  int log2Kprev;      // o = (o_orig << log2Kprev) | kprev
  int kl_sa, kl_mb, kl_sb;  // klow = (kprev >> kl_sa) + ((kprev & kl_mb) << kl_sb)
  int log2M;          // inter-level twiddle modulus (0 = none): W_M^(nrest * k)
  int sign;           // FWD mode only: -1 forward, +1 inverse exponent
  const float2* stage_tw;           // per-stage twiddle tables, (cos, -sin)
  int stage_tw_off[kMaxStages];     // offsets (in float2) of each stage's table
  float scale;        // applied with the chirp (MID) or at the store (FWD)
  int load_kind, epi_kind;
  int fxor, kxor;     // ifftshift on load rows / fftshift on store rows (tile-level index xor)
  long long crop_start, crop_stop, n_mul;   // epilogue: n = row*n_mul + nrest, keep [start,stop)
  int log2nmul;       // n_mul = 2^log2nmul (fast kernels)
  int final_epi;      // this pass writes the user-visible output (crop + epilogue kind apply)
  int store_planar;   // output is the scratch array in pair-planar form {re0,re1,im0,im1}
  int out_transpose;  // fast FWD-last pass: lane pairs own contiguous runs of rows in the output
  // chirp
  int chirp_kind;
  int log2Kmul;       // kfull = klow + (k << log2Kmul)
  long long N;        // full transform length (for fftfreq sign wrap)
  const double* chan_freq;   // Hz, per channel
  const double* chan_const;  // fast MID kernel: {(fc-fr)/fr, df/fc, D/fc} per channel
  double bd;                 // df / fr (0 for fr = inf)
  double df, fr_sub, inv_fr, a0, D;
  const float2* chirp_arr;
  long long chirp_sk, chirp_sc;
  // CHIRP_RAMP: per column, H_k = exp(-2 pi i s k_signed / N) outside the zeroed band
  const double* ramp_shift;     // s / N per column (cycles per bin)
  const long long* ramp_zero;   // [lo, hi) per column in fftshift-ed bin order; lo >= hi = none
  int ramp_hilbert;             // analytic-signal weights 1,2,..,2,1,0,..,0 (utils.py:50-54)
  long long tile0;    // fast kernels: first tile of this launch (tiles [tile0, ntiles) are processed)
  int tsum_log2;      // fast final INV pass: > 0 = sum 2^tsum_log2 consecutive time rows of the
                      // detected output in the epilogue (row R fused; see fast_pass_kernel TSUM)
  int tsum_q;         // ... with groups of tsum_q adjacent CTAs covering adjacent column groups
  const int* tsum_bins;   // fold fused behind the time sum (pbk_dedisp_fold_exec_device): phase bin
                          // of every output row; group sums are ADDED to out[bin] instead of out[row]
  // fast FWD-last pass of a channelizer plan with a DETECTED output (pbk_stft_detect_plan_create):
  // |z|^2 summed over 2^fsum_log2 adjacent fine channels in the epilogue, so the channelized
  // voltages never reach HBM; see pbk_fast.cuh (FSUM).
  int fsum_log2;      // > 0 enables; F = 2^fsum_log2 divides the number of first-level bins Kprev
  int fsum_g_log2;    // consecutive tiles that land in the same output cells (G = F / rows per tile)
  int fsum_row_shift; // coarse index = ((row ^ kxor) << fsum_row_shift) + (kprev >> fsum_log2)
  int fsum_pq;        // floats per output cell (2 = per-pol intensity, 1 = Stokes I / single pol)
  int fsum_split;     // the lane pair is the even / odd samples of ONE single-pol column of twice the
                      // length: X[k] = E + wO, X[k+n/2] = E - wO, w = exp(-2 pi i k / 2^fsum_log2n)
  int fsum_log2n;
  const int* fsum_bins;   // fold fused behind the detection (pbk_stft_fold_exec_device): phase bin of
                          // every segment; the sums are ADDED to out[bin, cell, p] instead of stored
                          // at out[segment, cell, p]
  long long fsum_cells;   // output cells per segment (row length of `out` in cells)
  int split;          // fast MID pass, P == 1: the lane pair is the even / odd samples of ONE column
                      // of length 2N (see fast_chirp); N, df and the tables are the half length's
  // batched launches of trial plans (pbk_dedisp_trials_plan_create) and overlap-save blocks
  // (pbk_dedisp_exec_blocks_device, trial_cc = 0): a launch of the LDG fast kernels with
  // gridDim.y = trials runs batch element blockIdx.y with its input at in + y * trial_in_bytes, its
  // output at out + y * trial_out_bytes and its chirp constants at chan_const + y * trial_cc.  Zero
  // / one by default: single launches compute what they always did.
  long long trial_in_bytes, trial_out_bytes, trial_cc;
  int trials;         // host side: gridDim.y of a fast launch (0 or 1 = one trial)
};

// ------------------------------------------------------------------------------------------
// packed pair arithmetic
// ------------------------------------------------------------------------------------------
struct c2 {
  float2 re, im;
};

__device__ __forceinline__ float2 p_add(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 p_sub(float2 a, float2 b) {
  return __fadd2_rn(a, make_float2(-b.x, -b.y));
}
__device__ __forceinline__ float2 p_mul(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 p_fma(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 p_neg(float2 a) { return make_float2(-a.x, -a.y); }
__device__ __forceinline__ float2 p_bc(float a) { return make_float2(a, a); }

__device__ __forceinline__ c2 operator+(c2 a, c2 b) { return {p_add(a.re, b.re), p_add(a.im, b.im)}; }
__device__ __forceinline__ c2 operator-(c2 a, c2 b) { return {p_sub(a.re, b.re), p_sub(a.im, b.im)}; }

// x * (c + i s) with per-lane (c, s)
__device__ __forceinline__ c2 cmul(c2 x, float2 c, float2 s) {
  c2 r;
  r.re = p_fma(x.re, c, p_neg(p_mul(x.im, s)));
  r.im = p_fma(x.im, c, p_mul(x.re, s));
  return r;
}

template <bool INV>
__device__ __forceinline__ void bf4(c2& x0, c2& x1, c2& x2, c2& x3) {
  c2 a0 = x0 + x2, a1 = x0 - x2, a2 = x1 + x3, a3 = x1 - x3;
  x0 = a0 + a2;
  x2 = a0 - a2;
  if (!INV) {  // a3 * (-i)
    x1.re = p_add(a1.re, a3.im); x1.im = p_sub(a1.im, a3.re);
    x3.re = p_sub(a1.re, a3.im); x3.im = p_add(a1.im, a3.re);
  } else {     // a3 * (+i)
    x1.re = p_sub(a1.re, a3.im); x1.im = p_add(a1.im, a3.re);
    x3.re = p_add(a1.re, a3.im); x3.im = p_sub(a1.im, a3.re);
  }
}

template <bool INV>
__device__ __forceinline__ c2 mul_const(c2 x, float c, float s_fwd) {
  // s_fwd is the imaginary part for the forward sign; inverse conjugates
  const float s = INV ? -s_fwd : s_fwd;
  return cmul(x, p_bc(c), p_bc(s));
}

template <int R, bool INV>
struct Butterfly;

template <bool INV>
struct Butterfly<2, INV> {
  static __device__ __forceinline__ void run(c2* v) {
    c2 t = v[0];
    v[0] = t + v[1];
    v[1] = t - v[1];
  }
};

template <bool INV>
struct Butterfly<4, INV> {
  static __device__ __forceinline__ void run(c2* v) { bf4<INV>(v[0], v[1], v[2], v[3]); }
};

template <bool INV>
struct Butterfly<8, INV> {
  static __device__ __forceinline__ void run(c2* v) {
    constexpr float h = 0.70710678118654752440f;
    bf4<INV>(v[0], v[2], v[4], v[6]);  // E0..E3 in v0,v2,v4,v6
    bf4<INV>(v[1], v[3], v[5], v[7]);  // O0..O3 in v1,v3,v5,v7
    c2 o1 = mul_const<INV>(v[3], h, -h);
    c2 o2;
    if (!INV) { o2.re = v[5].im; o2.im = p_neg(v[5].re); }
    else      { o2.re = p_neg(v[5].im); o2.im = v[5].re; }
    c2 o3 = mul_const<INV>(v[7], -h, -h);
    c2 e0 = v[0], e1 = v[2], e2 = v[4], e3 = v[6], o0 = v[1];
    v[0] = e0 + o0; v[4] = e0 - o0;
    v[1] = e1 + o1; v[5] = e1 - o1;
    v[2] = e2 + o2; v[6] = e2 - o2;
    v[3] = e3 + o3; v[7] = e3 - o3;
  }
};

template <bool INV>
struct Butterfly<16, INV> {
  static __device__ __forceinline__ void run(c2* v) {
    constexpr float C1 = 0.92387953251128675613f;  // cos(pi/8)
    constexpr float S1 = 0.38268343236508977173f;  // sin(pi/8)
    constexpr float h = 0.70710678118654752440f;
    // x[4a+b]: DFT4 over a for each b -> t[b][c] at v[4c+b]
#pragma unroll
    for (int b = 0; b < 4; ++b) bf4<INV>(v[b], v[4 + b], v[8 + b], v[12 + b]);
    // twiddle t[b][c] *= w16^(b*c)
    v[4 * 1 + 1] = mul_const<INV>(v[4 * 1 + 1], C1, -S1);   // e=1
    v[4 * 2 + 1] = mul_const<INV>(v[4 * 2 + 1], h, -h);     // e=2
    v[4 * 3 + 1] = mul_const<INV>(v[4 * 3 + 1], S1, -C1);   // e=3
    v[4 * 1 + 2] = mul_const<INV>(v[4 * 1 + 2], h, -h);     // e=2
    {                                                       // e=4 : -i (fwd) / +i (inv)
      c2 t = v[4 * 2 + 2];
      if (!INV) { v[4 * 2 + 2].re = t.im; v[4 * 2 + 2].im = p_neg(t.re); }
      else      { v[4 * 2 + 2].re = p_neg(t.im); v[4 * 2 + 2].im = t.re; }
    }
    v[4 * 3 + 2] = mul_const<INV>(v[4 * 3 + 2], -h, -h);    // e=6
    v[4 * 1 + 3] = mul_const<INV>(v[4 * 1 + 3], S1, -C1);   // e=3
    v[4 * 2 + 3] = mul_const<INV>(v[4 * 2 + 3], -h, -h);    // e=6
    v[4 * 3 + 3] = mul_const<INV>(v[4 * 3 + 3], -C1, S1);   // e=9
    // DFT4 over b for each c -> y[c + 4d] at v[4c+d]
#pragma unroll
    for (int c = 0; c < 4; ++c) bf4<INV>(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
    // transpose to natural order: out[c + 4d] = v[4c + d]
    c2 t[16];
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
      for (int d = 0; d < 4; ++d) t[c + 4 * d] = v[4 * c + d];
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = t[i];
  }
};

// ------------------------------------------------------------------------------------------
// exact twiddle  w = exp(-2*pi*i * e / 2^log2M)  -> (cos, -sin)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 unit_root(unsigned long long e, int log2M) {
  const long long M = 1ll << log2M;
  long long es = (long long)(e & (unsigned long long)(M - 1));
  if (es >= (M >> 1)) es -= M;
  // x = 2*es/M in [-1, 1): exact for |es| < 2^24, 1 ulp of the index otherwise
  const float x = (float)es * __int_as_float((127 - (log2M - 1)) << 23);
  float s, c;
  sincospif(x, &s, &c);
  return make_float2(c, -s);
}

__device__ __forceinline__ float2 cmul1(float2 a, float2 b) {
  return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}

// ------------------------------------------------------------------------------------------
// per-thread lane context
// ------------------------------------------------------------------------------------------
struct LaneCtx {
  long long bin[2], bout[2];   // element offsets (without the row term)
  unsigned int nrest[2];
  int chan[2];
  int col[2];
  unsigned int klow;           // same for both lanes when FAST; generic path recomputes per lane
  unsigned int klow1;
  bool valid[2];
};

__device__ __forceinline__ long long map_base(const AddrMap& m, long long o_orig, long long kprev,
                                              long long klow, long long nrest, int col, int P) {
  return o_orig * m.a_o + kprev * m.a_kp + klow * m.a_kl + nrest * m.a_n +
         (long long)(col / P) * m.a_c + (long long)(col % P) * m.a_p;
}

template <bool FAST>
__device__ __forceinline__ void lane_setup(const PassArgs& p, LaneCtx& L, int pr) {
  const long long q0 = ((long long)blockIdx.x << (p.log2pw + 1)) + 2 * pr;
#pragma unroll
  for (int l = 0; l < 2; ++l) {
    long long q = q0 + l;
    bool ok = q < p.Q;
    if (!ok) q = 0;
    const long long o = q / p.RI;
    const long long r = q - o * p.RI;
    const long long nrest = r / p.I;
    const int col = (int)(r - nrest * p.I);
    const long long o_orig = o >> p.log2Kprev;
    const long long kprev = o & ((1ll << p.log2Kprev) - 1);
    const long long klow = (kprev >> p.kl_sa) + ((kprev & p.kl_mb) << p.kl_sb);
    L.bin[l] = map_base(p.min, o_orig, kprev, klow, nrest, col, p.P);
    L.bout[l] = map_base(p.mout, o_orig, kprev, klow, nrest, col, p.P);
    L.nrest[l] = (unsigned int)nrest;
    L.chan[l] = col / p.P;
    L.col[l] = col;
    L.valid[l] = ok;
    if (l == 0) L.klow = (unsigned int)klow; else L.klow1 = (unsigned int)klow;
  }
}

// ------------------------------------------------------------------------------------------
// global load / store of one row for the thread's lane pair
// ------------------------------------------------------------------------------------------
// Scratch arrays between passes are "pair-planar" whenever the innermost extent is even: each
// 16-byte pair of adjacent lanes holds {re0, re1, im0, im1}.  e is a complex-element offset.
__device__ __forceinline__ float2 ld_lane_planar(const void* base, long long e) {
  const float* f = reinterpret_cast<const float*>(base) + ((e & ~1ll) << 1) + (e & 1);
  return make_float2(__ldg(f), __ldg(f + 2));
}
__device__ __forceinline__ void st_lane(const PassArgs& p, long long e, float re, float im) {
  if (p.store_planar) {
    float* f = reinterpret_cast<float*>(p.out) + ((e & ~1ll) << 1) + (e & 1);
    f[0] = re;
    f[2] = im;
  } else {
    reinterpret_cast<float2*>(p.out)[e] = make_float2(re, im);
  }
}

// packed raw samples (include/pbk.h: PBK_U4X2, PBK_U2X2)
__device__ __forceinline__ float dec4(unsigned c) { return (float)((int)(c & 15u) - 8); }
__device__ __forceinline__ float dec2(unsigned c) {
  const float mag = (((c ^ (c >> 1)) & 1u) == 0u) ? 3.3359f : 1.0f;   // codes 0 and 3 are the outer levels
  return (c & 2u) ? mag : -mag;
}
// complex element e of a packed array
__device__ __forceinline__ float2 ld_packed(const void* base, long long e, int kind) {
  const unsigned char* b = reinterpret_cast<const unsigned char*>(base);
  if (kind == LOAD_U4X2) {
    const unsigned v = __ldg(b + e);
    return make_float2(dec4(v), dec4(v >> 4));
  }
  const unsigned v = (unsigned)__ldg(b + (e >> 1)) >> ((e & 1) * 4);
  return make_float2(dec2(v & 3u), dec2((v >> 2) & 3u));
}

template <bool FAST>
__device__ __forceinline__ c2 load_row(const PassArgs& p, const LaneCtx& L, long long row) {
  c2 v;
  if (p.load_kind == LOAD_PLANAR) {
    if (FAST) {
      const float2* in = reinterpret_cast<const float2*>(p.in);
      const float4 t = __ldg(reinterpret_cast<const float4*>(in + L.bin[0] + row * p.min.a_row));
      v.re = make_float2(t.x, t.y);
      v.im = make_float2(t.z, t.w);
    } else {
      float2 a = make_float2(0.f, 0.f), b = a;
      if (L.valid[0]) a = ld_lane_planar(p.in, L.bin[0] + row * p.min.a_row);
      if (L.valid[1]) b = ld_lane_planar(p.in, L.bin[1] + row * p.min.a_row);
      v.re = make_float2(a.x, b.x);
      v.im = make_float2(a.y, b.y);
    }
  } else if (p.load_kind == LOAD_F32) {
    const float* in = reinterpret_cast<const float*>(p.in);
    float a = 0.f, b = 0.f;
    if (L.valid[0]) a = __ldg(in + L.bin[0] + row * p.min.a_row);
    if (L.valid[1]) b = __ldg(in + L.bin[1] + row * p.min.a_row);
    v.re = make_float2(a, b);
    v.im = make_float2(0.f, 0.f);
  } else if (p.load_kind == LOAD_C64) {
    const float2* in = reinterpret_cast<const float2*>(p.in);
    if (FAST) {
      const float4 t = __ldg(reinterpret_cast<const float4*>(in + L.bin[0] + row * p.min.a_row));
      v.re = make_float2(t.x, t.z);
      v.im = make_float2(t.y, t.w);
    } else {
      float2 a = make_float2(0.f, 0.f), b = a;
      if (L.valid[0]) a = __ldg(in + L.bin[0] + row * p.min.a_row);
      if (L.valid[1]) b = __ldg(in + L.bin[1] + row * p.min.a_row);
      v.re = make_float2(a.x, b.x);
      v.im = make_float2(a.y, b.y);
    }
  } else if (p.load_kind == LOAD_U4X2 || p.load_kind == LOAD_U2X2) {
    float2 a = make_float2(0.f, 0.f), b = a;
    if (L.valid[0]) a = ld_packed(p.in, L.bin[0] + row * p.min.a_row, p.load_kind);
    if (L.valid[1]) b = ld_packed(p.in, L.bin[1] + row * p.min.a_row, p.load_kind);
    v.re = make_float2(a.x, b.x);
    v.im = make_float2(a.y, b.y);
  } else {
    const char2* in = reinterpret_cast<const char2*>(p.in);
    if (FAST) {
      const char4 t = __ldg(reinterpret_cast<const char4*>(in + L.bin[0] + row * p.min.a_row));
      v.re = make_float2((float)t.x, (float)t.z);
      v.im = make_float2((float)t.y, (float)t.w);
    } else {
      char2 a = make_char2(0, 0), b = a;
      if (L.valid[0]) a = __ldg(in + L.bin[0] + row * p.min.a_row);
      if (L.valid[1]) b = __ldg(in + L.bin[1] + row * p.min.a_row);
      v.re = make_float2((float)a.x, (float)b.x);
      v.im = make_float2((float)a.y, (float)b.y);
    }
  }
  return v;
}

// complex64 store: scratch (pair-planar when store_planar) or a complex64 user array
template <bool FAST>
__device__ __forceinline__ void store_row_c64(const PassArgs& p, const LaneCtx& L, long long row,
                                              long long shift, c2 v) {
  float2* out = reinterpret_cast<float2*>(p.out);
  if (FAST) {
    *reinterpret_cast<float4*>(out + L.bout[0] + row * p.mout.a_row - shift) =
        p.store_planar ? make_float4(v.re.x, v.re.y, v.im.x, v.im.y)
                       : make_float4(v.re.x, v.im.x, v.re.y, v.im.y);
  } else {
    if (L.valid[0]) st_lane(p, L.bout[0] + row * p.mout.a_row - shift, v.re.x, v.im.x);
    if (L.valid[1]) st_lane(p, L.bout[1] + row * p.mout.a_row - shift, v.re.y, v.im.y);
  }
}

// final epilogue: crop on the time index, then c64 / per-pol intensity / Stokes I
template <bool FAST>
__device__ __forceinline__ void store_row_epi(const PassArgs& p, const LaneCtx& L, long long row,
                                              c2 v) {
  // time index of this row (same for both lanes when FAST; per lane otherwise)
  const long long n0 = row * p.n_mul + L.nrest[0];
  const long long n1 = row * p.n_mul + L.nrest[1];
  const bool k0 = n0 >= p.crop_start && n0 < p.crop_stop;
  const bool k1 = n1 >= p.crop_start && n1 < p.crop_stop;
  const long long shift = p.crop_start * p.mout.a_n;  // a_n = elements per unit time index
  if (p.epi_kind == EPI_C64) {
    if (FAST) {
      if (k0) store_row_c64<true>(p, L, row, shift, v);
    } else {
      if (L.valid[0] && k0) st_lane(p, L.bout[0] + row * p.mout.a_row - shift, v.re.x, v.im.x);
      if (L.valid[1] && k1) st_lane(p, L.bout[1] + row * p.mout.a_row - shift, v.re.y, v.im.y);
    }
  } else {
    const float2 pw = p_fma(v.re, v.re, p_mul(v.im, v.im));
    float* out = reinterpret_cast<float*>(p.out);
    if (p.epi_kind == EPI_INTENSITY) {
      if (FAST) {
        if (k0) *reinterpret_cast<float2*>(out + L.bout[0] + row * p.mout.a_row - shift) = pw;
      } else {
        if (L.valid[0] && k0) out[L.bout[0] + row * p.mout.a_row - shift] = pw.x;
        if (L.valid[1] && k1) out[L.bout[1] + row * p.mout.a_row - shift] = pw.y;
      }
    } else {  // Stokes I: the pair is (pol0, pol1) of one channel (host enforces P == 2)
      if (L.valid[0] && k0) out[L.bout[0] + row * p.mout.a_row - shift] = pw.x + pw.y;
    }
  }
}

// ------------------------------------------------------------------------------------------
// shared-memory tile: float4 {re0,re1,im0,im1} at [point ^ swz][pair]
// ------------------------------------------------------------------------------------------
struct Tile {
  float4* s;
  const float2* G;   // per-tile level-twiddle table [lane][16] (apply_level_tw)
  int log2pw;
  int swzmask;  // (points per 128 B) - 1
  __device__ __forceinline__ int idx(int pt, int pr) const {
    return (((pt ^ ((pt >> 4) & swzmask)) << log2pw) + pr);
  }
  __device__ __forceinline__ c2 ld(int pt, int pr) const {
    const float4 t = s[idx(pt, pr)];
    c2 v;
    v.re = make_float2(t.x, t.y);
    v.im = make_float2(t.z, t.w);
    return v;
  }
  __device__ __forceinline__ void st(int pt, int pr, c2 v) const {
    s[idx(pt, pr)] = make_float4(v.re.x, v.re.y, v.im.x, v.im.y);
  }
};

// stage twiddles from the table: tw[q*R + m] = w_M^(q*m) (forward sign); CONJ negates the sine
template <int R, bool CONJ, bool PRE>
__device__ __forceinline__ void apply_stage_tw(c2* v, const float2* __restrict__ tab, int q) {
  if (R == 2) {
    const float2 w = __ldg(tab + q * 2 + 1);
    v[1] = cmul(v[1], p_bc(w.x), p_bc(CONJ ? -w.y : w.y));
  } else {
    const float4* t4 = reinterpret_cast<const float4*>(tab + (size_t)q * R);
#pragma unroll
    for (int j = 0; j < R / 2; ++j) {
      const float4 w = __ldg(t4 + j);
      if (j > 0) v[2 * j] = cmul(v[2 * j], p_bc(w.x), p_bc(CONJ ? -w.y : w.y));
      v[2 * j + 1] = cmul(v[2 * j + 1], p_bc(w.z), p_bc(CONJ ? -w.w : w.w));
    }
  }
}

// inter-level twiddle for register m of a radix-R group: W_M^(nrest * (kbase + m*kstep))
//   = E * G[lane][m],  E = W_M^(nrest*kbase) (one exact root per task and lane),
//   G[lane][m] = W_M^(nrest_lane * kstep * m): a per-tile table in shared memory (the tile's kstep
//   is fixed), so a task needs one sincospif per lane instead of seven.
template <int R, bool CONJ, bool FAST>
__device__ __forceinline__ void apply_level_tw(const PassArgs& p, const LaneCtx& L, c2* v,
                                               unsigned int kbase, const float2* Gtab, int pr) {
  if (p.log2M == 0) return;
  const float2 E0 = unit_root((unsigned long long)L.nrest[0] * kbase, p.log2M);
  const float2 E1 = FAST ? E0 : unit_root((unsigned long long)L.nrest[1] * kbase, p.log2M);
  // table layout [m][lane]: the 16-byte pair entries of a warp are consecutive (no bank conflicts)
  const float4* G4 = reinterpret_cast<const float4*>(Gtab) + pr;
  const int npairs = 1 << p.log2pw;
#pragma unroll
  for (int m = 0; m < R; ++m) {
    const float4 g = m == 0 ? make_float4(1.f, 0.f, 1.f, 0.f) : G4[m * npairs];
    float2 w0 = m == 0 ? E0 : cmul1(E0, make_float2(g.x, g.y));
    float2 w1 = FAST ? w0 : (m == 0 ? E1 : cmul1(E1, make_float2(g.z, g.w)));
    if (CONJ) { w0.y = -w0.y; w1.y = -w1.y; }
    v[m] = cmul(v[m], make_float2(w0.x, w1.x), make_float2(w0.y, w1.y));
  }
}

// nrest of an arbitrary lane of this CTA's tile (same arithmetic as lane_setup)
__device__ __forceinline__ unsigned int lane_nrest(const PassArgs& p, int lane) {
  long long q = ((long long)blockIdx.x << (p.log2pw + 1)) + lane;
  if (q >= p.Q) q = 0;
  const long long o = q / p.RI;
  return (unsigned int)((q - o * p.RI) / p.I);
}

// ------------------------------------------------------------------------------------------
// chirp  H = exp(-2*pi*i*phi(k)) * scale,  phi in cycles evaluated in FP64
// reference: transforms/dedispersion.py:19-23 (f = f_chan + fftfreq; phase = coeff*f*(1/ref-1/f)^2)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 chirp_value(const PassArgs& p, double fchan, long long kfull) {
  // numpy fftfreq: indices >= ceil(N/2) are the negative frequencies (dedispersion.py:20)
  const long long ks = (kfull >= ((p.N + 1) >> 1)) ? kfull - p.N : kfull;
  const double f = fma((double)ks, p.df, fchan);
  const double a = fma(f - p.fr_sub, p.inv_fr, p.a0);   // (f - fr)/fr   (or -1 for fr = inf)
  const double phi = (p.D * a) * a / f;                 // cycles
  const double fr = phi - rint(phi);                    // exact reduction to [-0.5, 0.5]
  float s, c;
  sincospif(2.0f * (float)fr, &s, &c);
  return make_float2(c * p.scale, -s * p.scale);
}

// CHIRP_RAMP transfer function for column `col` at FFT bin kf of an N-point transform (any N):
// exp(-2 pi i s fftfreq(N,1)[kf]) (transforms.py:271), zero inside the band [lo, hi) given in
// fftshift-ed positions (transforms.py:350-359), optional analytic-signal weights (utils.py:50-54)
__device__ __forceinline__ float2 ramp_value(const PassArgs& p, int col, long long kf) {
  const long long ks = (kf >= ((p.N + 1) >> 1)) ? kf - p.N : kf;
  const double ph = (double)ks * p.ramp_shift[col];
  const double fr = ph - rint(ph);
  float s, c;
  sincospif(2.0f * (float)fr, &s, &c);
  long long sh = kf + (p.N >> 1);               // position after fftshift
  if (sh >= p.N) sh -= p.N;
  if (sh >= p.ramp_zero[2 * col] && sh < p.ramp_zero[2 * col + 1]) return make_float2(0.f, 0.f);
  float wgt = p.scale;
  if (p.ramp_hilbert) {   // h[0] = 1, h[1 : N//2] = 2, h[N//2] = 2 if N odd else 1, rest 0
    const long long h2 = p.N >> 1;
    if (kf == 0) wgt *= 1.f;
    else if (kf < h2) wgt *= 2.f;
    else if (kf == h2) wgt *= (p.N & 1) ? 2.f : 1.f;
    else wgt = 0.f;
  }
  return make_float2(c * wgt, -s * wgt);
}

template <bool FAST>
__device__ __forceinline__ void apply_chirp16(const PassArgs& p, const LaneCtx& L, c2* v,
                                              unsigned int kbase, unsigned int kstep) {
  if (p.chirp_kind == CHIRP_NONE) {
    if (p.scale != 1.0f) {
      const float2 sc = p_bc(p.scale);
#pragma unroll
      for (int m = 0; m < 16; ++m) { v[m].re = p_mul(v[m].re, sc); v[m].im = p_mul(v[m].im, sc); }
    }
    return;
  }
  if (p.chirp_kind == CHIRP_COMPUTED) {
    const double f0 = p.chan_freq[L.chan[0]];
    const double f1 = FAST ? f0 : p.chan_freq[L.chan[1]];
#pragma unroll
    for (int m = 0; m < 16; ++m) {
      const unsigned int k = kbase + m * kstep;
      const long long kf0 = (long long)L.klow + ((long long)k << p.log2Kmul);
      const float2 h0 = chirp_value(p, f0, kf0);
      if (FAST) {
        v[m] = cmul(v[m], p_bc(h0.x), p_bc(h0.y));
      } else {
        const long long kf1 = (long long)L.klow1 + ((long long)k << p.log2Kmul);
        const float2 h1 = chirp_value(p, f1, kf1);
        v[m] = cmul(v[m], make_float2(h0.x, h1.x), make_float2(h0.y, h1.y));
      }
    }
  } else if (p.chirp_kind == CHIRP_RAMP) {
    // linear phase ramp per column (transforms.py:271 time_shift) and/or a zeroed band
    // (transforms.py:350-359 freq_shift); phase in FP64, reduced exactly before sincospif
#pragma unroll
    for (int m = 0; m < 16; ++m) {
      const unsigned int k = kbase + m * kstep;
      float2 h[2];
#pragma unroll
      for (int l = 0; l < 2; ++l) {
        const long long kf = (long long)(l == 0 ? L.klow : (FAST ? L.klow : L.klow1)) +
                             ((long long)k << p.log2Kmul);
        h[l] = ramp_value(p, L.col[l], kf);
      }
      v[m] = cmul(v[m], make_float2(h[0].x, h[1].x), make_float2(h[0].y, h[1].y));
    }
  } else {  // explicit (N, C) complex64 array supplied by the caller (dedispersion.py:121-124)
#pragma unroll
    for (int m = 0; m < 16; ++m) {
      const unsigned int k = kbase + m * kstep;
      const long long kf0 = (long long)L.klow + ((long long)k << p.log2Kmul);
      const long long kf1 = (long long)(FAST ? L.klow : L.klow1) + ((long long)k << p.log2Kmul);
      const float2 h0 = __ldg(p.chirp_arr + kf0 * p.chirp_sk + (long long)L.chan[0] * p.chirp_sc);
      const float2 h1 = __ldg(p.chirp_arr + kf1 * p.chirp_sk + (long long)L.chan[1] * p.chirp_sc);
      v[m] = cmul(v[m], make_float2(h0.x * p.scale, h1.x * p.scale),
                  make_float2(h0.y * p.scale, h1.y * p.scale));
    }
  }
}

// digit reversal of the last-stage block index b -> low part of the tile-level frequency index.
// radices are (r1, 16, 16, ...): b = ((m1 * 16 + m2) * 16 + ...), klo = m1 + r1*(m2 + 16*(...)).
__device__ __forceinline__ unsigned int klo_of_block(unsigned int b, int nstages, int log2r1) {
  if (nstages <= 1) return 0;
  unsigned int klo = 0, mul_shift = log2r1 + 4 * (nstages - 2);
  // peel digits from the least significant (last radix-16 digit is most significant in k)
  for (int s = nstages - 2; s >= 1; --s) {
    mul_shift -= 4;
    klo += (b & 15u) << (mul_shift);
    b >>= 4;
  }
  klo += b;  // m1
  return klo;
}

// ------------------------------------------------------------------------------------------
// generic smem -> smem stage (radix 16), DIF (butterfly then twiddle) or DIT (conj twiddle first)
// ------------------------------------------------------------------------------------------
template <bool DIT>
__device__ __forceinline__ void smem_stage16(const PassArgs& p, const Tile& T, int stage,
                                             int log2S, int pr, int bfirst, int bstep, int nb) {
  const float2* tab = p.stage_tw + p.stage_tw_off[stage];
  const int S = 1 << log2S;
  for (int b = bfirst; b < nb; b += bstep) {
    const int q = b & (S - 1);
    const int base = ((b >> log2S) << (log2S + 4)) + q;
    c2 v[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = T.ld(base + (i << log2S), pr);
    if (DIT) {
      apply_stage_tw<16, true, true>(v, tab, q);
      Butterfly<16, true>::run(v);
    } else {
      Butterfly<16, false>::run(v);
      apply_stage_tw<16, false, false>(v, tab, q);
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) T.st(base + (i << log2S), pr, v[i]);
  }
}

// ------------------------------------------------------------------------------------------
// first forward stage: global -> registers -> (smem | global when the tile is one stage)
//   FWD/MID: DIF radix R1 with stage table 0.  SIGNINV (FWD mode ifft): conjugated exponent.
// ------------------------------------------------------------------------------------------
template <int R, bool FAST, bool SIGNINV, int MODE>
__device__ __forceinline__ void first_stage(const PassArgs& p, const LaneCtx& L, const Tile& T,
                                            int pr, int bfirst, int bstep) {
  const int log2S = p.log2L - (R == 2 ? 1 : R == 4 ? 2 : R == 8 ? 3 : 4);
  const int S = 1 << log2S;
  const float2* tab = p.stage_tw + p.stage_tw_off[0];
  for (int b = bfirst; b < S; b += bstep) {
    c2 v[R];
#pragma unroll
    for (int i = 0; i < R; ++i) v[i] = load_row<FAST>(p, L, (long long)((b + (i << log2S)) ^ p.fxor));
    Butterfly<R, SIGNINV>::run(v);
    if (p.nstages > 1) {
      apply_stage_tw<R, SIGNINV, false>(v, tab, b);
#pragma unroll
      for (int i = 0; i < R; ++i) T.st(b + (i << log2S), pr, v[i]);
    } else {
      // single-stage tile (L == R): FWD mode only; registers hold k = m
      apply_level_tw<R, SIGNINV, FAST>(p, L, v, 0u, T.G, pr);
      if (p.scale != 1.0f) {
        const float2 sc = p_bc(p.scale);
#pragma unroll
        for (int i = 0; i < R; ++i) { v[i].re = p_mul(v[i].re, sc); v[i].im = p_mul(v[i].im, sc); }
      }
#pragma unroll
      for (int i = 0; i < R; ++i) store_row_c64<FAST>(p, L, (long long)(i ^ p.kxor), 0, v[i]);
    }
  }
}

// last inverse stage (mirror of first_stage): smem -> registers -> epilogue
template <int R, bool FAST>
__device__ __forceinline__ void last_inv_stage(const PassArgs& p, const LaneCtx& L, const Tile& T,
                                               int pr, int bfirst, int bstep, bool final_epi) {
  const int log2S = p.log2L - (R == 2 ? 1 : R == 4 ? 2 : R == 8 ? 3 : 4);
  const int S = 1 << log2S;
  const float2* tab = p.stage_tw + p.stage_tw_off[0];
  for (int b = bfirst; b < S; b += bstep) {
    c2 v[R];
#pragma unroll
    for (int i = 0; i < R; ++i) v[i] = T.ld(b + (i << log2S), pr);
    apply_stage_tw<R, true, true>(v, tab, b);
    Butterfly<R, true>::run(v);
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const long long row = b + (i << log2S);
      if (final_epi) store_row_epi<FAST>(p, L, row, v[i]);
      else store_row_c64<FAST>(p, L, row, 0, v[i]);
    }
  }
}

template <bool FAST, bool SIGNINV, int MODE>
__device__ __forceinline__ void run_first(const PassArgs& p, const LaneCtx& L, const Tile& T, int pr,
                                          int bfirst, int bstep) {
  switch (p.log2r1) {
    case 1: first_stage<2, FAST, SIGNINV, MODE>(p, L, T, pr, bfirst, bstep); break;
    case 2: first_stage<4, FAST, SIGNINV, MODE>(p, L, T, pr, bfirst, bstep); break;
    case 3: first_stage<8, FAST, SIGNINV, MODE>(p, L, T, pr, bfirst, bstep); break;
    default: first_stage<16, FAST, SIGNINV, MODE>(p, L, T, pr, bfirst, bstep); break;
  }
}

template <bool FAST>
__device__ __forceinline__ void run_last_inv(const PassArgs& p, const LaneCtx& L, const Tile& T,
                                             int pr, int bfirst, int bstep, bool final_epi) {
  switch (p.log2r1) {
    case 1: last_inv_stage<2, FAST>(p, L, T, pr, bfirst, bstep, final_epi); break;
    case 2: last_inv_stage<4, FAST>(p, L, T, pr, bfirst, bstep, final_epi); break;
    case 3: last_inv_stage<8, FAST>(p, L, T, pr, bfirst, bstep, final_epi); break;
    default: last_inv_stage<16, FAST>(p, L, T, pr, bfirst, bstep, final_epi); break;
  }
}

// ------------------------------------------------------------------------------------------
// the pass kernel
// ------------------------------------------------------------------------------------------
template <int MODE, bool FAST, bool SIGNINV>
__global__ void __launch_bounds__(kThreads, 2) pass_kernel(const __grid_constant__ PassArgs p) {
  extern __shared__ float4 smem_dyn[];
  pdl_trigger();
  pdl_wait();
  Tile T;
  T.s = smem_dyn;
  T.log2pw = p.log2pw;
  {
    const int ppb = 8 >> p.log2pw;  // points per 128 bytes
    T.swzmask = ppb > 1 ? ppb - 1 : 0;
  }
  const int pw = 1 << p.log2pw;
  const int pr = threadIdx.x & (pw - 1);
  int bfirst = threadIdx.x >> p.log2pw;
  const int bstep = kThreads >> p.log2pw;

  LaneCtx L;
  lane_setup<FAST>(p, L, pr);
  // lane pairs past the end of the array do no work (they still reach every barrier)
  if (!L.valid[0] && !L.valid[1]) bfirst = 1 << 30;

  const int ns = p.nstages;
  const int nb16 = 1 << (p.log2L - 4);            // radix-16 groups per lane pair
  const unsigned int kstep = ns > 1 ? 1u << (p.log2L - 4) : 1u;  // k spacing of last-stage registers

  // level-twiddle table of this tile: G[lane][m] = W_M^(nrest_lane * kstep * m), behind the tile
  {
    float2* G = reinterpret_cast<float2*>(smem_dyn + (ns > 1 ? ((size_t)1 << (p.log2L + p.log2pw)) : 0));
    T.G = G;
    if (p.log2M != 0 && MODE != MODE_MID) {
      for (int idx = threadIdx.x; idx < (2 * pw) * 16; idx += kThreads) {
        const int m = idx / (2 * pw), lane = idx - m * (2 * pw);   // [m][lane]
        G[idx] = unit_root((unsigned long long)lane_nrest(p, lane) * (kstep * (unsigned)m), p.log2M);
      }
      __syncthreads();
    }
  }

  if (MODE == MODE_FWD) {
    // level transform, DIF: first stage from global, middle stages in smem, last stage to global
    if (ns == 1) {
      run_first<FAST, SIGNINV, MODE>(p, L, T, pr, bfirst, bstep);
      return;
    }
    run_first<FAST, SIGNINV, MODE>(p, L, T, pr, bfirst, bstep);
    __syncthreads();
    for (int s = 1; s < ns - 1; ++s) {
      const int log2S = 4 * (ns - 1 - s);
      if (SIGNINV) {
        // inverse exponent with the DIF graph: conjugated butterflies and twiddles
        const float2* tab = p.stage_tw + p.stage_tw_off[s];
        const int S = 1 << log2S;
        for (int b = bfirst; b < nb16; b += bstep) {
          const int q = b & (S - 1);
          const int base = ((b >> log2S) << (log2S + 4)) + q;
          c2 v[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = T.ld(base + (i << log2S), pr);
          Butterfly<16, true>::run(v);
          apply_stage_tw<16, true, false>(v, tab, q);
#pragma unroll
          for (int i = 0; i < 16; ++i) T.st(base + (i << log2S), pr, v[i]);
        }
      } else {
        smem_stage16<false>(p, T, s, log2S, pr, bfirst, bstep, nb16);
      }
      __syncthreads();
    }
    for (int b = bfirst; b < nb16; b += bstep) {
      c2 v[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = T.ld((b << 4) + i, pr);
      Butterfly<16, SIGNINV>::run(v);
      const unsigned int klo = klo_of_block((unsigned int)b, ns, p.log2r1);
      apply_level_tw<16, SIGNINV, FAST>(p, L, v, klo, T.G, pr);
      if (p.scale != 1.0f) {
        const float2 sc = p_bc(p.scale);
#pragma unroll
        for (int i = 0; i < 16; ++i) { v[i].re = p_mul(v[i].re, sc); v[i].im = p_mul(v[i].im, sc); }
      }
#pragma unroll
      for (int i = 0; i < 16; ++i)
        store_row_c64<FAST>(p, L, (long long)((klo + i * kstep) ^ (unsigned int)p.kxor), 0, v[i]);
    }
  } else if (MODE == MODE_MID) {
    // last level: forward DIF, chirp in registers, inverse DIT
    if (ns > 1) {
      run_first<FAST, false, MODE>(p, L, T, pr, bfirst, bstep);
      __syncthreads();
      for (int s = 1; s < ns - 1; ++s) {
        smem_stage16<false>(p, T, s, 4 * (ns - 1 - s), pr, bfirst, bstep, nb16);
        __syncthreads();
      }
    }
    for (int b = bfirst; b < nb16; b += bstep) {
      c2 v[16];
      if (ns > 1) {
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = T.ld((b << 4) + i, pr);
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = load_row<FAST>(p, L, (long long)i);
      }
      Butterfly<16, false>::run(v);
      const unsigned int klo = klo_of_block((unsigned int)b, ns, p.log2r1);
      apply_chirp16<FAST>(p, L, v, klo, kstep);
      Butterfly<16, true>::run(v);
      if (ns > 1) {
#pragma unroll
        for (int i = 0; i < 16; ++i) T.st((b << 4) + i, pr, v[i]);
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) store_row_epi<FAST>(p, L, (long long)i, v[i]);
      }
    }
    if (ns > 1) {
      __syncthreads();
      for (int s = ns - 2; s >= 1; --s) {
        smem_stage16<true>(p, T, s, 4 * (ns - 1 - s), pr, bfirst, bstep, nb16);
        __syncthreads();
      }
      run_last_inv<FAST>(p, L, T, pr, bfirst, bstep, true);
    }
  } else {  // MODE_INV: inverse level, DIT: conj level twiddle, radix-16 from global, ... , epilogue
    for (int b = bfirst; b < nb16; b += bstep) {
      const unsigned int klo = klo_of_block((unsigned int)b, ns, p.log2r1);
      c2 v[16];
#pragma unroll
      for (int i = 0; i < 16; ++i) v[i] = load_row<FAST>(p, L, (long long)(klo + i * kstep));
      apply_level_tw<16, true, FAST>(p, L, v, klo, T.G, pr);
      Butterfly<16, true>::run(v);
      if (ns > 1) {
#pragma unroll
        for (int i = 0; i < 16; ++i) T.st((b << 4) + i, pr, v[i]);
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) store_row_epi<FAST>(p, L, (long long)i, v[i]);
      }
    }
    if (ns > 1) {
      __syncthreads();
      for (int s = ns - 2; s >= 1; --s) {
        smem_stage16<true>(p, T, s, 4 * (ns - 1 - s), pr, bfirst, bstep, nb16);
        __syncthreads();
      }
      run_last_inv<FAST>(p, L, T, pr, bfirst, bstep, true);
    }
  }
}

}  // namespace pbk
