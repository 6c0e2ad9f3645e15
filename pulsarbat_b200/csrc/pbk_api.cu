// pbk_api.cu -- host side of libpbk.so: plans, pass scheduling and the C ABI of include/pbk.h.
//
// A plan turns one reference call into a short fixed list of kernel launches:
//   coherent_dedispersion (transforms/dedispersion.py:81-133), N = L1*..*Lm:
//       FWD(L1) .. FWD(Lm-1)  ->  MID(Lm: fft, chirp, ifft)  ->  INV(Lm-1) .. INV(L1)+epilogue
//   pb.fft.fft/ifft axis 0 (fft.py:30-48), stft/istft (contrib/misc.py:17-93):
//       FWD(L1) .. FWD(Lm) with a natural-order (optionally fftshift-ed) store in the last pass.
// All index arithmetic the reference does with reshape/swapaxes/fftshift is folded into the
// AddrMap of the first and last pass, so no transposed copy is ever made.
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/pbk.h"
#include "pbk_fast_launch.h"
#include "pbk_tma_launch.h"
#include "pbk_blue.cuh"
#include "pbk_f64.cuh"
#include "pbk_fft.cuh"
#include "pbk_hostcopy.h"
#include "pbk_misc.cuh"
#include "pbk_incoh.cuh"
#include "pbk_search.cuh"
#include "pbk_sk.cuh"
#include "pbk_fdmt.cuh"

using namespace pbk;

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define CUDA_TRY(expr)                                                                 \
  do {                                                                                 \
    cudaError_t e__ = (expr);                                                          \
    if (e__ != cudaSuccess)                                                            \
      return fail(e__ == cudaErrorMemoryAllocation ? PBK_ERR_NOMEM : PBK_ERR_CUDA,     \
                  "%s failed: %s", #expr, cudaGetErrorString(e__));                    \
  } while (0)

extern "C" const char* pbk_last_error(void) { return g_err; }
extern "C" int pbk_version(void) { return PBK_VERSION; }
extern "C" const char* pbk_status_string(int s) {
  switch (s) {
    case PBK_OK: return "ok";
    case PBK_ERR_INVALID: return "invalid argument";
    case PBK_ERR_UNSUPPORTED: return "unsupported";
    case PBK_ERR_CUDA: return "CUDA error";
    case PBK_ERR_NOMEM: return "out of memory";
  }
  return "unknown";
}
extern "C" int pbk_device_count(int* count) {
  if (!count) return fail(PBK_ERR_INVALID, "count is NULL");
  *count = 0;
  CUDA_TRY(cudaGetDeviceCount(count));
  return PBK_OK;
}

extern "C" int pbk_device_pci_bus_id(int device, char* buf, int n) {
  if (!buf || n < 16) return fail(PBK_ERR_INVALID, "buffer of at least 16 bytes expected");
  CUDA_TRY(cudaDeviceGetPCIBusId(buf, n, device));
  return PBK_OK;
}

extern "C" int pbk_device_mem_info(int device, size_t* free_bytes, size_t* total_bytes) {
  CUDA_TRY(cudaSetDevice(device));
  size_t f = 0, t = 0;
  CUDA_TRY(cudaMemGetInfo(&f, &t));
  if (free_bytes) *free_bytes = f;
  if (total_bytes) *total_bytes = t;
  return PBK_OK;
}

// ------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------
enum Role { ROLE_USER_IN = 0, ROLE_SCRATCH = 1, ROLE_USER_OUT = 2, ROLE_TMPF = 3 };
enum PlanKind { PLAN_DEDISP = 0, PLAN_FFT = 1, PLAN_INCOH = 2, PLAN_FDMT = 3 };

struct Pass {
  int mode = MODE_FWD;
  bool fast = false;      // uniform lane pairs (same time offset AND channel): vector generic path
  bool pair_ok = false;   // lane pairs usable by the fast family (P even, or P == 1: two channels)
  bool fast_load_transposed = false;   // fast FWD pass reads its tile through the transposing loader
  bool signinv = false;
  int in_role = ROLE_USER_IN, out_role = ROLE_SCRATCH;
  PassArgs a;
  unsigned grid = 0;
  size_t smem = 0;
  // compile-time-shaped kernel (pbk_fast.cuh); family < 0 = generic runtime-shaped kernel
  int family = -1;
  FastInfo finfo{};
  long long ntiles = 0;
  size_t ftab_off = 0;  // float2 offset into plan->d_ftab
  // TMA-pipelined variant of the same tile shape (pbk_tma.cuh); decided by setup_tma
  bool tma = false;
  TmaInfo tinfo{};
};

struct BlueState;   // arbitrary-length (Bluestein) plans, see below

struct pbk_plan {
  int kind = PLAN_DEDISP;
  BlueState* blue = nullptr;
  int device = 0;
  std::mutex mu;
  std::vector<Pass> passes;
  int nlevels = 0;
  int level_log2[3] = {0, 0, 0};
  // device resources owned by the plan
  void* scratch = nullptr;
  size_t scratch_bytes = 0;
  void* scratch2 = nullptr;     // second scratch array: intermediate passes run out of place
  float2* d_tw = nullptr;
  double* d_chanfreq = nullptr;
  double* d_chanconst = nullptr;   // per-channel constants of the fast MID chirp
  double* d_ramp_shift = nullptr;  // CHIRP_RAMP plans: s/N per column
  long long* d_ramp_zero = nullptr;   // and the zeroed band [lo, hi) per column
  bool chirp_series_ok = true;     // |delta/fc| small enough for the division-free chirp
  float2* d_ftab = nullptr;     // stage tables of the fast kernels
  int num_sms = 148;
  void* d_tmpf = nullptr;       // pre-downsample float buffer
  size_t tmpf_bytes = 0;
  bool fused_tsum = false;      // the time sum runs in the epilogue of the last pass (no d_tmpf)
  // channelizer plans with a detected output (pbk_stft_detect_plan_create)
  long long det_nseg = 0, det_cells = 0;
  int det_pq = 0;
  int* d_segbins = nullptr;          // phase bin per segment (channelizer) or output row
                                     // (dedispersion) of the current folded execution
  const int* exec_segbins = nullptr; // non-null while a fold execution runs the passes
  void* d_foldbuf = nullptr;         // dedispersion fold on the unfused route: the plan's output
  size_t fold_bytes = 0;             // lazily allocated d_segbins + d_foldbuf of a dedispersion plan
  bool split_column = false;    // single column run as its even / odd samples (see plan creation)
  bool split_ragged = false;    // ... with an odd crop edge: passes write d_tmpf, then a D2D copy
  size_t split_skip = 0;
  void* d_stage = nullptr;      // 16-byte aligned stand-in for a caller's array that is not (see
  size_t stage_bytes = 0;       // stage_ensure); lazily allocated, grown on demand
  // lazily allocated staging buffers for *_host execution
  void* h_din = nullptr;
  void* h_dout = nullptr;
  void* h_dchirp = nullptr;
  size_t in_bytes = 0, out_bytes = 0, chirp_bytes = 0;
  // dedisp description
  pbk_dedisp_desc desc{};
  int64_t out_rows = 0, row_elems = 0, elem_bytes = 0, full_rows = 0;
  int launches = 0;
  int segments = 0;             // timed segments per execution (pbk_plan_profile_read)
  // trial plans (pbk_dedisp_trials_plan_create): the forward passes run once per execution, the
  // MID pass and every pass after it once per trial DM, with that trial's chirp constants
  bool trials = false;
  int ndm = 1;
  int nshared = 0;              // leading passes shared by all trials
  std::vector<double> trial_D;  // PassArgs::D of each trial; d_chanconst holds ndm tables of 3C
  long long chanconst_stride = 0;
  int trials_per_launch = 1;    // T: trials batched along gridDim.y of each per-trial launch
  size_t work_bytes = 0;        // the per-trial scratch array holds T slabs of scratch_bytes
  // overlap-save blocks (pbk_dedisp_exec_blocks_device) of a single-DM plan
  int blocks_per_launch = 1;    // T: blocks batched along gridDim.y (choose_per_launch)
  // T slabs of scratch_bytes per scratch array the plan uses, allocated at the first batched
  // execution
  void* blk_scratch[2] = {nullptr, nullptr};
  size_t blk_bytes = 0;
  // optional per-launch device timing (pbk_plan_profile): ring of event sets, one per execution
  std::vector<std::vector<cudaEvent_t>> prof;
  long long prof_next = 0;
  int prof_cur = -1;
  bool prof_off = false;        // block executions are not timed
  // incoherent trial plans (pbk_incoh_trials_plan_create): one launch of incoh_trials_kernel<KD>
  pbk_incoh::Args incoh{};      // device pointers into d_incoh; in / out set per execution
  int incoh_kd = 0;
  unsigned incoh_grid = 0;
  size_t incoh_smem = 0;
  int* d_incoh = nullptr;       // perm, off, lo and ext tables
  size_t incoh_bytes = 0;
  // FDMT plans (pbk_fdmt_plan_create)
  struct FdmtPlan* fdmt = nullptr;
};

static void prof_mark(pbk_plan* pl, int idx, cudaStream_t st) {
  if (pl->prof_cur >= 0) cudaEventRecord(pl->prof[pl->prof_cur][idx], st);
}
static void prof_begin(pbk_plan* pl) {
  pl->prof_cur = (pl->prof.empty() || pl->prof_off)
                     ? -1 : (int)(pl->prof_next++ % (long long)pl->prof.size());
}

static int ilog2_exact(int64_t v) {
  if (v <= 0 || (v & (v - 1))) return -1;
  int l = 0;
  while ((1ll << l) < v) ++l;
  return l;
}

struct TableSet {
  std::vector<float2> host;
  int off_by_log2L[16][kMaxStages];
  bool have[16];
  TableSet() { memset(have, 0, sizeof(have)); memset(off_by_log2L, 0, sizeof(off_by_log2L)); }
  void ensure(int log2L) {
    if (have[log2L]) return;
    have[log2L] = true;
    const int ns = (log2L + 3) / 4;
    const int log2r1 = log2L - 4 * (ns - 1);
    const long long Lt = 1ll << log2L;
    for (int s = 0; s + 1 < ns; ++s) {
      const int R = s == 0 ? (1 << log2r1) : 16;
      const long long M = s == 0 ? Lt : (1ll << (4 * (ns - s)));
      const long long S = M / R;
      off_by_log2L[log2L][s] = (int)host.size();
      for (long long q = 0; q < S; ++q)
        for (int m = 0; m < R; ++m) {
          const long long e = (q * m) % M;
          const double ang = -2.0 * M_PI * (double)e / (double)M;
          host.push_back(make_float2((float)cos(ang), (float)sin(ang)));
        }
      while (host.size() % 2) host.push_back(make_float2(0.f, 0.f));  // keep 16 B alignment
    }
  }
};

static AddrMap plain_map(long long Lt, long long R, long long I, long long P) {
  AddrMap m;
  m.a_o = 0;  // filled by caller (elements per o_orig)
  m.a_kp = Lt * R * I;
  m.a_kl = 0;
  m.a_n = I;
  m.a_c = P;
  m.a_p = 1;
  m.a_row = R * I;
  return m;
}

static bool map_even(const AddrMap& m, long long P) {
  if ((m.a_o | m.a_kp | m.a_kl | m.a_n | m.a_row) & 1) return false;
  if (P % 2 == 0) return m.a_p == 1 && (m.a_c % 2 == 0);
  return P == 1 && m.a_c == 1;
}

static void set_geometry(Pass& ps, int log2L, long long Q, long long RI, int I, int P,
                         int log2Kprev) {
  PassArgs& a = ps.a;
  a.Q = Q;
  a.RI = RI;
  a.I = I;
  a.P = P;
  a.log2L = log2L;
  a.nstages = (log2L + 3) / 4;
  a.log2r1 = log2L - 4 * (a.nstages - 1);
  int lpw = std::min(7, std::max(0, 12 - log2L));
  const long long pairs = (Q + 1) / 2;
  while (lpw > 0 && (1ll << (lpw - 1)) >= pairs) --lpw;
  // small problems: prefer narrower tiles until every SM has a few CTAs to overlap (a 2^20-point
  // single column gives 128 tiles of 64 KiB otherwise, fewer than the 148 SMs)
  {
    static const long long min_grid = [] {
      const char* e = getenv("PBK_GENERIC_MINGRID");
      return e ? atoll(e) : 0ll;
    }();
    while (lpw > 1 && (Q + (2ll << lpw) - 1) / (2ll << lpw) < min_grid) --lpw;
  }
  a.log2pw = lpw;
  a.log2Kprev = log2Kprev;
  // tile (multi-stage tiles only) + per-tile level-twiddle table [lanes][16]
  ps.smem = (a.nstages > 1 ? ((size_t)1 << (log2L + lpw)) * sizeof(float4) : 0) +
            ((size_t)2 << lpw) * 16 * sizeof(float2);
  const long long W = 2ll << lpw;
  ps.grid = (unsigned)((Q + W - 1) / W);
}

static void defaults(PassArgs& a) {
  memset(&a, 0, sizeof(a));
  a.sign = -1;
  a.scale = 1.0f;
  a.load_kind = LOAD_C64;
  a.epi_kind = EPI_C64;
  a.crop_start = 0;
  a.crop_stop = LLONG_MAX;
  a.n_mul = 0;
  a.chirp_kind = CHIRP_NONE;
}

static void set_klow(PassArgs& a, int level /*1-based*/, const int* l) {
  a.kl_sa = 0; a.kl_mb = 0; a.kl_sb = 0;
  if (level == 3) { a.kl_sa = l[1]; a.kl_mb = (1 << l[1]) - 1; a.kl_sb = l[0]; }
}

// Level split N = 2^l[0] * .. * 2^l[m-1], chosen with a cost model built from measurements on
// B200 (scripts/chunk_bw.cu, scripts/chunk_bw2.cu; logs under profiles/): what a pass can pull
// from HBM depends almost only on the width of the contiguous chunk it touches per row,
//   row stride >= 64 KiB :  32 B 1.55 | 64 B 3.1 | 128 B 4.6 | >=256 B 6.0  TB/s
//   consecutive rows     :  32 B 3.8  | 64 B 5.7 | 128 B 5.7 | >=256 B 6.0  TB/s
// and a 64 KiB tile of 2^l points leaves 65536/2^l bytes per row.  Strided levels are paid
// twice (forward and inverse pass), the last level once (fused fft*chirp*ifft pass).
static double bw_strided(double chunk) {
  if (chunk >= 256) return 6.0;
  if (chunk >= 128) return 4.6;
  if (chunk >= 64) return 3.1;
  if (chunk >= 32) return 1.55;
  return 1.55 * chunk / 32.0;
}
static double bw_rows(double chunk) {
  if (chunk >= 256) return 6.0;
  if (chunk >= 64) return 5.7;
  if (chunk >= 32) return 3.8;
  return 3.8 * chunk / 32.0;
}
static double level_chunk_bytes(int l, long long lanes_avail) {
  double w = 65536.0 / (double)(1ll << l) / 8.0;   // lanes in a 64 KiB tile
  if (w > 128) w = 128;
  if (w > (double)lanes_avail) w = (double)lanes_avail;
  return w * 8.0;
}

namespace pbk { bool fast_info(int family, int log2L, FastInfo* info); }
static int preferred_family();

// true when a pass of tile length 2^l over I lanes can run on a compile-time-shaped kernel
static bool level_is_fast(int l, long long I) {
  const int fam = preferred_family();
  FastInfo fi;
  if (fam < 0 || (I & 1) || !pbk::fast_info(fam, l, &fi)) return false;
  const long long W = 2ll << fi.log2pw;
  return I % W == 0 || W % I == 0;
}

static int choose_levels(int n, long long I, int* l, bool need_mid16) {
  const char* e = getenv("PBK_LEVELS");   // developer override, e.g. PBK_LEVELS=11,11
  if (e) {
    int a = 0, b = 0, c = 0;
    const int got = sscanf(e, "%d,%d,%d", &a, &b, &c);
    if (got >= 1 && a + b + c == n) {
      l[0] = a; l[1] = b; l[2] = c;
      return got;
    }
  }
  const int lo = 4, hi = 12;
  // estimated seconds per execution: every pass moves the whole array once each way at the
  // bandwidth its chunk width allows, plus a fixed launch/ramp cost that decides small problems
  const double pass_tb = (double)(1ll << n) * (double)I * 16.0 * 1e-12;
  const double pass_fixed = 4e-6;
  // an array that stays in the 126 MB L2 is not limited by the HBM chunk-width effects
  const bool l2_resident = pass_tb * 1e12 <= 2.0 * (48ll << 20);
  auto bw_s = [&](double chunk) { return l2_resident ? 6.0 : bw_strided(chunk); };
  auto bw_r = [&](double chunk) { return l2_resident ? 6.0 : bw_rows(chunk); };
  double best = 1e30;
  int bm = 0, bl[3] = {0, 0, 0};
  auto consider = [&](int m, int a, int b, int c) {
    const int ls[3] = {a, b, c};
    if (ls[m - 1] < (need_mid16 ? 4 : 1) || ls[m - 1] > hi) return;
    double cost = 0;
    long long R = 1ll << n;
    for (int i = 0; i < m; ++i) {
      R >>= ls[i];
      if (i + 1 < m) {
        if (need_mid16 && ls[i] < lo) return;   // inverse passes start with a radix-16 stage
        // tiles longer than 2^8 need a third butterfly stage per pass
        // the runtime-shaped generic kernel issues ~3.5x the instructions of a fast one
        const double stages = (ls[i] <= 8 ? 1.0 : 1.0 + 0.15 * (ls[i] - 8)) *
                              (need_mid16 && !level_is_fast(ls[i], I) ? 2.2 : 1.0);
        cost += 2.0 * (stages * pass_tb / bw_s(level_chunk_bytes(ls[i], R * I)) + pass_fixed);
      } else {
        // the fused fft*chirp*ifft pass does two transforms of 2^l plus the chirp per tile and is
        // issue-bound beyond l = 6 (measured on cfg2: 1.51 / 1.86 / 2.28 ms for l = 6 / 7 / 8
        // against 1.45 ms for a plain pass); below 2^6 only the generic kernel exists
        static const double mid_factor[13] = {3.0,  3.0, 3.0, 3.0, 3.0, 3.0, 1.05,
                                              1.3,  1.6, 1.9, 2.2, 2.5, 2.8};
        const double f = need_mid16 ? mid_factor[ls[i]] * (level_is_fast(ls[i], I) ? 1.0 : 2.2)
                                    : (ls[i] <= 8 ? 1.0 : 1.0 + 0.15 * (ls[i] - 8));
        cost += f * pass_tb / bw_r(level_chunk_bytes(ls[i], I)) + pass_fixed;
      }
    }
    if (cost < best * (1.0 - 1e-9)) { best = cost; bm = m; bl[0] = a; bl[1] = b; bl[2] = c; }
  };
  if (n <= hi) consider(1, n, 0, 0);
  for (int a = 1; a <= hi && a < n; ++a) {
    if (n - a <= hi) consider(2, a, n - a, 0);
    for (int b = 1; b <= hi && a + b < n; ++b)
      if (n - a - b <= hi) consider(3, a, b, n - a - b);
  }
  if (bm == 0) return 0;
  for (int i = 0; i < 3; ++i) l[i] = bl[i];
  return bm;
}

template <int MODE, bool FAST, bool SIGNINV>
static cudaError_t launch_variant(const Pass& ps, cudaStream_t st) {
  auto kern = pass_kernel<MODE, FAST, SIGNINV>;
  static bool attr_done[16] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 16 && !attr_done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         200 * 1024);
    if (e != cudaSuccess) return e;
    attr_done[dev] = true;
  }
  return pdl_launch(kern, dim3(ps.grid), dim3(kThreads), ps.smem, st, ps.a);
}

static cudaError_t launch_pass(const Pass& ps, bool fast, cudaStream_t st) {
  switch (ps.mode) {
    case MODE_FWD:
      if (ps.signinv) return fast ? launch_variant<MODE_FWD, true, true>(ps, st)
                                  : launch_variant<MODE_FWD, false, true>(ps, st);
      return fast ? launch_variant<MODE_FWD, true, false>(ps, st)
                  : launch_variant<MODE_FWD, false, false>(ps, st);
    case MODE_MID:
      return fast ? launch_variant<MODE_MID, true, false>(ps, st)
                  : launch_variant<MODE_MID, false, false>(ps, st);
    default:
      return fast ? launch_variant<MODE_INV, true, false>(ps, st)
                  : launch_variant<MODE_INV, false, false>(ps, st);
  }
}

// ------------------------------------------------------------------------------------------
// fast-kernel dispatch (instantiations in pbk_fast_r8.cu / pbk_fast_r16.cu)
// ------------------------------------------------------------------------------------------
namespace pbk {
// one family is built: radix-16 stages, <= 128 registers per thread.  (A radix-8 / 64-register /
// 512-thread family was measured 4-8 % slower on every configuration and was removed.)
bool fast_info_r16(int log2L, FastInfo* info);
void fast_tables_r16(int log2L, float2* dst);
cudaError_t fast_launch_r16(int log2L, int mode, const PassArgs& a, const float2* d_tables,
                            long long ntiles, int num_sms, cudaStream_t st);
// ... plus half-width 2^8-point tiles for the detecting last pass of a channelizer plan
void fast_info_l8n(FastInfo* info);
void fast_tables_l8n(float2* dst);
cudaError_t fast_launch_l8n(int mode, const PassArgs& a, const float2* d_tables, long long ntiles,
                            int num_sms, cudaStream_t st);
bool fast_info(int family, int log2L, FastInfo* info) {
  if (family == FAMILY_R16N) {
    if (log2L != 8) return false;
    fast_info_l8n(info);
    return true;
  }
  return fast_info_r16(log2L, info);
}
void fast_tables(int family, int log2L, float2* dst) {
  if (family == FAMILY_R16N) fast_tables_l8n(dst);
  else fast_tables_r16(log2L, dst);
}
cudaError_t fast_launch(int family, int log2L, int mode, const PassArgs& a, const float2* d_tables,
                        long long ntiles, int num_sms, cudaStream_t st) {
  if (family == FAMILY_R16N) return fast_launch_l8n(mode, a, d_tables, ntiles, num_sms, st);
  return fast_launch_r16(log2L, mode, a, d_tables, ntiles, num_sms, st);
}
}  // namespace pbk

// developer knob: PBK_FAMILY=0 forces the generic runtime-shaped kernels everywhere
static int preferred_family() {
  const char* e = getenv("PBK_FAMILY");
  if (e && !strcmp(e, "0")) return -1;
  return FAMILY_R16;
}

// decide which passes can run on the compile-time-shaped kernels and stage their tables
static int setup_fast(pbk_plan* pl) {
  const int fam = preferred_family();
  std::vector<float2> host;
  for (auto& ps : pl->passes) {
    ps.family = -1;
    if (fam < 0 || !ps.pair_ok) continue;
    if (ps.signinv && (ps.mode != MODE_FWD || pl->kind != PLAN_FFT)) continue;
    if (ps.signinv && load_is_raw(ps.a.load_kind)) continue;
    // the fast kernels are specialised to the dedispersion passes (see pbk_fast.cuh) plus the
    // last pass of a forward FFT / STFT plan (FWD-last: no level twiddle, scale, fftshift)
    const bool fwd_last = ps.mode == MODE_FWD && ps.a.log2M == 0 && ps.out_role == ROLE_USER_OUT &&
                          pl->kind == PLAN_FFT && !load_is_raw(ps.a.load_kind);
    if (ps.a.kxor && !fwd_last) continue;
    // ifftshift on the load rows (ISTFT first pass) is only done by the transposed loader, whose
    // tile is a whole level: single-level plans whose lane pairs own contiguous runs of rows
    const bool in_rows_contig = ps.a.min.a_row == 2 && ps.a.P == 2 && ps.a.min.a_p == 1 &&
                                ps.in_role == ROLE_USER_IN && ps.a.load_kind == LOAD_C64;
    if (ps.a.fxor && !(fwd_last && in_rows_contig)) continue;
    if (ps.a.scale != 1.0f && ps.mode != MODE_MID && !fwd_last) continue;
    if (ps.mode != MODE_MID && ps.a.log2M == 0 && !fwd_last) continue;
    if (ps.mode == MODE_MID && (ps.a.chirp_kind != CHIRP_COMPUTED || load_is_raw(ps.a.load_kind) ||
                                !pl->chirp_series_ok))
      continue;
    if (ps.mode != MODE_FWD && ps.in_role == ROLE_SCRATCH && ps.a.load_kind != LOAD_PLANAR) continue;
    if (ps.out_role == ROLE_SCRATCH && !ps.a.store_planar) continue;
    FastInfo fi;
    if (!fast_info(fam, ps.a.log2L, &fi)) continue;
    const long long W = 2ll << fi.log2pw;
    // a tile is W adjacent lanes: inside one row of the (.., I) array (I % W == 0), or, for arrays
    // with few channels, W / I whole rows (consecutive time offsets / consecutive kprev blocks)
    const bool wide = ps.a.I % W == 0 && W % ps.a.P == 0;
    // (last-level passes -- MID, FWD-last -- have RI == I: their tiles then span W / I consecutive
    // kprev blocks, which must not run over into the next outer block)
    const bool lastlevel = ps.mode == MODE_MID || fwd_last;
    const bool narrow = ps.a.I < W && W % ps.a.I == 0 && ps.a.I % 2 == 0 &&
                        (lastlevel ? (1ll << ps.a.log2Kprev) % (W / ps.a.I) == 0
                                   : ps.a.RI % W == 0);
    if (!(wide || narrow) || ps.a.Q % W) continue;
    if (fwd_last) {
      // output addressing: either the lane pair is adjacent in the output and rows are strided
      // (plain FFT, multi-level STFT of few channels), or every pair owns a contiguous run of rows
      // (single-level STFT: transposed through shared memory)
      const AddrMap& mo = ps.a.mout;
      const bool rows_contig = mo.a_row == 2 && ps.a.P == 2 && mo.a_p == 1;
      if (mo.a_row * 8 >= (1ll << 32)) continue;
      ps.a.out_transpose = (rows_contig && !narrow) ? 1 : 0;
      ps.a.final_epi = 1;
      ps.a.epi_kind = EPI_C64;
      if (in_rows_contig && ps.a.min.a_c != ps.a.P) {   // ISTFT input: pairs far apart
        if (narrow) continue;
        ps.fast_load_transposed = true;
      }
    } else if (in_rows_contig && ps.a.min.a_c != ps.a.P) {
      continue;   // would need the transposed loader in a non-final pass
    }
    if (ps.a.min.a_row * 8 >= (1ll << 32) || ps.a.mout.a_row * 8 >= (1ll << 32)) continue;
    ps.family = fam;
    ps.finfo = fi;
    ps.ntiles = ps.a.Q / W;
    ps.ftab_off = host.size();
    host.resize(host.size() + fi.tw_count + (fi.tw_count & 1));
    fast_tables(fam, ps.a.log2L, host.data() + ps.ftab_off);
  }
  if (!host.empty()) {
    CUDA_TRY(cudaMalloc(&pl->d_ftab, host.size() * sizeof(float2)));
    CUDA_TRY(cudaMemcpy(pl->d_ftab, host.data(), host.size() * sizeof(float2),
                        cudaMemcpyHostToDevice));
  }
  CUDA_TRY(cudaDeviceGetAttribute(&pl->num_sms, cudaDevAttrMultiProcessorCount, pl->device));
  return PBK_OK;
}


// ------------------------------------------------------------------------------------------
// TMA-pipelined passes (pbk_tma.cuh)
// ------------------------------------------------------------------------------------------
// Which passes use the TMA kernels.  $PBK_TMA = 0: none; unset: the (kind, tile length) pairs that
// measured at least as fast as the LDG kernels on B200 (profiles/r02_tma_vs_ldg_passes.log -- both
// variants produce bit-identical results, so this is purely a speed choice); 1: every eligible
// pass; or a list of kinds "tsum,inv,fwd,mid,final" (final = last inverse pass without a time
// sum) to force those kinds at every length.
static bool tma_kind_enabled(const char* kind, int log2L) {
  const char* e = getenv("PBK_TMA");
  if (e && !strcmp(e, "0")) return false;
  if (e && !strcmp(e, "1")) return true;
  if (e) {
    const size_t n = strlen(kind);
    for (const char* q = e; (q = strstr(q, kind)) != nullptr; q += n)
      if ((q == e || q[-1] == ',') && (q[n] == 0 || q[n] == ',')) return true;
    return false;
  }
  // measured on cfg2 / cfg3-shard sized arrays, LDG -> TMA per pass:
  //   fwd   l6 0.373->0.366  l7 1.488->1.439  l8 1.447->1.416  l9 1.910->1.884 ms
  //   inv   l7 1.478->1.473  l8 1.431->1.433  (l6 0.363->0.369)
  //   mid   l6 1.537->1.522 (whole cfg2 step, passes back to back: 6.877->6.765)  l8 1.863->1.599
  //         l10 5.41->4.25  (with the group runs in registers / shared memory, pbk_tma.cuh; with
  //         them in local memory l6 and l7 lost: 1.500->1.606, 0.410->0.440)
  //   tsum  l8 0.963->0.963  l9 1.203->1.184  (l7 0.906->1.050)
  //   final l7 1.498->1.454  l8 1.414->1.412  (l9 1.894->1.914)
  if (!strcmp(kind, "fwd")) return true;
  if (!strcmp(kind, "inv")) return log2L >= 7;
  if (!strcmp(kind, "mid")) return true;
  if (!strcmp(kind, "tsum")) return log2L >= 8;
  if (!strcmp(kind, "final")) return log2L == 7 || log2L == 8;
  return false;
}

typedef CUresult (*TensorMapEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                      const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                      const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static TensorMapEncodeFn tensor_map_encoder() {
  static TensorMapEncodeFn fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess)
      f = nullptr;
    cudaGetLastError();
    return reinterpret_cast<TensorMapEncodeFn>(f);
  }();
  return fn;
}

// rank-4 float32 view of a pass input: (2 I floats | R inner time offsets | L tile rows | blocks),
// box = one tile's rows (at most 256 per box) x 2 W floats.  See pbk_tma.cuh: issue().
static bool tma_encode(const Pass& ps, const void* base, CUtensorMap* tm) {
  TensorMapEncodeFn enc = tensor_map_encoder();
  if (!enc) return false;
  const PassArgs& a = ps.a;
  const cuuint64_t I = (cuuint64_t)a.I, RI = (cuuint64_t)a.RI, L = 1ull << a.log2L;
  static const int promo = [] {
    const char* e = getenv("PBK_TMA_L2PROMO");
    return e ? atoi(e) : 0;
  }();
  const CUtensorMapL2promotion l2p = promo == 256 ? CU_TENSOR_MAP_L2_PROMOTION_L2_256B
                                   : promo == 128 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B
                                   : promo == 64  ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B
                                                  : CU_TENSOR_MAP_L2_PROMOTION_NONE;
  const cuuint64_t dims[4] = {2 * I, RI / I, L, (cuuint64_t)(a.Q / a.RI)};
  const cuuint64_t strides[3] = {I * 8, RI * 8, L * RI * 8};
  const cuuint32_t box[4] = {(cuuint32_t)(4u << ps.tinfo.log2pw), 1, (cuuint32_t)ps.tinfo.box_rows, 1};
  const cuuint32_t es[4] = {1, 1, 1, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void*>(base), dims, strides, box,
             es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, l2p,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// decide which fast passes run on the TMA-pipelined kernels (called after setup_fast and after the
// fused time sum has been chosen)
static void setup_tma(pbk_plan* pl) {
  if (!tensor_map_encoder()) return;
  const char* only = getenv("PBK_TMA_PASS");     // developer knob: TMA on this pass index only
  int idx = -1;
  for (auto& ps : pl->passes) {
    ps.tma = false;
    ++idx;
    if (only && atoi(only) != idx) continue;
    if (ps.family < 0 || ps.signinv || ps.fast_load_transposed) continue;
    const PassArgs& a = ps.a;
    TmaInfo ti;
    if (!tma_info(a.log2L, &ti) || ti.log2pw != ps.finfo.log2pw) continue;
    if (ti.mid_only && ps.mode != MODE_MID) continue;
    // 2^10-point MID tiles: 1.348 -> 1.209 ms (32768 tiles), 5.41 -> 4.85 ms (131072 tiles), but
    // 0.053 -> 0.059 ms at 1024 tiles, where one 512-thread CTA per SM leaves SMs idle
    if (ti.mid_only && ps.ntiles < 4096 && !getenv("PBK_TMA")) continue;
    const long long W = 2ll << ti.log2pw, L = 1ll << a.log2L;
    if (a.I % W || W % a.P || a.Q % W) continue;                 // wide tiles only
    const bool planar_in = ps.in_role == ROLE_SCRATCH && a.load_kind == LOAD_PLANAR;
    const bool c64_in = ps.in_role == ROLE_USER_IN && a.load_kind == LOAD_C64 && ps.mode == MODE_FWD;
    if (!planar_in && !c64_in) continue;
    if (ps.mode == MODE_FWD && (a.final_epi || ps.out_role != ROLE_SCRATCH)) continue;
    if (ps.mode == MODE_MID && (a.final_epi || a.split)) continue;
    if (a.fxor || a.kxor || a.scale != 1.0f && ps.mode != MODE_MID) continue;
    // the input must be the plain (blocks, L, R, I) array the tensor map describes
    const AddrMap& m = a.min;
    if (m.a_n != a.I || m.a_row != a.RI || m.a_kp != L * a.RI || m.a_c != a.P || m.a_p != 1 ||
        !(m.a_o == 0 || m.a_o == (L * a.RI) << a.log2Kprev))
      continue;
    if (a.Q / a.RI >= (1ll << 31) || 2ll * a.I >= (1ll << 32)) continue;
    const bool tsum = ps.mode == MODE_INV && a.tsum_log2 > 0;
    if (tsum && !ti.tsum_ok) continue;
    // a time-summing pass has at most (tiles / q) >> (log2 M + 1) runs of tiles (a run spans two
    // groups of summed rows); when that is fewer than two per SM, one 512-thread CTA per SM
    // leaves SMs idle that the 256-thread CTAs of the LDG kernel would use (2^20 x 64 lanes, M = 64:
    // 0.38 ms LDG, 0.57 ms TMA)
    if (tsum && !getenv("PBK_TMA") &&
        ((ps.ntiles / a.tsum_q) >> (a.tsum_log2 + 1)) * a.tsum_q < 2ll * pl->num_sms)
      continue;
    const char* kind = ps.mode == MODE_FWD ? "fwd" : ps.mode == MODE_MID ? "mid"
                       : tsum ? "tsum" : a.final_epi ? "final" : "inv";
    if (!tma_kind_enabled(kind, a.log2L)) continue;
    ps.tma = true;
    ps.tinfo = ti;
  }
}

static int upload_tables(pbk_plan* pl, TableSet& ts) {
  if (ts.host.empty()) ts.host.push_back(make_float2(1.f, 0.f));
  CUDA_TRY(cudaMalloc(&pl->d_tw, ts.host.size() * sizeof(float2)));
  CUDA_TRY(cudaMemcpy(pl->d_tw, ts.host.data(), ts.host.size() * sizeof(float2),
                      cudaMemcpyHostToDevice));
  for (auto& ps : pl->passes) {
    ps.a.stage_tw = pl->d_tw;
    for (int s = 0; s < kMaxStages; ++s) ps.a.stage_tw_off[s] = ts.off_by_log2L[ps.a.log2L][s];
  }
  return PBK_OK;
}

static void blue_free(BlueState* b);
static int blue_exec(pbk_plan* pl, const void* d_in, void* d_out, const void* d_chirp,
                     cudaStream_t st, int trial = -1);

// scratch arrays are pair-planar ({re0,re1,im0,im1} per 16-byte lane pair) when the innermost
// extent is even; every pass, generic or fast, reads and writes them through that layout
static void mark_scratch_layout(pbk_plan* pl, long long I) {
  const bool planar = (I % 2 == 0);
  for (auto& ps : pl->passes) {
    if (planar && ps.in_role == ROLE_SCRATCH) ps.a.load_kind = LOAD_PLANAR;
    ps.a.store_planar = (planar && ps.out_role == ROLE_SCRATCH) ? 1 : 0;
  }
}

// ------------------------------------------------------------------------------------------
// dedispersion plan
// ------------------------------------------------------------------------------------------
struct RampSpec {   // linear-phase / band-zeroing transfer function per column (CHIRP_RAMP)
  const double* shift_samples;
  const int64_t* zero_lo;
  const int64_t* zero_hi;
  int flags;   // PBK_RAMP_HILBERT, PBK_RAMP_REAL_INPUT
};

static int load_kind_of(int in_dtype) {
  switch (in_dtype) {
    case PBK_I8X2: return LOAD_I8X2;
    case PBK_U4X2: return LOAD_U4X2;
    case PBK_U2X2: return LOAD_U2X2;
    case PBK_F32: return LOAD_F32;
    default: return LOAD_C64;
  }
}

// trial DMs of a trial plan; a single-DM plan passes {&desc->dm, 1, false}
struct TrialSpec {
  const double* dms;
  int ndm;
  bool trials;
};

static int dedisp_plan_create_impl(const pbk_dedisp_desc* d, const RampSpec* ramp,
                                   const TrialSpec& tr, pbk_plan** out);
static int blue_dedisp_plan_create(const pbk_dedisp_desc* d, const RampSpec* ramp, pbk_plan** out);

// PassArgs::D of the chirp, dedispersion.py:30,46 in Hz^2 s
static double chirp_D(double dm) { return (1.0 / 2.41e-4) * dm * 1e12; }

// per-column ramp description (shift / N, zeroed band) on the device, owned by the plan
static int upload_ramp(pbk_plan* pl, const RampSpec* ramp, long long C, long long N) {
  std::vector<double> sh((size_t)C);
  std::vector<long long> zr((size_t)C * 2);
  for (long long c = 0; c < C; ++c) {
    sh[c] = (ramp->shift_samples ? ramp->shift_samples[c] : 0.0) / (double)N;
    zr[2 * c] = ramp->zero_lo ? ramp->zero_lo[c] : 0;
    zr[2 * c + 1] = ramp->zero_hi ? ramp->zero_hi[c] : 0;
  }
  CUDA_TRY(cudaMalloc(&pl->d_ramp_shift, sh.size() * sizeof(double)));
  CUDA_TRY(cudaMalloc(&pl->d_ramp_zero, zr.size() * sizeof(long long)));
  CUDA_TRY(cudaMemcpy(pl->d_ramp_shift, sh.data(), sh.size() * sizeof(double),
                      cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(pl->d_ramp_zero, zr.data(), zr.size() * sizeof(long long),
                      cudaMemcpyHostToDevice));
  return PBK_OK;
}

extern "C" int pbk_dedisp_plan_create(const pbk_dedisp_desc* d, pbk_plan** out) {
  if (!d) return fail(PBK_ERR_INVALID, "NULL argument");
  return dedisp_plan_create_impl(d, nullptr, TrialSpec{&d->dm, 1, false}, out);
}

extern "C" int pbk_dedisp_trials_plan_create(const pbk_dedisp_desc* d, const double* dms,
                                             int32_t ndm, pbk_plan** out) {
  if (!d || !out || !dms) return fail(PBK_ERR_INVALID, "NULL argument");
  *out = nullptr;
  if (ndm < 1) return fail(PBK_ERR_INVALID, "ndm must be >= 1, got %d", (int)ndm);
  if (d->explicit_chirp) return fail(PBK_ERR_INVALID, "trial plans generate their chirps");
  for (int k = 0; k < ndm; ++k)
    if (!std::isfinite(dms[k])) return fail(PBK_ERR_INVALID, "trial DM %d is not finite", k);
  pbk_dedisp_desc h = *d;
  h.dm = dms[0];
  return dedisp_plan_create_impl(&h, nullptr, TrialSpec{dms, (int)ndm, true}, out);
}

extern "C" int pbk_plan_trials(const pbk_plan* pl, int32_t* ndm) {
  if (!pl || !ndm) return fail(PBK_ERR_INVALID, "NULL argument");
  *ndm = pl->ndm;
  return PBK_OK;
}

extern "C" int pbk_ramp_plan_create(int64_t nsamp, int64_t ncols, const double* shift_samples,
                                    const int64_t* zero_lo, const int64_t* zero_hi,
                                    int32_t flags, int32_t device, pbk_plan** plan) {
  if (!plan) return fail(PBK_ERR_INVALID, "plan is NULL");
  if (nsamp <= 0 || ncols <= 0) return fail(PBK_ERR_INVALID, "shape must be positive");
  std::vector<double> freqs((size_t)ncols, 1.0);
  pbk_dedisp_desc d;
  memset(&d, 0, sizeof(d));
  d.nsamp = nsamp;
  d.nchan = ncols;
  d.npol = 1;
  d.in_dtype = (flags & PBK_RAMP_REAL_INPUT) ? PBK_F32 : PBK_C64;
  d.out_kind = PBK_OUT_C64;
  d.dm = 0.0;
  d.sample_rate_hz = 1.0;
  d.ref_freq_hz = 1.0;
  d.chan_freq_hz = freqs.data();
  d.crop_start = 0;
  d.crop_stop = nsamp;
  d.downsample = 1;
  d.device = device;
  RampSpec r{shift_samples, zero_lo, zero_hi, flags};
  return dedisp_plan_create_impl(&d, &r, TrialSpec{&d.dm, 1, false}, plan);
}

// Executions per launch: the trials of a trial plan, or the overlap-save blocks of a single-DM
// plan (pbk_dedisp_exec_blocks_device).  A pass of a small block has fewer tiles than the GPU holds
// CTAs (one 2^20-sample column: 128 tiles on 148 SMs), so T executions of the batched passes
// [first, end) run as one launch with gridDim.y = T: just enough for two waves of resident CTAs in
// every batched pass, at most `limit`, and bounded by the memory of T scratch slabs in each of the
// `nbuf` batched scratch arrays (together within the 1/5-of-device rule of the second scratch
// array).  Only the LDG fast kernels take a batch index; a batched pass on the generic or TMA
// kernels, a Bluestein length, a one-level plan (a trial's MID pass would read the caller's
// input), an output staged through d_tmpf and a slab that is not a multiple of 16 bytes keep T = 1.
static int choose_per_launch(const pbk_plan* pl, size_t first, long long limit, int nbuf) {
  if (pl->blue || pl->nlevels < 2 || pl->split_ragged ||
      pl->out_bytes % 16 || pl->passes.back().out_role != ROLE_USER_OUT)
    return 1;
  long long want = 1;
  for (size_t i = first; i < pl->passes.size(); ++i) {
    const Pass& ps = pl->passes[i];
    if (ps.family < 0 || ps.tma || ps.ntiles <= 0) return 1;
    const long long resident = (long long)pl->num_sms * ps.finfo.minb;
    want = std::max(want, (2 * resident + ps.ntiles - 1) / ps.ntiles);
  }
  size_t free_b = 0, total_b = 0;
  if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) {
    cudaGetLastError();
    return 1;
  }
  long long T = std::min<long long>(want, limit);
  while (T > 1 && (size_t)T * nbuf * pl->scratch_bytes > total_b / 5) --T;
  return (int)T;
}

// Blocks per launch of a single-DM plan: every pass is batched, in the plan's scratch arrays
// (both of a ping-pong pair), up to the grid's y limit.
static void set_blocks_per_launch(pbk_plan* pl) {
  pl->blocks_per_launch = choose_per_launch(pl, 0, 65535, pl->scratch2 ? 2 : 1);
}

// the trial fields of a plan whose passes (or Bluestein state) are built: trials per launch, the
// per-trial scratch slabs, launch and segment counts for the trial schedule (see run_trial_passes)
static int set_trials(pbk_plan* pl, const TrialSpec& tr) {
  pl->trials = true;
  pl->ndm = tr.ndm;
  pl->trial_D.resize(tr.ndm);
  for (int k = 0; k < tr.ndm; ++k) pl->trial_D[k] = chirp_D(tr.dms[k]);
  if (pl->blue) {
    pl->launches *= tr.ndm;
    return PBK_OK;
  }
  const int ds = (pl->desc.downsample > 1 && !pl->fused_tsum) ? 1 : 0;
  pl->nshared = pl->nlevels - 1;
  pl->trials_per_launch = choose_per_launch(pl, pl->nshared, pl->ndm, 1);
  if (pl->nshared > 0) {
    // the per-trial passes work in buffer nshared & 1 of the ping-pong pair
    void*& work = (pl->nshared & 1) ? pl->scratch2 : pl->scratch;
    if (pl->work_bytes == 0) pl->work_bytes = pl->scratch_bytes;
    const size_t need = (size_t)pl->trials_per_launch * pl->scratch_bytes;
    if (need > pl->work_bytes) {
      cudaFree(work);
      work = nullptr;
      pl->work_bytes = 0;
      CUDA_TRY(cudaMalloc(&work, need));
      pl->work_bytes = need;
    }
  }
  const int per = (int)pl->passes.size() - pl->nshared + ds;
  const int batches = (tr.ndm + pl->trials_per_launch - 1) / pl->trials_per_launch;
  pl->launches = pl->nshared + batches * per;
  pl->segments = pl->launches;
  return PBK_OK;
}

static int dedisp_plan_create_impl(const pbk_dedisp_desc* d, const RampSpec* ramp,
                                   const TrialSpec& tr, pbk_plan** out) {
  if (!d || !out) return fail(PBK_ERR_INVALID, "NULL argument");
  *out = nullptr;
  if (d->nsamp <= 0 || d->nchan <= 0 || d->npol <= 0)
    return fail(PBK_ERR_INVALID, "shape must be positive");
  if (!d->chan_freq_hz) return fail(PBK_ERR_INVALID, "chan_freq_hz is NULL");
  if (!(d->sample_rate_hz > 0)) return fail(PBK_ERR_INVALID, "sample_rate_hz must be > 0");
  if (d->in_dtype != PBK_C64 && d->in_dtype != PBK_I8X2 && d->in_dtype != PBK_U4X2 &&
      d->in_dtype != PBK_U2X2 && !(ramp && d->in_dtype == PBK_F32))
    return fail(PBK_ERR_INVALID, "unknown in_dtype %d", d->in_dtype);
  if ((d->in_dtype == PBK_U4X2 || d->in_dtype == PBK_U2X2) && (d->nchan * d->npol) % 2)
    return fail(PBK_ERR_INVALID, "packed input needs an even nchan * npol, got %lld",
                (long long)(d->nchan * d->npol));
  if (d->out_kind < PBK_OUT_C64 || d->out_kind > PBK_OUT_STOKES_I)
    return fail(PBK_ERR_INVALID, "unknown out_kind %d", d->out_kind);
  if (d->out_kind == PBK_OUT_STOKES_I && d->npol != 2)
    return fail(PBK_ERR_INVALID, "Stokes I needs npol == 2, got %lld", (long long)d->npol);
  if (d->downsample < 1) return fail(PBK_ERR_INVALID, "downsample must be >= 1");
  if (d->downsample > 1 && d->out_kind == PBK_OUT_C64)
    return fail(PBK_ERR_INVALID, "downsample applies to float outputs only");
  if (d->crop_start < 0 || d->crop_stop > d->nsamp)
    return fail(PBK_ERR_INVALID, "crop [%lld, %lld) outside [0, %lld]", (long long)d->crop_start,
                (long long)d->crop_stop, (long long)d->nsamp);
  const int n = ilog2_exact(d->nsamp);
  // ONE complex64 column (a BasebandSignal with a single channel, BASELINE config 1) has no lane
  // pairs for the compile-time-shaped kernels.  Its even and odd samples do: the (N/2, 2) view of
  // the same memory is a two-"channel" single-pol array, transformed at half length by the fast
  // kernels, with the radix-2 recombination, the chirp at bins k and k - N/2 and the inverse
  // split done in registers by the middle pass (pbk_fast.cuh: fast_chirp, p.split).
  if (!ramp && n >= 13 && d->nchan == 1 && d->npol == 1 && d->in_dtype == PBK_C64 &&
      !d->explicit_chirp && d->downsample == 1 && d->out_kind != PBK_OUT_STOKES_I &&
      d->crop_stop >= d->crop_start &&
      std::fabs(d->chan_freq_hz[0]) >= 8.0 * d->sample_rate_hz && !getenv("PBK_NO_SPLIT")) {
    pbk_dedisp_desc h = *d;
    const double f2[2] = {d->chan_freq_hz[0], d->chan_freq_hz[0]};
    h.nsamp = d->nsamp / 2;
    h.nchan = 2;
    h.sample_rate_hz = d->sample_rate_hz / 2;   // same bin width: df = (SR/2) / (N/2)
    h.chan_freq_hz = f2;
    h.crop_start = d->crop_start / 2;           // whole (even, odd) rows covering the crop
    h.crop_stop = (d->crop_stop + 1) / 2;
    pbk_plan* pl = nullptr;
    const int rc = dedisp_plan_create_impl(&h, nullptr, tr, &pl);
    if (rc == PBK_OK) {
      bool all_fast = true;
      for (auto& ps : pl->passes) all_fast = all_fast && ps.family >= 0;
      if (all_fast) {
        for (auto& ps : pl->passes)
          if (ps.mode == MODE_MID) { ps.a.split = 1; ps.a.scale *= 0.5f; }
        pl->desc = *d;                          // report the caller's geometry
        pl->desc.chan_freq_hz = nullptr;
        const bool ragged = (d->crop_start | d->crop_stop) & 1;
        const size_t rows_bytes = pl->out_bytes;   // whole rows of the half-length view
        pl->out_rows = pl->full_rows = d->crop_stop - d->crop_start;
        pl->row_elems = 1;
        pl->out_bytes = (size_t)pl->out_rows * pl->elem_bytes;
        pl->split_column = true;
        if (ragged && pl->out_rows > 0) {
          // a crop edge inside a row: the passes write whole rows to a plan-owned buffer and the
          // requested samples are copied out (device to device, at most 8 bytes skipped)
          pl->split_skip = (size_t)(d->crop_start & 1) * pl->elem_bytes;
          pl->tmpf_bytes = rows_bytes;
          cudaError_t e = cudaMalloc(&pl->d_tmpf, pl->tmpf_bytes);
          if (e != cudaSuccess) {
            pbk_plan_destroy(pl);
            return fail(PBK_ERR_NOMEM, "split buffer (%zu bytes): %s", rows_bytes,
                        cudaGetErrorString(e));
          }
          pl->split_ragged = true;
        }
        int rs;
        if (tr.trials && (rs = set_trials(pl, tr)) != PBK_OK) {   // again, for this geometry
          pbk_plan_destroy(pl);
          return rs;
        }
        if (!tr.trials) set_blocks_per_launch(pl);             // again, for this geometry
        *out = pl;
        return PBK_OK;
      }
      pbk_plan_destroy(pl);                     // no fast coverage for this shape: generic path
    }
  }
  if (n < 4) {
    // not a power of two (or shorter than 16): Bluestein on top of the power-of-two passes
    if (d->nsamp < 2)
      return fail(PBK_ERR_UNSUPPORTED, "nsamp = %lld is too short", (long long)d->nsamp);
    const int rc = blue_dedisp_plan_create(d, ramp, out);
    if (rc == PBK_OK && tr.trials) set_trials(*out, tr);   // the whole execution runs per trial
    return rc;
  }
  int l[3] = {0, 0, 0};
  const long long I = d->nchan * d->npol;
  const int m = choose_levels(n, I, l, true);
  if (m == 0) return fail(PBK_ERR_UNSUPPORTED, "nsamp = 2^%d is too long", n);
  if (I > INT_MAX / 2) return fail(PBK_ERR_UNSUPPORTED, "nchan*npol too large");

  int ndev = 0;
  CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (d->device < 0 || d->device >= ndev)
    return fail(PBK_ERR_CUDA, "device %d not available (%d CUDA devices)", d->device, ndev);
  CUDA_TRY(cudaSetDevice(d->device));

  pbk_plan* pl = new pbk_plan();
  pl->kind = PLAN_DEDISP;
  pl->device = d->device;
  pl->desc = *d;
  pl->desc.chan_freq_hz = nullptr;
  pl->nlevels = m;
  for (int i = 0; i < m; ++i) pl->level_log2[i] = l[i];

  const long long N = d->nsamp;
  const int P = (int)d->npol;
  const long long C = d->nchan;
  const long long crop_rows = std::max<long long>(0, d->crop_stop - d->crop_start);
  pl->full_rows = crop_rows;
  pl->out_rows = d->downsample > 1 ? crop_rows / d->downsample : crop_rows;
  pl->row_elems = d->out_kind == PBK_OUT_STOKES_I ? C : I;
  pl->elem_bytes = d->out_kind == PBK_OUT_C64 ? 8 : 4;
  pl->in_bytes = ((size_t)N * I * load_bits(load_kind_of(d->in_dtype))) >> 3;
  pl->out_bytes = (size_t)pl->out_rows * pl->row_elems * pl->elem_bytes;
  pl->chirp_bytes = d->explicit_chirp ? (size_t)N * C * 8 : 0;

  TableSet ts;
  const bool fast_ok = (I % 2 == 0) && (P % 2 == 0);
  const bool pair_ok = (I % 2 == 0) && (P % 2 == 0 || P == 1);
  long long Kprev[3], R[3];
  {
    long long k = 1;
    for (int i = 0; i < m; ++i) { Kprev[i] = k; k <<= l[i]; }
    long long r = 1;
    for (int i = m - 1; i >= 0; --i) { R[i] = r; r <<= l[i]; }
  }
  auto log2ll = [](long long v) { int s = 0; while ((1ll << s) < v) ++s; return s; };

  auto final_epilogue = [&](Pass& ps, int level0) {
    PassArgs& a = ps.a;
    a.epi_kind = d->out_kind;
    a.crop_start = d->crop_start;
    a.crop_stop = d->crop_stop;
    a.n_mul = R[level0];
    a.log2nmul = log2ll(R[level0]);
    a.final_epi = 1;
    if (d->out_kind == PBK_OUT_STOKES_I) {
      a.mout.a_o = 0; a.mout.a_kp = 0; a.mout.a_kl = 0;
      a.mout.a_n = C; a.mout.a_c = 1; a.mout.a_p = 0; a.mout.a_row = R[level0] * C;
    }
    ps.out_role = d->downsample > 1 ? ROLE_TMPF : ROLE_USER_OUT;
  };

  // forward levels 1..m-1
  for (int i = 0; i + 1 < m; ++i) {
    Pass ps;
    defaults(ps.a);
    ps.mode = MODE_FWD;
    set_geometry(ps, l[i], Kprev[i] * R[i] * I, R[i] * I, (int)I, P, log2ll(Kprev[i]));
    ps.a.min = plain_map(1ll << l[i], R[i], I, P);
    ps.a.mout = ps.a.min;
    ps.a.log2M = l[i] + log2ll(R[i]);
    set_klow(ps.a, i + 1, l);
    ps.in_role = i == 0 ? ROLE_USER_IN : ROLE_SCRATCH;
    ps.out_role = ROLE_SCRATCH;
    if (i == 0)
      ps.a.load_kind = load_kind_of(d->in_dtype);
    ps.fast = fast_ok;
    ps.pair_ok = pair_ok;
    ts.ensure(l[i]);
    pl->passes.push_back(ps);
  }
  // middle
  {
    const int i = m - 1;
    Pass ps;
    defaults(ps.a);
    ps.mode = MODE_MID;
    set_geometry(ps, l[i], Kprev[i] * I, I, (int)I, P, log2ll(Kprev[i]));
    ps.a.min = plain_map(1ll << l[i], 1, I, P);
    ps.a.mout = ps.a.min;
    set_klow(ps.a, i + 1, l);
    ps.a.log2Kmul = log2ll(Kprev[i]);
    ps.a.chirp_kind = ramp ? CHIRP_RAMP : d->explicit_chirp ? CHIRP_ARRAY : CHIRP_COMPUTED;
    ps.a.N = N;
    {
      const double dt = 1.0 / d->sample_rate_hz;      // Signal.dt, core.py:250-253
      ps.a.df = 1.0 / ((double)N * dt);               // numpy fftfreq: val = 1/(n*d)
      if (std::isinf(d->ref_freq_hz)) { ps.a.fr_sub = 0; ps.a.inv_fr = 0; ps.a.a0 = -1.0; }
      else { ps.a.fr_sub = d->ref_freq_hz; ps.a.inv_fr = 1.0 / d->ref_freq_hz; ps.a.a0 = 0; }
      ps.a.D = chirp_D(d->dm);
    }
    ps.a.scale = (float)(1.0 / (double)N);
    ps.a.chirp_sk = C;
    ps.a.chirp_sc = 1;
    ps.in_role = m == 1 ? ROLE_USER_IN : ROLE_SCRATCH;
    ps.out_role = ROLE_SCRATCH;
    if (m == 1) {
      ps.a.load_kind = load_kind_of(d->in_dtype);
      final_epilogue(ps, 0);
    }
    ps.fast = fast_ok;
    ps.pair_ok = pair_ok;
    ts.ensure(l[i]);
    pl->passes.push_back(ps);
  }
  // inverse levels m-1..1
  for (int i = m - 2; i >= 0; --i) {
    Pass ps;
    defaults(ps.a);
    ps.mode = MODE_INV;
    set_geometry(ps, l[i], Kprev[i] * R[i] * I, R[i] * I, (int)I, P, log2ll(Kprev[i]));
    ps.a.min = plain_map(1ll << l[i], R[i], I, P);
    ps.a.mout = ps.a.min;
    ps.a.log2M = l[i] + log2ll(R[i]);
    set_klow(ps.a, i + 1, l);
    ps.in_role = ROLE_SCRATCH;
    ps.out_role = ROLE_SCRATCH;
    if (i == 0) final_epilogue(ps, 0);
    ps.fast = fast_ok;
    ps.pair_ok = pair_ok;
    pl->passes.push_back(ps);
  }

  int rc = PBK_OK;
  auto cleanup = [&](int code) { pbk_plan_destroy(pl); return code; };
  mark_scratch_layout(pl, I);
  for (long long c = 0; c < C; ++c)   // the fast MID chirp needs |f - fc| <= |fc| / 16
    if (!(std::fabs(d->chan_freq_hz[c]) >= 8.0 * d->sample_rate_hz)) pl->chirp_series_ok = false;
  if ((rc = upload_tables(pl, ts)) != PBK_OK) return cleanup(rc);
  if ((rc = setup_fast(pl)) != PBK_OK) return cleanup(rc);
  {
    cudaError_t e = cudaMalloc(&pl->d_chanfreq, (size_t)C * sizeof(double));
    if (e == cudaSuccess)
      e = cudaMemcpy(pl->d_chanfreq, d->chan_freq_hz, (size_t)C * sizeof(double),
                     cudaMemcpyHostToDevice);
    if (e != cudaSuccess)
      return cleanup(fail(PBK_ERR_CUDA, "chan_freq upload: %s", cudaGetErrorString(e)));
  }
  if (m > 1) {
    pl->scratch_bytes = (size_t)N * I * 8;
    cudaError_t e = cudaMalloc(&pl->scratch, pl->scratch_bytes);
    if (e != cudaSuccess)
      return cleanup(fail(PBK_ERR_NOMEM, "scratch (%zu bytes): %s", pl->scratch_bytes,
                          cudaGetErrorString(e)));
  }
  // Time sum fused into the last inverse pass (fast_pass_kernel TSUM): power-of-two factor that
  // divides half the inner extent of the outermost level, wide tiles on the compile-time-shaped
  // kernels.
  if (d->downsample > 1 && pl->out_rows > 0 && m > 1 && !getenv("PBK_NO_FUSED_SUM")) {
    Pass& last = pl->passes.back();
    const int lm = ilog2_exact(d->downsample);
    const long long W = 2ll << last.finfo.log2pw;
    if (last.family >= 0 && last.mode == MODE_INV && lm > 0 && lm < last.a.log2nmul &&
        I % W == 0 && W % P == 0 &&
        last.finfo.tsum_ok) {
      last.a.tsum_log2 = lm;
      const long long ncg = I / W;   // column groups per row; q of them are read side by side
      last.a.tsum_q = ncg % 4 == 0 ? 4 : ncg % 2 == 0 ? 2 : 1;
      last.a.crop_stop = d->crop_start + pl->out_rows * d->downsample;
      last.out_role = ROLE_USER_OUT;
      pl->fused_tsum = true;
    }
  }
  if (d->downsample > 1 && crop_rows > 0 && !pl->fused_tsum) {
    pl->tmpf_bytes = (size_t)crop_rows * pl->row_elems * 4;
    cudaError_t e = cudaMalloc(&pl->d_tmpf, pl->tmpf_bytes);
    if (e != cudaSuccess)
      return cleanup(fail(PBK_ERR_NOMEM, "downsample buffer (%zu bytes): %s", pl->tmpf_bytes,
                          cudaGetErrorString(e)));
  }
  {
    // constants of the division-free chirp (pbk_fast.cuh: fast_chirp), in long double on the host;
    // a trial plan holds one table per trial DM, each computed as its single-DM plan computes it
    std::vector<double> cc((size_t)C * 3 * tr.ndm);
    const long double fr = d->ref_freq_hz, df = (long double)d->sample_rate_hz / (long double)N;
    for (int k = 0; k < tr.ndm; ++k) {
      const long double Dl = (1.0L / 2.41e-4L) * (long double)tr.dms[k] * 1e12L;
      double* t = cc.data() + (size_t)k * 3 * C;
      for (long long c = 0; c < C; ++c) {
        const long double fc = d->chan_freq_hz[c];
        t[3 * c + 0] = std::isinf(d->ref_freq_hz) ? -1.0 : (double)((fc - fr) / fr);
        t[3 * c + 1] = (double)(df / fc);
        t[3 * c + 2] = (double)(Dl / fc);
      }
    }
    pl->chanconst_stride = 3 * C;
    cudaError_t e = cudaMalloc(&pl->d_chanconst, cc.size() * sizeof(double));
    if (e == cudaSuccess)
      e = cudaMemcpy(pl->d_chanconst, cc.data(), cc.size() * sizeof(double),
                     cudaMemcpyHostToDevice);
    if (e != cudaSuccess)
      return cleanup(fail(PBK_ERR_CUDA, "chan_const upload: %s", cudaGetErrorString(e)));
  }
  if (ramp && (rc = upload_ramp(pl, ramp, C, N)) != PBK_OK) return cleanup(rc);
  for (auto& ps : pl->passes) {
    ps.a.ramp_hilbert = (ramp && (ramp->flags & PBK_RAMP_HILBERT)) ? 1 : 0;
    ps.a.ramp_shift = pl->d_ramp_shift;
    ps.a.ramp_zero = pl->d_ramp_zero;
    ps.a.chan_freq = pl->d_chanfreq;
    ps.a.chan_const = pl->d_chanconst;
    ps.a.bd = std::isinf(d->ref_freq_hz) ? 0.0
                                         : (d->sample_rate_hz / (double)N) / d->ref_freq_hz;
  }
  // Out-of-place intermediate passes: a pass that reads and writes the same scratch array is
  // 2-3 % slower than one that writes another array (cfg2: 1.505 -> 1.463 ms and 1.476 -> 1.426 ms,
  // profiles/r01_pingpong_scratch.log), so when the scratch is small against the device memory
  // (<= 1/5 of it, and 3x its size still free: a 34 GB cfg5 shard qualifies on a 180 GB part) a
  // second one is allocated and pass i reads
  // buffer (i-1)&1 and writes buffer i&1.  PBK_NO_PINGPONG=1 keeps the passes in place.
  if (pl->scratch && !getenv("PBK_NO_PINGPONG")) {
    bool any = false;
    for (const auto& ps : pl->passes)
      any = any || (ps.in_role == ROLE_SCRATCH && ps.out_role == ROLE_SCRATCH);
    size_t free_b = 0, total_b = 0;
    if (any && cudaMemGetInfo(&free_b, &total_b) == cudaSuccess &&
        pl->scratch_bytes <= total_b / 5 && free_b >= 3 * pl->scratch_bytes &&
        cudaMalloc(&pl->scratch2, pl->scratch_bytes) != cudaSuccess)
      pl->scratch2 = nullptr;
    cudaGetLastError();
  }
  if (tr.trials && pl->scratch && !pl->scratch2) {
    // the forward result must survive every trial: the per-trial passes work in the other array
    cudaError_t e = cudaMalloc(&pl->scratch2, pl->scratch_bytes);
    if (e != cudaSuccess) {
      pl->scratch2 = nullptr;
      return cleanup(fail(PBK_ERR_NOMEM, "second scratch (%zu bytes): %s", pl->scratch_bytes,
                          cudaGetErrorString(e)));
    }
  }
  setup_tma(pl);
  const int ds = (d->downsample > 1 && !pl->fused_tsum) ? 1 : 0;
  pl->launches = (int)pl->passes.size() + ds;
  pl->segments = pl->launches;
  if (tr.trials && (rc = set_trials(pl, tr)) != PBK_OK) return cleanup(rc);
  if (!tr.trials && !ramp) set_blocks_per_launch(pl);
  *out = pl;
  return PBK_OK;
}

extern "C" int pbk_dedisp_out_shape(const pbk_plan* pl, int64_t* rows, int64_t* row_elems,
                                    int64_t* elem_bytes) {
  if (!pl || pl->kind != PLAN_DEDISP) return fail(PBK_ERR_INVALID, "not a dedispersion plan");
  if (rows) *rows = pl->out_rows;
  if (row_elems) *row_elems = pl->row_elems;
  if (elem_bytes) *elem_bytes = pl->elem_bytes;
  return PBK_OK;
}

// the scratch arrays one pass reads (if its input is scratch) and writes (if its output is)
struct ScratchPair {
  void* in;
  void* out;
};

// Pass i of a schedule that works in the pair of arrays buf: with a second array the passes
// ping-pong, pass i reading buffer (i-1)&1 and writing buffer i&1; otherwise they work in place.
static ScratchPair pass_scratch(void* const buf[2], size_t i) {
  return {buf[1] ? buf[(i + 1) & 1] : buf[0], buf[1] ? buf[i & 1] : buf[0]};
}

static void* role_ptr(const pbk_plan* pl, int role, const void* uin, void* uout, void* scr) {
  switch (role) {
    case ROLE_USER_IN: return const_cast<void*>(uin);
    case ROLE_SCRATCH: return scr;
    case ROLE_USER_OUT: return uout;
    default: return pl->d_tmpf;
  }
}

static bool misaligned16(const void* p) { return ((uintptr_t)p & 15) != 0; }

// Epilogues that only the compile-time-shaped (fast / TMA) kernels implement: the time sum (and the
// fold behind it), the detection with its frequency sum (and fold), and the even / odd
// recombination.  The generic pass_kernel would silently skip them and write a differently shaped
// result, so such a pass never takes it.
static bool needs_fast_kernel(const Pass& ps) {
  return ps.a.tsum_log2 > 0 || ps.a.fsum_log2 > 0 || ps.a.fsum_split || ps.a.split;
}

// The fast kernels move 16-byte vectors, while the C ABI only promises element alignment.  When the
// last pass needs them and the caller's output is not 16-byte aligned, it writes this plan-owned
// buffer and the execution copies it out (device to device), as split_ragged does with d_tmpf.
static bool last_pass_needs_fast(const pbk_plan* pl) {
  return !pl->passes.empty() && pl->passes.back().out_role == ROLE_USER_OUT &&
         needs_fast_kernel(pl->passes.back());
}

static int stage_ensure(pbk_plan* pl, size_t bytes) {
  if (pl->stage_bytes >= bytes) return PBK_OK;
  cudaFree(pl->d_stage);   // waits for the work queued on the old buffer
  pl->d_stage = nullptr;
  pl->stage_bytes = 0;
  CUDA_TRY(cudaMalloc(&pl->d_stage, bytes));
  pl->stage_bytes = bytes;
  return PBK_OK;
}

static int launch_one(pbk_plan* pl, const Pass& ps, const void* d_in, void* d_out,
                      const void* d_chirp, ScratchPair scr, cudaStream_t st) {
  Pass p = ps;
  p.a.in = role_ptr(pl, ps.in_role, d_in, d_out, scr.in);
  p.a.out = role_ptr(pl, ps.out_role, d_in, d_out, scr.out);
  p.a.chirp_arr = reinterpret_cast<const float2*>(d_chirp);
  if (p.a.fsum_log2 > 0) p.a.fsum_bins = pl->exec_segbins;
  if (p.a.tsum_log2 > 0) p.a.tsum_bins = pl->exec_segbins;
  const bool aligned = (((uintptr_t)p.a.in | (uintptr_t)p.a.out) & 15) == 0;
  if (needs_fast_kernel(ps) && !(ps.family >= 0 && aligned))
    return fail(PBK_ERR_UNSUPPORTED, "%s pass with a fused %s epilogue needs the "
                "compile-time-shaped kernels and 16-byte aligned arrays (in %p, out %p)",
                ps.mode == MODE_FWD ? "FWD" : ps.mode == MODE_MID ? "MID" : "INV",
                ps.a.tsum_log2 > 0 ? "time-sum" : ps.a.fsum_log2 > 0 ? "detection" : "even/odd",
                p.a.in, p.a.out);
  if (p.a.trials > 1 && (ps.tma || ps.family < 0 || !aligned))
    return fail(PBK_ERR_UNSUPPORTED, "a batch of %d trials needs the LDG fast kernels and 16-byte "
                "aligned arrays", p.a.trials);
  cudaError_t e;
  CUtensorMap tm;
  if (ps.tma && aligned && tma_encode(ps, p.a.in, &tm)) {
    e = tma_launch(ps.a.log2L, ps.mode, p.a, tm, pl->d_ftab + ps.ftab_off, ps.ntiles, pl->num_sms,
                   st);
  } else if (ps.family >= 0 && aligned) {
    if (ps.fast_load_transposed)
      p.a.load_kind = ps.a.load_kind == LOAD_PLANAR ? LOAD_TRANSP_PLANAR : LOAD_TRANSP;
    e = fast_launch(ps.family, ps.a.log2L, ps.mode, p.a, pl->d_ftab + ps.ftab_off, ps.ntiles,
                    pl->num_sms, st);
  }
  else
    e = launch_pass(p, ps.fast && aligned, st);
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "kernel launch: %s", cudaGetErrorString(e));
  return PBK_OK;
}

// Passes [0, end) of the plan (every pass when end < 0), one launch each, ping-ponging between
// the plan's scratch arrays; timed segment i is pass i.  A whole execution also records the closing
// mark.  A trial plan runs its shared passes here (end = nshared), and the first batch of trials
// records that mark as its own first one (run_trial_passes).
static int run_passes(pbk_plan* pl, const void* d_in, void* d_out, const void* d_chirp,
                      cudaStream_t st, int end = -1) {
  const int np = (int)pl->passes.size();
  if (end < 0) end = np;
  prof_begin(pl);
  void* const buf[2] = {pl->scratch, pl->scratch2};
  for (int i = 0; i < end; ++i) {
    prof_mark(pl, i, st);
    const int rc = launch_one(pl, pl->passes[i], d_in, d_out, d_chirp, pass_scratch(buf, i), st);
    if (rc != PBK_OK) return rc;
  }
  if (end == np) prof_mark(pl, np, st);
  return PBK_OK;
}

// Trial schedule.  The shared forward passes run once (run_passes up to nshared); their result
// stays where the last of them wrote it.  Each batch of up to T trials then runs MID from that
// result into the other array (slab y of T for trial k0 + y), the inverse passes in place there,
// and the last pass into its output slabs.  One-level plans share nothing: every trial reads the
// caller's input.
static int run_trial_passes(pbk_plan* pl, const void* d_in, void* d_out, cudaStream_t st, int k,
                            int t, int seg) {
  const int ns = pl->nshared;
  void* buf[2] = {pl->scratch, pl->scratch2};
  void* shared = ns > 0 ? buf[(ns - 1) & 1] : nullptr;
  void* work = ns > 0 ? buf[ns & 1] : nullptr;
  for (size_t i = ns; i < pl->passes.size(); ++i) {
    Pass q = pl->passes[i];
    q.a.D = pl->trial_D[k];
    q.a.chan_const = pl->d_chanconst + (size_t)k * pl->chanconst_stride;
    if (t > 1) {   // trials k .. k + t - 1 along gridDim.y (choose_trials_per_launch)
      q.a.trials = t;
      q.a.trial_cc = pl->chanconst_stride;
      q.a.trial_in_bytes = (int)i == ns ? 0 : (long long)pl->scratch_bytes;
      q.a.trial_out_bytes = q.out_role == ROLE_USER_OUT ? (long long)pl->out_bytes
                                                        : (long long)pl->scratch_bytes;
    }
    prof_mark(pl, seg++, st);
    const int rc =
        launch_one(pl, q, d_in, d_out, nullptr, {(int)i == ns ? shared : work, work}, st);
    if (rc != PBK_OK) return rc;
  }
  prof_mark(pl, seg, st);
  return PBK_OK;
}

static int exec_dedisp(pbk_plan* pl, const void* d_in, void* d_out, const void* d_chirp,
                       cudaStream_t st, int batch, bool stage_any = false);

extern "C" int pbk_dedisp_exec_device(pbk_plan* pl, const void* d_in, void* d_out,
                                      const void* d_chirp, void* stream) {
  if (!pl || pl->kind != PLAN_DEDISP) return fail(PBK_ERR_INVALID, "not a dedispersion plan");
  if (!d_in) return fail(PBK_ERR_INVALID, "input pointer is NULL");
  if (pl->desc.explicit_chirp && !d_chirp) return fail(PBK_ERR_INVALID, "plan expects a chirp");
  if (pl->out_rows == 0) return PBK_OK;  // empty crop (dedispersion.py:130-133 returns no rows)
  if (!d_out) return fail(PBK_ERR_INVALID, "output pointer is NULL");
  CUDA_TRY(cudaSetDevice(pl->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (!pl->trials) {
    if (pl->blue) return blue_exec(pl, d_in, d_out, d_chirp, st);
    return exec_dedisp(pl, d_in, d_out, d_chirp, st, -1);
  }
  // trial k writes the slab out + k * out_bytes
  char* out = static_cast<char*>(d_out);
  int rc;
  if (pl->blue) {
    for (int k = 0; k < pl->ndm; ++k)
      if ((rc = blue_exec(pl, d_in, out + (size_t)k * pl->out_bytes, nullptr, st, k)) != PBK_OK)
        return rc;
    return PBK_OK;
  }
  if ((rc = run_passes(pl, d_in, nullptr, nullptr, st, pl->nshared)) != PBK_OK) return rc;
  const int T = pl->trials_per_launch;
  for (int b = 0; b * T < pl->ndm; ++b)
    if ((rc = exec_dedisp(pl, d_in, out + (size_t)b * T * pl->out_bytes, nullptr, st, b)) != PBK_OK)
      return rc;
  return PBK_OK;
}

// One execution of a plan (batch < 0), or batch `batch` of a trial plan whose shared passes have
// run (trials batch * T .. on), into d_out.  stage_any: stage an output that is not 16-byte aligned
// whenever the last pass writes it, as batches of trials always do (see below).
static int exec_dedisp(pbk_plan* pl, const void* d_in, void* d_out, const void* d_chirp,
                       cudaStream_t st, int batch, bool stage_any) {
  const int trial = batch < 0 ? -1 : batch * pl->trials_per_launch;
  const int ntr = batch < 0 ? 1 : std::min(pl->trials_per_launch, pl->ndm - trial);
  const size_t out_bytes = (size_t)ntr * pl->out_bytes;
  void* dst = pl->split_ragged ? pl->d_tmpf : d_out;
  // A trial slab is only element-aligned when the slab size is not a multiple of 16 bytes; it is
  // staged whenever the caller's output would be, so that every trial runs on the kernels an
  // aligned single-DM execution takes and gives the same bits.
  const bool stage = misaligned16(dst) &&
                     (trial < 0 && !stage_any ? last_pass_needs_fast(pl)
                                              : pl->passes.back().out_role == ROLE_USER_OUT);
  int rc;
  if (stage) {
    if ((rc = stage_ensure(pl, out_bytes)) != PBK_OK) return rc;
    dst = pl->d_stage;
  }
  if (pl->fused_tsum)   // the last pass adds its group sums to the output
    CUDA_TRY(cudaMemsetAsync(dst, 0, out_bytes, st));
  // timed segments of this execution (or batch): [seg0, seg0 + per)
  const int batches = (pl->ndm + pl->trials_per_launch - 1) / pl->trials_per_launch;
  const int per = trial < 0 ? pl->segments : (pl->segments - pl->nshared) / batches;
  const int seg0 = trial < 0 ? 0 : pl->nshared + batch * per;
  rc = trial < 0 ? run_passes(pl, d_in, dst, d_chirp, st)
                 : run_trial_passes(pl, d_in, dst, st, trial, ntr, seg0);
  if (rc != PBK_OK) return rc;
  if (stage)
    CUDA_TRY(cudaMemcpyAsync(d_out, pl->d_stage, out_bytes, cudaMemcpyDeviceToDevice, st));
  if (pl->split_ragged)
    CUDA_TRY(cudaMemcpyAsync(d_out, static_cast<const char*>(pl->d_tmpf) + pl->split_skip,
                             pl->out_bytes, cudaMemcpyDeviceToDevice, st));
  if (pl->desc.downsample > 1 && !pl->fused_tsum) {
    cudaError_t e = launch_downsample(reinterpret_cast<const float*>(pl->d_tmpf),
                                      reinterpret_cast<float*>(d_out), pl->out_rows,
                                      pl->row_elems, pl->desc.downsample, st);
    if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "downsample launch: %s", cudaGetErrorString(e));
    prof_mark(pl, seg0 + per, st);
  }
  return PBK_OK;
}

// Overlap-save blocks b0 .. b0 + t - 1 of a stream as one launch per pass (gridDim.y = t): block
// b0 + y reads the stream at in + y * stride, works in slab y of the block scratch arrays
// (ping-ponging between them as run_passes does between the plan's own) and writes out + y * slab.
static int run_block_batch(pbk_plan* pl, const char* in, char* out, int t, size_t stride,
                           cudaStream_t st) {
  if (pl->fused_tsum)   // the last pass adds its group sums to the output
    CUDA_TRY(cudaMemsetAsync(out, 0, (size_t)t * pl->out_bytes, st));
  for (size_t i = 0; i < pl->passes.size(); ++i) {
    Pass q = pl->passes[i];
    q.a.trials = t;
    q.a.trial_in_bytes = q.in_role == ROLE_USER_IN ? (long long)stride
                                                   : (long long)pl->scratch_bytes;
    q.a.trial_out_bytes = q.out_role == ROLE_USER_OUT ? (long long)pl->out_bytes
                                                      : (long long)pl->scratch_bytes;
    const int rc = launch_one(pl, q, in, out, nullptr, pass_scratch(pl->blk_scratch, i), st);
    if (rc != PBK_OK) return rc;
  }
  return PBK_OK;
}

// T slabs in each scratch array the plan uses, for batched block executions
static int blocks_scratch_ensure(pbk_plan* pl) {
  if (pl->blk_scratch[0]) return PBK_OK;
  const size_t bytes = (size_t)pl->blocks_per_launch * pl->scratch_bytes;
  void* b[2] = {nullptr, nullptr};
  for (int j = 0; j < (pl->scratch2 ? 2 : 1); ++j) {
    const cudaError_t e = cudaMalloc(&b[j], bytes);
    if (e != cudaSuccess) {
      cudaFree(b[0]);
      return fail(PBK_ERR_NOMEM, "block scratch (%zu bytes): %s", bytes, cudaGetErrorString(e));
    }
  }
  pl->blk_scratch[0] = b[0];
  pl->blk_scratch[1] = b[1];
  pl->blk_bytes = bytes;
  return PBK_OK;
}

extern "C" int pbk_dedisp_exec_blocks_device(pbk_plan* pl, const void* d_in, int64_t nblocks,
                                             void* d_out, void* stream) {
  if (!pl || pl->kind != PLAN_DEDISP) return fail(PBK_ERR_INVALID, "not a dedispersion plan");
  if (!d_in) return fail(PBK_ERR_INVALID, "input pointer is NULL");
  if (nblocks < 0)
    return fail(PBK_ERR_INVALID, "nblocks must be >= 0, got %lld", (long long)nblocks);
  if (pl->trials)
    return fail(PBK_ERR_UNSUPPORTED, "block execution of a trial plan is not supported");
  if (pl->desc.explicit_chirp)
    return fail(PBK_ERR_UNSUPPORTED, "block execution of an explicit-chirp plan is not supported");
  if (nblocks == 0 || pl->out_rows == 0) return PBK_OK;
  if (!d_out) return fail(PBK_ERR_INVALID, "output pointer is NULL");
  CUDA_TRY(cudaSetDevice(pl->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const pbk_dedisp_desc& d = pl->desc;
  const size_t in_row = ((size_t)d.nchan * d.npol * load_bits(load_kind_of(d.in_dtype))) >> 3;
  const size_t stride = (size_t)(d.crop_stop - d.crop_start) * in_row;
  const char* in = static_cast<const char*>(d_in);
  char* out = static_cast<char*>(d_out);
  const int T = (misaligned16(in) || misaligned16(out) || stride % 16) ? 1 : pl->blocks_per_launch;
  struct ProfOff {   // pbk_plan_profile times single executions only
    pbk_plan* pl;
    explicit ProfOff(pbk_plan* p) : pl(p) { pl->prof_off = true; }
    ~ProfOff() { pl->prof_off = false; }
  } prof_off(pl);
  int rc;
  if (T == 1) {
    // the single execution at each block's pointers; an output slab that is not 16-byte aligned
    // is staged so that every block runs on the kernels of an aligned execution
    for (int64_t b = 0; b < nblocks; ++b) {
      const char* bi = in + (size_t)b * stride;
      char* bo = out + (size_t)b * pl->out_bytes;
      rc = pl->blue ? blue_exec(pl, bi, bo, nullptr, st)
                    : exec_dedisp(pl, bi, bo, nullptr, st, -1, true);
      if (rc != PBK_OK) return rc;
    }
    return PBK_OK;
  }
  if ((rc = blocks_scratch_ensure(pl)) != PBK_OK) return rc;
  for (int64_t b0 = 0; b0 < nblocks; b0 += T) {
    const int t = (int)std::min<int64_t>(T, nblocks - b0);
    rc = run_block_batch(pl, in + (size_t)b0 * stride, out + (size_t)b0 * pl->out_bytes, t, stride,
                         st);
    if (rc != PBK_OK) return rc;
  }
  return PBK_OK;
}

extern "C" int pbk_plan_blocks_per_launch(const pbk_plan* pl, int32_t* T) {
  if (!pl || !T) return fail(PBK_ERR_INVALID, "NULL argument");
  *T = pl->blocks_per_launch;
  return PBK_OK;
}

static int ensure_buf(void** p, size_t bytes) {
  if (*p || bytes == 0) return PBK_OK;
  CUDA_TRY(cudaMalloc(p, bytes));
  return PBK_OK;
}

// Coherent dedispersion -> detection -> time sum -> fold.  Fused route (the time sum runs in the
// epilogue of the last inverse pass, large intermediate, few rows per bin): the phase bin of every
// output row is computed first, and the last pass adds its group sums to profile[bin] instead of
// out[row], so the intensity never reaches HBM.  Otherwise the plan's normal execution writes a
// plan-owned buffer and pbk_fold's kernel folds it.
extern "C" int pbk_dedisp_fold_exec_device(pbk_plan* pl, const void* d_in, void* d_profile,
                                           void* d_counts, const double* coeffs, int32_t ncoef,
                                           double sample_rate_hz, int64_t n0, int32_t nbin,
                                           void* stream) {
  if (!pl || pl->kind != PLAN_DEDISP) return fail(PBK_ERR_INVALID, "not a dedispersion plan");
  if (pl->trials) return fail(PBK_ERR_UNSUPPORTED, "folding a trial plan is not supported");
  if (pl->desc.out_kind != PBK_OUT_INTENSITY && pl->desc.out_kind != PBK_OUT_STOKES_I)
    return fail(PBK_ERR_INVALID, "folding needs a plan with out_kind INTENSITY or STOKES_I");
  if (pl->desc.explicit_chirp) return fail(PBK_ERR_INVALID, "folding takes no explicit chirp");
  if (!d_in || !d_profile || !d_counts || !coeffs) return fail(PBK_ERR_INVALID, "NULL pointer");
  if (nbin <= 0) return fail(PBK_ERR_INVALID, "nbin must be positive");
  if (ncoef < 1 || ncoef > kFoldMaxCoef)
    return fail(PBK_ERR_INVALID, "ncoef must be in [1, %d]", kFoldMaxCoef);
  if (!(sample_rate_hz > 0) || !std::isfinite(sample_rate_hz))
    return fail(PBK_ERR_INVALID, "sample_rate_hz must be finite and > 0");
  for (int i = 0; i < ncoef; ++i)
    if (!std::isfinite(coeffs[i]))
      return fail(PBK_ERR_INVALID, "phase coefficient %d is not finite", i);
  if (pl->out_rows == 0) return PBK_OK;   // empty crop: nothing to fold
  CUDA_TRY(cudaSetDevice(pl->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  FoldArgs fa;
  memset(&fa, 0, sizeof(fa));
  for (int i = 0; i < ncoef; ++i) fa.coef[i] = coeffs[i];
  fa.ncoef = ncoef;
  fa.sample_rate = sample_rate_hz;
  fa.n0 = n0;
  fa.nbin = nbin;
  fa.nsamp = pl->out_rows;
  fa.row_elems = pl->row_elems;
  fold_args_finish(fa);
  fa.counts = reinterpret_cast<unsigned long long*>(d_counts);
  // The fused route saves the intermediate's round trip, which only costs HBM traffic once it is
  // well beyond the 126 MB L2, but it sends every group sum of a profile cell to the same address.
  // MEASURED (B200 1000 W, cfg2 geometry, scripts/dedisp_fold_bw.py, profiles/r03_dedisp_fold.log):
  // per-pol x8 / 1024 bins (256 MiB, 512 rows per bin) 0.987x the two steps, x4 (1024 rows per
  // bin) 0.96x; Stokes I x4 (256 MiB, 1024 rows per bin) 1.017x, x64 (16 MiB) 1.005x, 16 bins up
  // to 1.23x.  So: fused only for an intermediate of >= 256 MiB with <= 512 rows per bin.
  // The fused pass runs on the fast kernels only, which need 16-byte aligned arrays: a profile
  // aligned only to its float32 elements takes the unfused route.
  const bool fuse = pl->fused_tsum &&
                    (size_t)pl->out_rows * pl->row_elems * 4 >= ((size_t)256 << 20) &&
                    pl->out_rows <= 512ll * nbin && !misaligned16(d_profile);
  if (fuse) {
    if (!pl->d_segbins) {
      const size_t b = (size_t)pl->out_rows * sizeof(int);
      CUDA_TRY(cudaMalloc(&pl->d_segbins, b));
      pl->fold_bytes += b;
    }
    const unsigned blocks = (unsigned)std::min<long long>((pl->out_rows + 255) / 256, 148 * 4);
    fold_bins_kernel<<<blocks, 256, 0, st>>>(fa, pl->d_segbins);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "fold bins launch: %s", cudaGetErrorString(e));
    pl->exec_segbins = pl->d_segbins;
    const int rc = run_passes(pl, d_in, d_profile, nullptr, st);   // no memset: it accumulates
    pl->exec_segbins = nullptr;
    return rc;
  }
  if (!pl->d_foldbuf) {
    CUDA_TRY(cudaMalloc(&pl->d_foldbuf, pl->out_bytes));
    pl->fold_bytes += pl->out_bytes;
  }
  const int rc = pbk_dedisp_exec_device(pl, d_in, pl->d_foldbuf, nullptr, stream);
  if (rc != PBK_OK) return rc;
  fa.in = reinterpret_cast<const float*>(pl->d_foldbuf);
  fa.profile = reinterpret_cast<float*>(d_profile);
  cudaError_t e = launch_fold(fa, st);
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "fold launch: %s", cudaGetErrorString(e));
  return PBK_OK;
}

extern "C" int pbk_dedisp_exec_host(pbk_plan* pl, const void* in, void* out, const void* chirp) {
  if (!pl || pl->kind != PLAN_DEDISP) return fail(PBK_ERR_INVALID, "not a dedispersion plan");
  if (!in) return fail(PBK_ERR_INVALID, "input pointer is NULL");
  if (pl->desc.explicit_chirp && !chirp) return fail(PBK_ERR_INVALID, "plan expects a chirp");
  if (pl->out_rows == 0) return PBK_OK;
  if (!out) return fail(PBK_ERR_INVALID, "output pointer is NULL");
  std::lock_guard<std::mutex> lock(pl->mu);
  CUDA_TRY(cudaSetDevice(pl->device));
  int rc;
  const size_t out_bytes = pl->out_bytes * pl->ndm;   // a trial plan writes ndm slabs
  if ((rc = ensure_buf(&pl->h_din, pl->in_bytes)) != PBK_OK) return rc;
  if ((rc = ensure_buf(&pl->h_dout, out_bytes)) != PBK_OK) return rc;
  if ((rc = ensure_buf(&pl->h_dchirp, pl->chirp_bytes)) != PBK_OK) return rc;
  cudaStream_t st = cudaStreamPerThread;
  // pageable blocks go through the multi-threaded bounce pipeline (pbk_hostcopy.h)
  CUDA_TRY(host_to_device(pl->h_din, in, pl->in_bytes, st));
  if (pl->chirp_bytes) CUDA_TRY(host_to_device(pl->h_dchirp, chirp, pl->chirp_bytes, st));
  rc = pbk_dedisp_exec_device(pl, pl->h_din, pl->h_dout, pl->h_dchirp, st);
  if (rc != PBK_OK) return rc;
  CUDA_TRY(device_to_host(out, pl->h_dout, out_bytes, st));
  return PBK_OK;
}

// ------------------------------------------------------------------------------------------
// FFT / STFT plans (forward-structured passes only)
// ------------------------------------------------------------------------------------------
struct ExtMap {  // external array addressing: o*eo + idx*ei + c*ec + p*ep
  long long eo, ei, ec, ep;
};
static int blue_fft_plan_create(long long O, long long n, long long C, long long P, bool inverse,
                                ExtMap in, ExtMap outm, float scale, bool shift_out, bool shift_in,
                                int device, pbk_plan** out, int in_kind);

// in_kind: load kind of the user's input (LOAD_C64, or raw baseband decoded in the first pass)
// detected channelizer output (pbk_stft_detect_plan_create): |z|^2 summed over `fsum` adjacent
// fine channels in the epilogue of the last pass
struct DetectSpec {
  int pq = 0;          // floats per output cell: 0 = no detection, 1 = summed over the pair, 2 = per pol
  long long fsum = 1;
  bool split = false;  // the pair is the even / odd samples of one single-pol column (n is HALF)
  bool volt = false;   // split with complex64 VOLTAGES out (plain stft of one single-pol channel)
};

static int build_fft_plan(long long O, long long n, long long C, long long P, bool inverse,
                          ExtMap in, ExtMap outm, float scale, bool shift_out, bool shift_in,
                          int device, pbk_plan** out, int in_kind = LOAD_C64,
                          const DetectSpec* det = nullptr) {
  *out = nullptr;
  const int ln = ilog2_exact(n);
  if (ln < 1) {
    if (n < 2) return fail(PBK_ERR_UNSUPPORTED, "transform length %lld is too short", (long long)n);
    // the even / odd recombination and the detecting epilogue live in the last tile pass: the
    // Bluestein plan has neither, so the caller takes its plain path
    if (det)
      return fail(PBK_ERR_UNSUPPORTED, "length %lld is not a power of two: no even / odd or "
                  "detecting last pass", (long long)n);
    // not a power of two: Bluestein on top of the power-of-two passes (pbk_blue.cuh)
    return blue_fft_plan_create(O, n, C, P, inverse, in, outm, scale, shift_out, shift_in, device,
                                out, in_kind);
  }
  int l[3] = {0, 0, 0};
  const int m = choose_levels(ln, C * P, l, false);
  if (m == 0) return fail(PBK_ERR_UNSUPPORTED, "transform length 2^%d is too long", ln);
  const long long I = C * P;
  if (I > INT_MAX / 2 || O <= 0 || I <= 0) return fail(PBK_ERR_INVALID, "bad batch shape");
  int ndev = 0;
  CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev)
    return fail(PBK_ERR_CUDA, "device %d not available (%d CUDA devices)", device, ndev);
  CUDA_TRY(cudaSetDevice(device));

  pbk_plan* pl = new pbk_plan();
  pl->kind = PLAN_FFT;
  pl->device = device;
  pl->nlevels = m;
  for (int i = 0; i < m; ++i) pl->level_log2[i] = l[i];
  pl->in_bytes = ((size_t)O * n * I * load_bits(in_kind)) >> 3;
  pl->out_bytes = (size_t)O * n * I * 8;
  TableSet ts;
  long long Kprev[3], R[3];
  {
    long long k = 1;
    for (int i = 0; i < m; ++i) { Kprev[i] = k; k <<= l[i]; }
    long long r = 1;
    for (int i = m - 1; i >= 0; --i) { R[i] = r; r <<= l[i]; }
  }
  auto log2ll = [](long long v) { int s = 0; while ((1ll << s) < v) ++s; return s; };
  for (int i = 0; i < m; ++i) {
    Pass ps;
    defaults(ps.a);
    ps.mode = MODE_FWD;
    ps.signinv = inverse;
    ps.a.sign = inverse ? +1 : -1;
    set_geometry(ps, l[i], O * Kprev[i] * R[i] * I, R[i] * I, (int)I, (int)P, log2ll(Kprev[i]));
    AddrMap pm = plain_map(1ll << l[i], R[i], I, P);
    pm.a_o = n * I;
    ps.a.min = pm;
    ps.a.mout = pm;
    if (i == 0) {
      AddrMap& a = ps.a.min;
      a.a_o = in.eo; a.a_kp = 0; a.a_kl = 0; a.a_n = in.ei; a.a_c = in.ec; a.a_p = in.ep;
      a.a_row = R[0] * in.ei;
      ps.a.load_kind = in_kind;
      if (shift_in) ps.a.fxor = 1 << (l[0] - 1);
    }
    if (i == m - 1) {
      AddrMap& a = ps.a.mout;
      a.a_o = outm.eo; a.a_kp = 0; a.a_kl = outm.ei; a.a_n = 0; a.a_c = outm.ec; a.a_p = outm.ep;
      a.a_row = Kprev[i] * outm.ei;
      ps.a.scale = scale;
      if (shift_out) ps.a.kxor = 1 << (l[i] - 1);
    }
    ps.a.log2M = i == m - 1 ? 0 : l[i] + log2ll(R[i]);
    set_klow(ps.a, i + 1, l);
    ps.in_role = i == 0 ? ROLE_USER_IN : ROLE_SCRATCH;
    ps.out_role = i == m - 1 ? ROLE_USER_OUT : ROLE_SCRATCH;
    ps.fast = (I % 2 == 0) && map_even(ps.a.min, P) && map_even(ps.a.mout, P) &&
              ((O * Kprev[i] * R[i] * I) % 2 == 0);
    ps.pair_ok = ps.fast;
    ts.ensure(l[i]);
    pl->passes.push_back(ps);
  }
  mark_scratch_layout(pl, I);
  int rc = upload_tables(pl, ts);
  if (rc == PBK_OK) rc = setup_fast(pl);
  if (rc != PBK_OK) { pbk_plan_destroy(pl); return rc; }
  if (det && det->volt) {
    // plain channelizer of ONE single-pol column on the compile-time-shaped kernels: this plan
    // transforms the (n, 2) even / odd view at half length and the last pass recombines
    // X[k] = E + wO, X[k + n] = E - wO in registers and stores both halves of the fftshift-ed
    // segment (pbk_fast.cuh, FWDLAST).  Needs the two-level plan with the narrow fast last pass.
    Pass& last = pl->passes.back();
    const bool ok = m == 2 && I == 2 && !inverse && last.family >= 0 && last.a.final_epi &&
                    !last.a.out_transpose && last.a.load_kind == LOAD_PLANAR;
    if (!ok) {
      pbk_plan_destroy(pl);
      return fail(PBK_ERR_UNSUPPORTED, "even/odd channelizer needs a two-level segment length");
    }
    PassArgs& a = last.a;
    a.fsum_split = 1;
    a.fsum_log2n = ln + 1;
    a.log2Kmul = l[0];
    a.mout = AddrMap{2 * n, 0, 0, 0, 0, 0, 0};      // complex64 elements per (full-length) segment
  }
  if (det && det->pq) {
    // The epilogue sums the 2^k first-level bins that share an output cell: it needs the two-level
    // plan of a long segment (fine channel = kprev + Kprev * row), one channel (I == 2: a lane
    // pair per bin) on the compile-time-shaped narrow kernel, and F a multiple of the bins a tile
    // holds that divides Kprev.  Anything else: PBK_ERR_UNSUPPORTED (callers then detect the
    // channelized voltages with pbk_detect_scrunch).
    Pass& last = pl->passes.back();
    const long long Kp = 1ll << l[0];
    const long long rows_per_tile = last.family >= 0 ? (2ll << last.finfo.log2pw) / I : 0;
    const int lf = ilog2_exact(det->fsum);
    const bool ok = m == 2 && I == 2 && !inverse && last.family >= 0 && last.a.final_epi &&
                    !last.a.out_transpose && last.a.load_kind == LOAD_PLANAR && lf > 0 &&
                    rows_per_tile > 0 && det->fsum % rows_per_tile == 0 && Kp % det->fsum == 0 &&
                    last.ntiles % (det->fsum / rows_per_tile) == 0;
    if (!ok) {
      pbk_plan_destroy(pl);
      return fail(PBK_ERR_UNSUPPORTED, "fused detection needs one channel, a two-level segment "
                  "length and a frequency sum that divides its first level (got n = %lld, "
                  "nchan*npol = %lld, freq_sum = %lld)", (long long)n, (long long)I,
                  (long long)det->fsum);
    }
    PassArgs& a = last.a;
    long long rpt = rows_per_tile;
    {
      // half-width tiles (four 128-thread CTAs per SM instead of two of 256) when the shape allows:
      // same stage tables, so the slot staged by setup_fast is reused.  $PBK_NO_NARROW_FSUM=1 keeps
      // the full-width tiles.
      FastInfo fn;
      if (!getenv("PBK_NO_NARROW_FSUM") && fast_info(FAMILY_R16N, a.log2L, &fn) &&
          fn.tw_count == last.finfo.tw_count) {
        const long long Wn = 2ll << fn.log2pw, rn = Wn / I;
        if (rn > 0 && det->fsum % rn == 0 && Kp % rn == 0 && a.Q % Wn == 0 &&
            (a.Q / Wn) % (det->fsum / rn) == 0) {
          last.family = FAMILY_R16N;
          last.finfo = fn;
          last.ntiles = a.Q / Wn;
          rpt = rn;
        }
      }
    }
    a.fsum_log2 = lf;
    a.fsum_g_log2 = ilog2_exact(det->fsum / rpt);
    a.fsum_row_shift = l[0] - lf;
    a.fsum_pq = det->pq;
    a.fsum_split = det->split ? 1 : 0;
    a.fsum_log2n = ln + 1;                      // split: the full segment is twice this plan's n
    a.log2Kmul = l[0];
    a.epi_kind = EPI_INTENSITY;
    const long long cells = (det->split ? 2 * n : n) / det->fsum;     // output cells per segment
    a.mout = AddrMap{cells * det->pq, 0, 0, 0, 0, 0, 0};
    a.fsum_cells = cells;
    // I == 2: a lane row of the tile is a contiguous run of L rows of the scratch array (16 B per
    // row), so the tile is read coalesced and transposed through shared memory
    if (!getenv("PBK_NO_TRANSP_DETECT")) last.fast_load_transposed = true;
    pl->out_bytes = (size_t)O * cells * det->pq * 4;
    pl->det_nseg = O;
    pl->det_cells = cells;
    pl->det_pq = det->pq;
  }
  if (m > 1) {
    pl->scratch_bytes = (size_t)O * n * I * 8;
    cudaError_t e = cudaMalloc(&pl->scratch, pl->scratch_bytes);
    if (e != cudaSuccess) {
      pbk_plan_destroy(pl);
      return fail(PBK_ERR_NOMEM, "scratch (%zu bytes): %s", (size_t)O * n * I * 8,
                  cudaGetErrorString(e));
    }
  }
  setup_tma(pl);
  pl->launches = (int)pl->passes.size();
  pl->segments = pl->launches;
  *out = pl;
  return PBK_OK;
}


// ------------------------------------------------------------------------------------------
// arbitrary transform lengths (Bluestein, kernels in pbk_blue.cuh)
// ------------------------------------------------------------------------------------------
struct BlueState {
  long long O = 1, n = 0, M = 0, I = 1;
  int P = 1;
  pbk_plan* fwdM = nullptr;   // (O, M, I) forward FFT, out of place
  pbk_plan* invM = nullptr;   // (O, M, I) inverse FFT with the 1/M scale
  float2 *w = nullptr, *bhat = nullptr, *A = nullptr, *B = nullptr, *T = nullptr;
  bool dedisp = false, inverse = false;
  BlueIO in{}, out{};
  PassArgs chirp{};           // dedispersion: chirp description for blue_midH_kernel
  int out_kind = PBK_OUT_C64;
  long long crop_rows = 0, downsample = 1;
};

static long long blue_pad_len(long long n) {
  long long M = 16;
  while (M < 2 * n - 1) M <<= 1;
  return M;
}

template <typename K, typename... A>
static cudaError_t launch_grid(K kern, long long total, cudaStream_t st, A... args) {
  if (total <= 0) return cudaSuccess;
  long long blocks = (total + 255) / 256;
  if (blocks > 148ll * 16) blocks = 148ll * 16;
  kern<<<(unsigned)blocks, 256, 0, st>>>(args...);
  return cudaGetLastError();
}

static void blue_free(BlueState* b) {
  if (!b) return;
  pbk_plan_destroy(b->fwdM);
  pbk_plan_destroy(b->invM);
  cudaFree(b->w);
  cudaFree(b->bhat);
  cudaFree(b->A);
  cudaFree(b->B);
  cudaFree(b->T);
  delete b;
}

// common part: chirp table, filter spectrum, the two M-point FFT plans and the work buffers
static int blue_setup(BlueState* b, int device) {
  b->M = blue_pad_len(b->n);
  if (b->M > (1ll << 30)) return fail(PBK_ERR_UNSUPPORTED, "transform length %lld is too long", b->n);
  const ExtMap em{b->M * b->I, b->I, 1, 0};
  int rc = build_fft_plan(b->O, b->M, b->I, 1, false, em, em, 1.0f, false, false, device, &b->fwdM);
  if (rc != PBK_OK) return rc;
  rc = build_fft_plan(b->O, b->M, b->I, 1, true, em, em, (float)(1.0 / (double)b->M), false, false,
                      device, &b->invM);
  if (rc != PBK_OK) return rc;
  const size_t work = (size_t)b->O * b->M * b->I * sizeof(float2);
  CUDA_TRY(cudaMalloc(&b->w, (size_t)b->n * sizeof(float2)));
  CUDA_TRY(cudaMalloc(&b->bhat, (size_t)b->M * sizeof(float2)));
  CUDA_TRY(cudaMalloc(&b->A, work));
  CUDA_TRY(cudaMalloc(&b->B, work));
  cudaError_t e = launch_grid(blue_chirp_kernel, b->n, 0, b->w, b->n);
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "chirp table: %s", cudaGetErrorString(e));
  // spectrum of the filter: one M-point column FFT at plan time
  float2* filt = nullptr;
  CUDA_TRY(cudaMalloc(&filt, (size_t)b->M * sizeof(float2)));
  e = launch_grid(blue_filter_kernel, b->M, 0, (const float2*)b->w, filt, b->n, b->M);
  pbk_plan* one = nullptr;
  const ExtMap e1{b->M, 1, 1, 0};
  rc = e == cudaSuccess ? build_fft_plan(1, b->M, 1, 1, false, e1, e1, 1.0f, false, false, device, &one)
                        : fail(PBK_ERR_CUDA, "filter: %s", cudaGetErrorString(e));
  if (rc == PBK_OK) rc = run_passes(one, filt, b->bhat, nullptr, 0);
  if (rc == PBK_OK && cudaDeviceSynchronize() != cudaSuccess)
    rc = fail(PBK_ERR_CUDA, "filter spectrum: %s", cudaGetErrorString(cudaGetLastError()));
  pbk_plan_destroy(one);
  cudaFree(filt);
  return rc;
}

// forward or inverse DFT of length n through two M-point FFTs: in -> A -> B -> A -> out
static int blue_convolve(BlueState* b, bool conj, cudaStream_t st) {
  int rc = run_passes(b->fwdM, b->A, b->B, nullptr, st);
  if (rc != PBK_OK) return rc;
  cudaError_t e = launch_grid(blue_mul_kernel, b->O * b->M * b->I, st, b->B, (const float2*)b->bhat,
                              b->O, b->M, b->I, conj ? 1 : 0);
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "bluestein multiply: %s", cudaGetErrorString(e));
  return run_passes(b->invM, b->B, b->A, nullptr, st);
}

// (trial >= 0: the chirp of that trial of a trial plan)
static int blue_exec(pbk_plan* pl, const void* d_in, void* d_out, const void* d_chirp,
                     cudaStream_t st, int trial) {
  BlueState* b = pl->blue;
  const long long total = b->O * b->M * b->I;
  cudaError_t e = launch_grid(blue_pre_kernel, total, st, d_in, b->A, (const float2*)b->w, b->in);
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "bluestein pre: %s", cudaGetErrorString(e));
  int rc = blue_convolve(b, b->in.conj_w != 0, st);
  if (rc != PBK_OK) return rc;
  if (b->dedisp) {
    PassArgs ch = b->chirp;
    ch.chirp_arr = reinterpret_cast<const float2*>(d_chirp);
    if (trial >= 0) ch.D = pl->trial_D[trial];
    e = launch_grid(blue_midH_kernel, b->M * b->I, st, b->A, b->n, b->M, b->I, b->P, ch);
    if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "bluestein chirp: %s", cudaGetErrorString(e));
    if ((rc = blue_convolve(b, true, st)) != PBK_OK) return rc;
  }
  float2* dst = reinterpret_cast<float2*>(b->out_kind == PBK_OUT_C64 ? d_out : (void*)b->T);
  const long long rows = b->out.hi - b->out.lo;
  e = launch_grid(blue_post_kernel, b->O * rows * b->I, st, (const float2*)b->A, dst,
                  (const float2*)b->w, b->out);
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "bluestein post: %s", cudaGetErrorString(e));
  if (b->out_kind != PBK_OUT_C64) {
    e = launch_detect(b->T, reinterpret_cast<float*>(d_out), pl->out_rows, b->I,
                      b->out_kind == PBK_OUT_STOKES_I, b->downsample, st);
    if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "detect launch: %s", cudaGetErrorString(e));
  }
  return PBK_OK;
}

// coherent dedispersion of a length that is not a power of two
static int blue_dedisp_plan_create(const pbk_dedisp_desc* d, const RampSpec* ramp,
                                   pbk_plan** out) {
  const long long N = d->nsamp, C = d->nchan, I = d->nchan * d->npol;
  int ndev = 0;
  CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (d->device < 0 || d->device >= ndev)
    return fail(PBK_ERR_CUDA, "device %d not available (%d CUDA devices)", d->device, ndev);
  CUDA_TRY(cudaSetDevice(d->device));
  pbk_plan* pl = new pbk_plan();
  BlueState* b = new BlueState();
  pl->blue = b;
  pl->kind = PLAN_DEDISP;
  pl->device = d->device;
  pl->desc = *d;
  pl->desc.chan_freq_hz = nullptr;
  b->O = 1; b->n = N; b->I = I; b->P = (int)d->npol;
  b->dedisp = true;
  b->out_kind = d->out_kind;
  b->downsample = d->downsample;
  const long long crop_rows = std::max<long long>(0, d->crop_stop - d->crop_start);
  b->crop_rows = crop_rows;
  pl->full_rows = crop_rows;
  pl->out_rows = d->downsample > 1 ? crop_rows / d->downsample : crop_rows;
  pl->row_elems = d->out_kind == PBK_OUT_STOKES_I ? C : I;
  pl->elem_bytes = d->out_kind == PBK_OUT_C64 ? 8 : 4;
  pl->in_bytes = ((size_t)N * I * load_bits(load_kind_of(d->in_dtype))) >> 3;
  pl->out_bytes = (size_t)pl->out_rows * pl->row_elems * pl->elem_bytes;
  pl->chirp_bytes = d->explicit_chirp ? (size_t)N * C * 8 : 0;
  auto cleanup = [&](int code) { pbk_plan_destroy(pl); return code; };
  int rc = blue_setup(b, d->device);
  if (rc != PBK_OK) return cleanup(rc);
  b->in = BlueIO{BlueMap{0, I, d->npol, 1}, 1, N, b->M, I, (int)d->npol,
                 load_kind_of(d->in_dtype),
                 0, 0, 1.0f, 0, N};
  b->out = BlueIO{BlueMap{0, I, d->npol, 1}, 1, N, b->M, I, (int)d->npol, EPI_C64, 1, 0,
                  (float)(1.0 / (double)N), d->crop_start, std::max(d->crop_start, d->crop_stop)};
  defaults(b->chirp);
  b->chirp.chirp_kind = ramp ? CHIRP_RAMP : d->explicit_chirp ? CHIRP_ARRAY : CHIRP_COMPUTED;
  b->chirp.N = N;
  if (ramp) {
    if ((rc = upload_ramp(pl, ramp, C, N)) != PBK_OK) return cleanup(rc);
    b->chirp.ramp_shift = pl->d_ramp_shift;
    b->chirp.ramp_zero = pl->d_ramp_zero;
    b->chirp.ramp_hilbert = (ramp->flags & PBK_RAMP_HILBERT) ? 1 : 0;
  }
  b->chirp.df = 1.0 / ((double)N * (1.0 / d->sample_rate_hz));
  if (std::isinf(d->ref_freq_hz)) { b->chirp.fr_sub = 0; b->chirp.inv_fr = 0; b->chirp.a0 = -1.0; }
  else { b->chirp.fr_sub = d->ref_freq_hz; b->chirp.inv_fr = 1.0 / d->ref_freq_hz; b->chirp.a0 = 0; }
  b->chirp.D = chirp_D(d->dm);
  b->chirp.scale = 1.0f;
  b->chirp.chirp_sk = C;
  b->chirp.chirp_sc = 1;
  {
    cudaError_t e = cudaMalloc(&pl->d_chanfreq, (size_t)C * sizeof(double));
    if (e == cudaSuccess)
      e = cudaMemcpy(pl->d_chanfreq, d->chan_freq_hz, (size_t)C * sizeof(double),
                     cudaMemcpyHostToDevice);
    if (e == cudaSuccess && d->out_kind != PBK_OUT_C64 && crop_rows > 0)
      e = cudaMalloc(&b->T, (size_t)crop_rows * I * sizeof(float2));
    if (e != cudaSuccess) return cleanup(fail(PBK_ERR_CUDA, "alloc: %s", cudaGetErrorString(e)));
  }
  b->chirp.chan_freq = pl->d_chanfreq;
  pl->launches = 5 + 2 * (b->fwdM->launches + b->invM->launches) +
                 (d->out_kind != PBK_OUT_C64 ? 1 : 0);
  pl->segments = 0;
  *out = pl;
  return PBK_OK;
}

// plain / STFT transform of a length that is not a power of two
static int blue_fft_plan_create(long long O, long long n, long long C, long long P, bool inverse,
                                ExtMap in, ExtMap outm, float scale, bool shift_out, bool shift_in,
                                int device, pbk_plan** out, int in_kind) {
  int ndev = 0;
  CUDA_TRY(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev)
    return fail(PBK_ERR_CUDA, "device %d not available (%d CUDA devices)", device, ndev);
  CUDA_TRY(cudaSetDevice(device));
  pbk_plan* pl = new pbk_plan();
  BlueState* b = new BlueState();
  pl->blue = b;
  pl->kind = PLAN_FFT;
  pl->device = device;
  b->O = O; b->n = n; b->I = C * P; b->P = (int)P;
  b->inverse = inverse;
  pl->in_bytes = ((size_t)O * n * C * P * load_bits(in_kind)) >> 3;
  pl->out_bytes = (size_t)O * n * C * P * 8;
  int rc = blue_setup(b, device);
  if (rc != PBK_OK) { pbk_plan_destroy(pl); return rc; }
  b->in = BlueIO{BlueMap{in.eo, in.ei, in.ec, in.ep}, O, n, b->M, C * P, (int)P, in_kind,
                 inverse ? 1 : 0, shift_in ? n / 2 : 0, 1.0f, 0, n};
  b->out = BlueIO{BlueMap{outm.eo, outm.ei, outm.ec, outm.ep}, O, n, b->M, C * P, (int)P, EPI_C64,
                  inverse ? 1 : 0, shift_out ? n / 2 : 0, scale, 0, n};
  pl->launches = 3 + b->fwdM->launches + b->invM->launches;
  pl->segments = 0;
  *out = pl;
  return PBK_OK;
}

extern "C" int pbk_fft_plan_create(int64_t outer, int64_t n, int64_t inner, int32_t inverse,
                                   int32_t device, pbk_plan** plan) {
  if (!plan) return fail(PBK_ERR_INVALID, "plan is NULL");
  if (outer <= 0 || n <= 0 || inner <= 0) return fail(PBK_ERR_INVALID, "shape must be positive");
  ExtMap in{n * inner, inner, 1, 0};
  ExtMap om{n * inner, inner, 1, 0};
  const float scale = inverse ? (float)(1.0 / (double)n) : 1.0f;
  return build_fft_plan(outer, n, inner, 1, inverse != 0, in, om, scale, false, false, device,
                        plan);
}

static int stft_plan_create(int64_t nseg, int64_t nperseg, int64_t nchan, int64_t npol,
                            int32_t inverse, int32_t in_dtype, int32_t device, pbk_plan** plan) {
  if (!plan) return fail(PBK_ERR_INVALID, "plan is NULL");
  if (nseg <= 0 || nperseg <= 0 || nchan <= 0 || npol <= 0)
    return fail(PBK_ERR_INVALID, "shape must be positive");
  if (in_dtype != PBK_C64 && in_dtype != PBK_I8X2 && in_dtype != PBK_U4X2 && in_dtype != PBK_U2X2)
    return fail(PBK_ERR_INVALID, "unknown in_dtype %d", in_dtype);
  if (in_dtype != PBK_C64 && inverse)
    return fail(PBK_ERR_INVALID, "raw input applies to the forward transform only");
  if ((in_dtype == PBK_U4X2 || in_dtype == PBK_U2X2) && (nchan * npol) % 2)
    return fail(PBK_ERR_INVALID, "packed input needs an even nchan * npol, got %lld",
                (long long)(nchan * npol));
  const long long n = nperseg, C = nchan, P = npol;
  if (!inverse && in_dtype == PBK_C64 && C == 1 && P == 1 && n % 2 == 0 &&
      ilog2_exact(n / 2) >= 1 && !getenv("PBK_NO_SPLIT")) {
    // one single-pol column has no lane pair; its even and odd samples do (see
    // pbk_stft_detect_plan_create): half-length plan on the (n/2, 2) view, recombined in the
    // last pass.  Only power-of-two halves have that last pass (a Bluestein plan would return
    // the two half-length spectra unrecombined).  Shapes it does not cover fall through to the
    // plan below (generic kernels).
    DetectSpec det;
    det.split = det.volt = true;
    const long long h = n / 2;
    ExtMap in{h * 2, 2, 2, 1};
    ExtMap om{h * 2, 2, h * 2, 1};     // unused: the recombining store has its own output map
    const int rc = build_fft_plan(nseg, h, 1, 2, false, in, om, (float)(1.0 / (double)n), false,
                                  false, device, plan, LOAD_C64, &det);
    if (rc != PBK_ERR_UNSUPPORTED) return rc;
  }
  if (!inverse) {
    // in[(s*n + t), c, p] ; out[s, c*n + shift(k), p] ; scale 1/n   (misc.py:41-52)
    ExtMap in{n * C * P, C * P, P, 1};
    ExtMap om{C * n * P, P, n * P, 1};
    return build_fft_plan(nseg, n, C, P, false, in, om, (float)(1.0 / (double)n), true, false,
                          device, plan, load_kind_of(in_dtype));
  }
  // in[s, c*n + k', p] with ifftshift ; out[(s*n + t), c, p] ; (x*n) then ifft => unit scale
  ExtMap in{C * n * P, P, n * P, 1};
  ExtMap om{n * C * P, C * P, P, 1};
  return build_fft_plan(nseg, n, C, P, true, in, om, 1.0f, false, true, device, plan);
}

extern "C" int pbk_stft_plan_create(int64_t nseg, int64_t nperseg, int64_t nchan, int64_t npol,
                                    int32_t inverse, int32_t device, pbk_plan** plan) {
  return stft_plan_create(nseg, nperseg, nchan, npol, inverse, PBK_C64, device, plan);
}

extern "C" int pbk_stft_detect_plan_create(int64_t nseg, int64_t nperseg, int64_t nchan,
                                           int64_t npol, int32_t out_kind, int64_t freq_sum,
                                           int32_t device, pbk_plan** plan) {
  if (!plan) return fail(PBK_ERR_INVALID, "plan is NULL");
  if (nseg <= 0 || nperseg <= 0 || nchan <= 0 || npol <= 0 || freq_sum < 1)
    return fail(PBK_ERR_INVALID, "shape must be positive");
  if (out_kind != PBK_OUT_INTENSITY && out_kind != PBK_OUT_STOKES_I)
    return fail(PBK_ERR_INVALID, "out_kind must be INTENSITY or STOKES_I");
  if (out_kind == PBK_OUT_STOKES_I && npol != 2)
    return fail(PBK_ERR_INVALID, "Stokes I needs npol == 2");
  if (nchan != 1 || (npol != 1 && npol != 2) || nperseg % 2)
    return fail(PBK_ERR_UNSUPPORTED, "fused detection is built for one channel of one or two "
                "polarisations and an even segment length");
  const long long n = nperseg;
  DetectSpec det;
  det.fsum = freq_sum;
  if (npol == 1) {
    // one single-pol column: its even and odd samples are a lane pair -- the (n/2, 2) view of the
    // same memory is channelized at half length and the radix-2 recombination X[k] = E + wO,
    // X[k + n/2] = E - wO happens in registers in front of the detection (the same trick as the
    // single-column dedispersion plan)
    det.pq = 1;
    det.split = true;
    const long long h = n / 2;
    ExtMap in{h * 2, 2, 2, 1};
    ExtMap om{h * 2, 2, h * 2, 1};     // unused: the detected epilogue has its own output map
    return build_fft_plan(nseg, h, 1, 2, false, in, om, (float)(1.0 / (double)n), false, false,
                          device, plan, LOAD_C64, &det);
  }
  det.pq = out_kind == PBK_OUT_STOKES_I ? 1 : 2;
  ExtMap in{n * 2, 2, 2, 1};
  ExtMap om{n * 2, 2, n * 2, 1};
  return build_fft_plan(nseg, n, 1, 2, false, in, om, (float)(1.0 / (double)n), true, false,
                        device, plan, LOAD_C64, &det);
}

extern "C" int pbk_stft_plan_create_raw(int64_t nseg, int64_t nperseg, int64_t nchan,
                                        int64_t npol, int32_t in_dtype, int32_t device,
                                        pbk_plan** plan) {
  return stft_plan_create(nseg, nperseg, nchan, npol, 0, in_dtype, device, plan);
}

extern "C" int pbk_fft_exec_device(pbk_plan* pl, const void* d_in, void* d_out, void* stream) {
  if (!pl || pl->kind != PLAN_FFT) return fail(PBK_ERR_INVALID, "not an FFT plan");
  if (!d_in || !d_out) return fail(PBK_ERR_INVALID, "NULL data pointer");
  CUDA_TRY(cudaSetDevice(pl->device));
  if (pl->blue) return blue_exec(pl, d_in, d_out, nullptr, reinterpret_cast<cudaStream_t>(stream));
  if (d_in == d_out && pl->passes.size() == 1)
    return fail(PBK_ERR_INVALID, "single-pass transforms cannot run in place");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (!(last_pass_needs_fast(pl) && misaligned16(d_out)))
    return run_passes(pl, d_in, d_out, nullptr, st);
  int rc = stage_ensure(pl, pl->out_bytes);   // detecting or even / odd last pass: see stage_ensure
  if (rc == PBK_OK) rc = run_passes(pl, d_in, pl->d_stage, nullptr, st);
  if (rc != PBK_OK) return rc;
  CUDA_TRY(cudaMemcpyAsync(d_out, pl->d_stage, pl->out_bytes, cudaMemcpyDeviceToDevice, st));
  return PBK_OK;
}

extern "C" int pbk_stft_fold_exec_device(pbk_plan* pl, const void* d_in, void* d_profile,
                                         void* d_counts, const double* coeffs, int32_t ncoef,
                                         double sample_rate_hz, int64_t n0, int32_t nbin,
                                         void* stream) {
  if (!pl || pl->kind != PLAN_FFT || pl->det_pq == 0)
    return fail(PBK_ERR_INVALID, "not a detected channelizer plan");
  if (!d_in || !d_profile || !d_counts || !coeffs) return fail(PBK_ERR_INVALID, "NULL pointer");
  if (nbin <= 0) return fail(PBK_ERR_INVALID, "nbin must be positive");
  if (ncoef < 1 || ncoef > kFoldMaxCoef)
    return fail(PBK_ERR_INVALID, "ncoef must be in [1, %d]", kFoldMaxCoef);
  if (!(sample_rate_hz > 0) || !std::isfinite(sample_rate_hz))
    return fail(PBK_ERR_INVALID, "sample_rate_hz must be finite and > 0");
  for (int i = 0; i < ncoef; ++i)
    if (!std::isfinite(coeffs[i]))
      return fail(PBK_ERR_INVALID, "phase coefficient %d is not finite", i);
  CUDA_TRY(cudaSetDevice(pl->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (!pl->d_segbins) CUDA_TRY(cudaMalloc(&pl->d_segbins, (size_t)pl->det_nseg * sizeof(int)));
  FoldArgs fa;
  memset(&fa, 0, sizeof(fa));
  for (int i = 0; i < ncoef; ++i) fa.coef[i] = coeffs[i];
  fa.ncoef = ncoef;
  fa.sample_rate = sample_rate_hz;
  fa.n0 = n0;
  fa.nbin = nbin;
  fa.nsamp = pl->det_nseg;
  fa.row_elems = pl->det_cells * pl->det_pq;
  fold_args_finish(fa);
  fa.counts = reinterpret_cast<unsigned long long*>(d_counts);
  const unsigned blocks = (unsigned)std::min<long long>((pl->det_nseg + 255) / 256, 148 * 4);
  fold_bins_kernel<<<blocks, 256, 0, st>>>(fa, pl->d_segbins);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "fold bins launch: %s", cudaGetErrorString(e));
  // a profile aligned only to its float32 elements is accumulated in the plan's aligned staging
  // buffer: copied in, added to by the detecting pass, copied back
  void* prof = d_profile;
  const size_t prof_bytes = (size_t)nbin * pl->det_cells * pl->det_pq * sizeof(float);
  if (misaligned16(d_profile)) {
    int rc = stage_ensure(pl, prof_bytes);
    if (rc != PBK_OK) return rc;
    prof = pl->d_stage;
    CUDA_TRY(cudaMemcpyAsync(prof, d_profile, prof_bytes, cudaMemcpyDeviceToDevice, st));
  }
  pl->exec_segbins = pl->d_segbins;
  const int rc = run_passes(pl, d_in, prof, nullptr, st);
  pl->exec_segbins = nullptr;
  if (rc != PBK_OK) return rc;
  if (prof != d_profile)
    CUDA_TRY(cudaMemcpyAsync(d_profile, prof, prof_bytes, cudaMemcpyDeviceToDevice, st));
  return PBK_OK;
}

extern "C" int pbk_fft_exec_host(pbk_plan* pl, const void* in, void* out) {
  if (!pl || pl->kind != PLAN_FFT) return fail(PBK_ERR_INVALID, "not an FFT plan");
  if (!in || !out) return fail(PBK_ERR_INVALID, "NULL data pointer");
  std::lock_guard<std::mutex> lock(pl->mu);
  CUDA_TRY(cudaSetDevice(pl->device));
  int rc;
  if ((rc = ensure_buf(&pl->h_din, pl->in_bytes)) != PBK_OK) return rc;
  if ((rc = ensure_buf(&pl->h_dout, pl->out_bytes)) != PBK_OK) return rc;
  cudaStream_t st = cudaStreamPerThread;
  CUDA_TRY(host_to_device(pl->h_din, in, pl->in_bytes, st));
  rc = pbk_fft_exec_device(pl, pl->h_din, pl->h_dout, st);
  if (rc != PBK_OK) return rc;
  CUDA_TRY(device_to_host(out, pl->h_dout, pl->out_bytes, st));
  return PBK_OK;
}

static void prof_free(pbk_plan* pl) {
  for (auto& set : pl->prof)
    for (auto ev : set) cudaEventDestroy(ev);
  pl->prof.clear();
  pl->prof_next = 0;
  pl->prof_cur = -1;
}

extern "C" int pbk_plan_profile(pbk_plan* pl, int32_t nslots) {
  if (!pl) return fail(PBK_ERR_INVALID, "plan is NULL");
  if (nslots < 0 || nslots > 4096) return fail(PBK_ERR_INVALID, "nslots must be in [0, 4096]");
  std::lock_guard<std::mutex> lock(pl->mu);
  CUDA_TRY(cudaSetDevice(pl->device));
  prof_free(pl);
  pl->prof.resize(nslots);
  for (auto& set : pl->prof) {
    set.resize(pl->segments + 1);
    for (auto& ev : set) CUDA_TRY(cudaEventCreate(&ev));
  }
  return PBK_OK;
}

extern "C" int pbk_plan_profile_read(pbk_plan* pl, int32_t slot, float* ms, int32_t n) {
  if (!pl || !ms) return fail(PBK_ERR_INVALID, "NULL argument");
  if (slot < 0 || slot >= (int)pl->prof.size()) return fail(PBK_ERR_INVALID, "bad slot %d", slot);
  if (n < pl->segments) return fail(PBK_ERR_INVALID, "need room for %d segments", pl->segments);
  CUDA_TRY(cudaSetDevice(pl->device));
  const auto& set = pl->prof[slot];
  for (int i = 0; i < pl->segments; ++i) {
    ms[i] = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms[i], set[i], set[i + 1]));
  }
  return PBK_OK;
}

struct FdmtPlan;
static void fdmt_destroy(FdmtPlan* f);
static size_t fdmt_bytes(const FdmtPlan* f);
static int fdmt_describe(const FdmtPlan* f, char* buf, size_t n);

extern "C" void pbk_plan_destroy(pbk_plan* pl) {
  if (!pl) return;
  cudaSetDevice(pl->device);
  prof_free(pl);
  blue_free(pl->blue);
  cudaFree(pl->scratch);
  cudaFree(pl->scratch2);
  cudaFree(pl->blk_scratch[0]);
  cudaFree(pl->blk_scratch[1]);
  cudaFree(pl->d_tw);
  cudaFree(pl->d_ftab);
  cudaFree(pl->d_chanfreq);
  cudaFree(pl->d_chanconst);
  cudaFree(pl->d_ramp_shift);
  cudaFree(pl->d_ramp_zero);
  cudaFree(pl->d_tmpf);
  cudaFree(pl->d_segbins);
  cudaFree(pl->d_foldbuf);
  cudaFree(pl->d_stage);
  cudaFree(pl->d_incoh);
  fdmt_destroy(pl->fdmt);
  cudaFree(pl->h_din);
  cudaFree(pl->h_dout);
  cudaFree(pl->h_dchirp);
  delete pl;
}

extern "C" int pbk_plan_info(const pbk_plan* pl, int32_t* launches, int64_t* workspace_bytes,
                             int32_t* levels, int32_t* level_log2) {
  if (!pl) return fail(PBK_ERR_INVALID, "plan is NULL");
  if (launches) *launches = pl->launches;
  if (workspace_bytes) *workspace_bytes =
      (int64_t)(pl->scratch_bytes * (pl->scratch2 ? 2 : 1) +
                (pl->work_bytes > pl->scratch_bytes ? pl->work_bytes - pl->scratch_bytes : 0) +
                pl->blk_bytes * ((pl->blk_scratch[0] ? 1 : 0) + (pl->blk_scratch[1] ? 1 : 0)) +
                pl->tmpf_bytes + pl->fold_bytes +
                pl->stage_bytes + pl->incoh_bytes + fdmt_bytes(pl->fdmt));
  if (levels) *levels = pl->nlevels;
  if (level_log2)
    for (int i = 0; i < 3; ++i) level_log2[i] = pl->level_log2[i];
  return PBK_OK;
}

extern "C" int pbk_plan_describe(const pbk_plan* pl, char* buf, size_t n) {
  if (!pl || !buf || n == 0) return fail(PBK_ERR_INVALID, "NULL argument");
  size_t off = 0;
  buf[0] = 0;
  if (pl->kind == PLAN_FDMT) return fdmt_describe(pl->fdmt, buf, n);
  if (pl->kind == PLAN_INCOH) {
    const pbk_incoh::Args& a = pl->incoh;
    snprintf(buf, n, "INCOH:ndm=%d:C=%d:P=%d:rows=%d:KD=%d:TT=%d:CC=%d:smem=%zu:tiles=%u", pl->ndm,
             a.C, a.P, a.rows, pl->incoh_kd, a.TT, a.CC, pl->incoh_smem, pl->incoh_grid);
    return PBK_OK;
  }
  if (pl->blue) {
    snprintf(buf, n, "BLUESTEIN:n=%lld:M=2^%d:lanes=%lld", pl->blue->n, ilog2_exact(pl->blue->M),
             pl->blue->I);
    if (pl->trials) {
      off = strlen(buf);
      snprintf(buf + off, n - off, ":trials=%d:per_launch=%d", pl->ndm, pl->trials_per_launch);
    }
    return PBK_OK;
  }
  for (size_t i = 0; i < pl->passes.size() && off + 1 < n; ++i) {
    const Pass& ps = pl->passes[i];
    const char* mode = ps.mode == MODE_FWD ? "FWD" : ps.mode == MODE_MID ? "MID" : "INV";
    int w;
    // a trial plan lists its shared passes, then "TRIALS" and the passes that run per trial
    if (pl->trials && (int)i == pl->nshared) {
      w = snprintf(buf + off, n - off, "%sTRIALS:ndm=%d:per_launch=%d", i == 0 ? "" : ";",
                   pl->ndm, pl->trials_per_launch);
      if (w < 0 || off + (size_t)w + 1 >= n) break;
      off += (size_t)w;
    }
    const bool first = i == 0 && !(pl->trials && pl->nshared == 0);
    const char* sep = first ? "" : ";";
    if (ps.family >= 0)
      w = snprintf(buf + off, n - off, "%s%s:L=2^%d:%s:W=%d:tiles=%lld:threads=%d%s%s", sep,
                   mode, ps.a.log2L, ps.tma ? "tma-r16" : "fast-r16",
                   2 << ps.finfo.log2pw, ps.ntiles, ps.tma ? ps.tinfo.threads : ps.finfo.threads,
                   ps.a.tsum_log2 > 0 ? ":timesum" : "",
                   ps.a.split || ps.a.fsum_split ? ":evenodd" : "");
    else
      w = snprintf(buf + off, n - off, "%s%s:L=2^%d:%s:W=%d:tiles=%u:threads=%d", sep,
                   mode, ps.a.log2L, ps.fast ? "generic-vec" : "generic", 2 << ps.a.log2pw,
                   ps.grid, kThreads);
    if (w < 0) break;
    off += (size_t)w;
  }
  return PBK_OK;
}

extern "C" int pbk_plan_segments(const pbk_plan* pl, int32_t* segments) {
  if (!pl || !segments) return fail(PBK_ERR_INVALID, "NULL argument");
  *segments = pl->segments;
  return PBK_OK;
}

// ------------------------------------------------------------------------------------------
// incoherent dedispersion at many trial DMs, summed over frequency (pbk_incoh.cuh)
// ------------------------------------------------------------------------------------------
// Shared memory of one CTA is at most this much, so that two CTAs fit an SM whatever the span.
static constexpr size_t kIncohSmemCap = 100 * 1024;

// Block tables of one (KD, CC) choice over the trials in sorted order; returns the shared memory
// one CTA needs.
static size_t incoh_tables(const std::vector<int>& order, const int64_t* delays, int ndm, int C,
                           int P, int KD, int CC, std::vector<int>& tab, int* stride_out) {
  const int nb = (ndm + KD - 1) / KD, nq = (C + CC - 1) / CC;
  tab.assign((size_t)nb * KD + (size_t)nb * KD * C + 2 * (size_t)nb * nq, 0);
  int* perm = tab.data();
  int* off = perm + (size_t)nb * KD;
  int* lo = off + (size_t)nb * KD * C;
  int* ext = lo + (size_t)nb * nq;
  long long ext_max = 0;
  for (int b = 0; b < nb; ++b)
    for (int q = 0; q < nq; ++q) {
      long long mn = LLONG_MAX, mx = LLONG_MIN;
      for (int s = b * KD; s < std::min(ndm, (b + 1) * KD); ++s)
        for (int c = q * CC; c < std::min(C, (q + 1) * CC); ++c) {
          const long long d = delays[(size_t)order[s] * C + c];
          mn = std::min(mn, d);
          mx = std::max(mx, d);
        }
      lo[b * nq + q] = (int)mn;
      ext[b * nq + q] = (int)(mx - mn);
      ext_max = std::max(ext_max, mx - mn);
    }
  for (int s = 0; s < nb * KD; ++s) {
    perm[s] = s < ndm ? order[s] : -1;
    for (int c = 0; c < C; ++c)
      off[(size_t)s * C + c] =
          s < ndm ? (int)(delays[(size_t)order[s] * C + c] - lo[(s / KD) * nq + c / CC]) : 0;
  }
  // a staged channel holds ext + TT rows of P floats; any accumulator index < kFlat stays inside.
  // The stride is padded so that the staging stores of a warp hit distinct banks: with 16 floats
  // per staged row (CC * P == 16) a warp stores two rows, which stride = 2P (mod 32) separates.
  long long stride = ext_max * P + pbk_incoh::kFlat;
  if (stride > INT_MAX / 2) return SIZE_MAX;
  const int want = CC * P == 16 ? (2 * P) % 32 : 1;
  while ((int)(stride % 32) != want) ++stride;
  *stride_out = (int)stride;
  return (size_t)stride * CC * sizeof(float);
}

extern "C" int pbk_incoh_trials_plan_create(int64_t nsamp_in, int64_t nchan, int64_t npol,
                                            int64_t rows, const int64_t* delays, int32_t ndm,
                                            int32_t device, pbk_plan** out) {
  if (!delays || !out) return fail(PBK_ERR_INVALID, "NULL pointer");
  *out = nullptr;
  if (ndm < 1 || nchan < 1 || npol < 1 || nsamp_in < 0 || rows < 0)
    return fail(PBK_ERR_INVALID, "bad shape (ndm, nchan and npol must be >= 1, rows >= 0)");
  for (int64_t i = 0; i < (int64_t)ndm * nchan; ++i)
    if (delays[i] < 0 || delays[i] > nsamp_in - rows)
      return fail(PBK_ERR_INVALID, "delay[%lld][%lld] = %lld reads outside the input of %lld rows",
                  (long long)(i / nchan), (long long)(i % nchan), (long long)delays[i],
                  (long long)nsamp_in);
  if (rows > INT_MAX || nsamp_in > INT_MAX || nchan > INT_MAX)
    return fail(PBK_ERR_UNSUPPORTED, "rows, delays and channels must fit 32-bit indices");
  if (npol > pbk_incoh::kMaxP)
    return fail(PBK_ERR_UNSUPPORTED, "npol = %lld: at most %d floats per cell", (long long)npol,
                pbk_incoh::kMaxP);
  const int C = (int)nchan, P = (int)npol;
  // sorted by sweep (the delay of the first channel less that of the last, monotone in DM for a
  // fixed reference frequency), so that a block of KD trials spans few rows
  std::vector<int> order(ndm);
  for (int k = 0; k < ndm; ++k) order[k] = k;
  std::stable_sort(order.begin(), order.end(), [&](int x, int y) {
    const int64_t* dx = delays + (size_t)x * C;
    const int64_t* dy = delays + (size_t)y * C;
    const int64_t sx = dx[0] - dx[C - 1], sy = dy[0] - dy[C - 1];
    return sx != sy ? sx < sy : dx[0] < dy[0];
  });
  // the largest tile that fits: KD shrinks first, then CC; KD = CC = 1 stages TT rows of one
  // channel (ext = 0) and always fits
  std::vector<int> tab;
  int KD = 0, CC = 0, stride = 0;
  size_t smem = 0;
  for (int cc = std::min(C, std::max(1, 16 / P)); cc >= 1 && !KD; cc = cc > 1 ? cc / 2 : 0)
    for (int kd = 8; kd >= 1 && !KD; kd /= 2) {
      if (kd > 1 && ndm <= kd / 2) continue;    // half the warps would idle
      smem = incoh_tables(order, delays, ndm, C, P, kd, cc, tab, &stride);
      if (smem <= kIncohSmemCap) KD = kd, CC = cc;
    }
  if (!KD) return fail(PBK_ERR_UNSUPPORTED, "no tile fits shared memory");
  const int TT = pbk_incoh::kFlat / P;
  const long long nb = (ndm + KD - 1) / KD, ntiles = (rows + TT - 1) / TT;
  if (nb * ntiles > INT_MAX) return fail(PBK_ERR_UNSUPPORTED, "too many tiles for one launch");
  CUDA_TRY(cudaSetDevice(device));
  pbk_plan* pl = new pbk_plan();
  pl->kind = PLAN_INCOH;
  pl->device = device;
  pl->ndm = ndm;
  auto cleanup = [&](int code) { pbk_plan_destroy(pl); return code; };
  pl->incoh_bytes = tab.size() * sizeof(int);
  cudaError_t e = cudaMalloc(&pl->d_incoh, pl->incoh_bytes);
  if (e == cudaSuccess)
    e = cudaMemcpy(pl->d_incoh, tab.data(), pl->incoh_bytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(pbk_incoh::kernel_of(KD), cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)kIncohSmemCap);   // the cap, never less: other plans share it
  if (e != cudaSuccess)
    return cleanup(fail(e == cudaErrorMemoryAllocation ? PBK_ERR_NOMEM : PBK_ERR_CUDA,
                        "incoherent trial plan: %s", cudaGetErrorString(e)));
  pbk_incoh::Args& a = pl->incoh;
  a.row_elems = (long long)C * P;
  a.C = C, a.P = P, a.rows = (int)rows, a.TT = TT, a.CC = CC, a.nq = (C + CC - 1) / CC;
  a.stride = stride;
  a.nb = (int)nb;
  a.perm = pl->d_incoh;
  a.off = a.perm + nb * KD;
  a.lo = a.off + nb * KD * C;
  a.ext = a.lo + nb * a.nq;
  pl->incoh_kd = KD;
  pl->incoh_grid = (unsigned)(nb * ntiles);
  pl->incoh_smem = smem;
  pl->launches = rows > 0 ? 1 : 0;
  pl->in_bytes = (size_t)nsamp_in * C * P * sizeof(float);
  pl->out_bytes = (size_t)ndm * rows * P * sizeof(float);
  *out = pl;
  return PBK_OK;
}

extern "C" int pbk_incoh_trials_exec_device(pbk_plan* pl, const void* d_in, void* d_out,
                                            void* stream) {
  if (!pl || pl->kind != PLAN_INCOH) return fail(PBK_ERR_INVALID, "not an incoherent-trials plan");
  if (!d_in || !d_out) return fail(PBK_ERR_INVALID, "NULL data pointer");
  if (((uintptr_t)d_in | (uintptr_t)d_out) & 3)
    return fail(PBK_ERR_INVALID, "float32 arrays must be 4-byte aligned");
  if (pl->incoh.rows == 0) return PBK_OK;
  CUDA_TRY(cudaSetDevice(pl->device));
  pbk_incoh::Args a = pl->incoh;
  a.in = reinterpret_cast<const float*>(d_in);
  a.out = reinterpret_cast<float*>(d_out);
  cudaError_t e = pbk_incoh::launch(pl->incoh_kd, a, pl->incoh_grid, pl->incoh_smem,
                                    reinterpret_cast<cudaStream_t>(stream));
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "incoherent trials launch: %s", cudaGetErrorString(e));
  return PBK_OK;
}

extern "C" int pbk_incoh_trials_exec_host(pbk_plan* pl, const void* in, void* out) {
  if (!pl || pl->kind != PLAN_INCOH) return fail(PBK_ERR_INVALID, "not an incoherent-trials plan");
  if (!in || !out) return fail(PBK_ERR_INVALID, "NULL data pointer");
  if (pl->incoh.rows == 0) return PBK_OK;
  std::lock_guard<std::mutex> lock(pl->mu);
  CUDA_TRY(cudaSetDevice(pl->device));
  int rc;
  if ((rc = ensure_buf(&pl->h_din, pl->in_bytes)) != PBK_OK) return rc;
  if ((rc = ensure_buf(&pl->h_dout, pl->out_bytes)) != PBK_OK) return rc;
  cudaStream_t st = cudaStreamPerThread;
  CUDA_TRY(host_to_device(pl->h_din, in, pl->in_bytes, st));
  if ((rc = pbk_incoh_trials_exec_device(pl, pl->h_din, pl->h_dout, st)) != PBK_OK) return rc;
  CUDA_TRY(device_to_host(out, pl->h_dout, pl->out_bytes, st));
  return PBK_OK;
}

// ------------------------------------------------------------------------------------------
// fast dispersion measure transform (pbk_fdmt.cuh, tables from pbk_fdmt_tables.cu)
// ------------------------------------------------------------------------------------------
// Shared memory of one fused CTA is at most this much, so that two CTAs fit an SM.
static constexpr size_t kFdmtSmemCap = 100 * 1024;

struct FdmtPlan {
  pbk_fdmt::Tables t;
  long long nsamp = 0, D = 0, d_min = 0;
  int C = 0, P = 0, k = 0, T = 0;
  size_t smem = 0;
  int bufB_floats = 0;
  long long J = 0;              // output rows per chunk
  int nchunks = 0;
  long long stride = 0;         // floats per state row
  size_t buf_bytes = 0;         // each state buffer
  float* buf[2] = {nullptr, nullptr};
  int* d_tab = nullptr;         // row0, row0_off, nnodes, ent_off, then int4 entries and last
  size_t tab_bytes = 0;
  std::vector<long long> ent_off;   // per level, in int4 entries
  long long last_off = 0;
  int row0_off_at = 0, nnodes_at = 0, ent_off_at = 0, ent_at = 0;   // int offsets in d_tab
};

static void fdmt_destroy(FdmtPlan* f) {
  if (!f) return;
  cudaFree(f->buf[0]);
  cudaFree(f->buf[1]);
  cudaFree(f->d_tab);
  delete f;
}

static size_t fdmt_bytes(const FdmtPlan* f) {
  return f ? f->tab_bytes + f->buf_bytes * ((f->buf[0] ? 1 : 0) + (f->buf[1] ? 1 : 0)) : 0;
}

static int fdmt_describe(const FdmtPlan* f, char* buf, size_t n) {
  snprintf(buf, n, "FDMT:C=%d:P=%d:D=%lld:levels=%d:fused=%d:T=%d:smem=%zu:chunks=%d:rows=%lld",
           f->C, f->P, f->D, f->t.L, f->k, f->T, f->smem, f->nchunks, f->t.rows);
  return PBK_OK;
}

// Shared floats of the fused kernel at fusion depth k and tile T over every level-k node, and the
// offset of its second buffer; 0 when some node's subtree cannot be held.
static size_t fdmt_fused_smem(const pbk_fdmt::Tables& t, int k, int T, int P, int* bufB) {
  if (k == 0) { *bufB = 0; return 0; }
  long long a_max = 0, b_max = 0;
  for (int n = 0; n < t.nnodes[k]; ++n) {
    const long long H = t.row0[k][n + 1] - t.row0[k][n] - 1, WT = T + H;
    long long rm = 0;
    for (int l = 0; l <= k; ++l) {
      const int s = k - l;
      rm = std::max<long long>(rm, t.row0[l][std::min((n + 1) << s, t.nnodes[l])] - t.row0[l][n << s]);
    }
    const int ca = n << k, cb = std::min((n + 1) << k, t.C);
    long long nl = 1;
    for (int c = ca; c < cb; ++c) nl = std::max<long long>(nl, t.row0[0][c + 1] - t.row0[0][c]);
    a_max = std::max(a_max, rm * WT * P);
    b_max = std::max(b_max, std::max(rm * WT * P, (WT + nl - 1) * (cb - ca) * P));
    if (a_max + b_max > (long long)(kFdmtSmemCap / sizeof(float))) return 0;
  }
  a_max = (a_max + 3) & ~3LL;
  *bufB = (int)a_max;
  return (size_t)(a_max + b_max) * sizeof(float);
}

// Largest tile (a multiple of 32, at most 2048 times) that fits at depth k; 0 if none.
static int fdmt_tile(const pbk_fdmt::Tables& t, int k, int P, long long wlen) {
  if (k == 0) return 1024;
  int best = 0, b;
  for (int T = 32; T <= 2048 && T < wlen + 32; T += 32)
    if (fdmt_fused_smem(t, k, T, P, &b)) best = T; else break;
  return best;
}

extern "C" int pbk_fdmt_plan_create(int64_t nsamp, int64_t nchan, int64_t npol, double f_lo_hz,
                                    double f_hi_hz, double ref_freq_hz, int64_t max_delay,
                                    int64_t d_min, int64_t max_workspace_bytes, int32_t device,
                                    pbk_plan** out) {
  if (!out) return fail(PBK_ERR_INVALID, "NULL pointer");
  *out = nullptr;
  if (nsamp < 1 || nchan < 1 || npol < 1)
    return fail(PBK_ERR_INVALID, "bad shape (nsamp, nchan and npol must be >= 1)");
  if (!(f_lo_hz > 0) || !(f_hi_hz > f_lo_hz) || !std::isfinite(f_hi_hz))
    return fail(PBK_ERR_INVALID, "need 0 < f_lo < f_hi");
  if (!(ref_freq_hz > 0) || !std::isfinite(ref_freq_hz))
    return fail(PBK_ERR_INVALID, "ref_freq must be positive and finite");
  if (max_delay < 0 || d_min < 0 || d_min > max_delay)
    return fail(PBK_ERR_INVALID, "need 0 <= d_min <= max_delay");
  if (max_workspace_bytes < 0) return fail(PBK_ERR_INVALID, "negative workspace cap");
  if (nsamp > INT_MAX || nchan > INT_MAX || npol > INT_MAX || max_delay >= INT_MAX - nsamp)
    return fail(PBK_ERR_UNSUPPORTED, "nsamp, nchan, npol and nsamp + max_delay must fit 32-bit indices");
  CUDA_TRY(cudaSetDevice(device));    // before anything is allocated: nothing to free on failure
  FdmtPlan* f = new FdmtPlan();
  auto drop = [&](int code) { fdmt_destroy(f); return code; };
  const int C = (int)nchan, P = (int)npol;
  if (pbk_fdmt::build_tables(nsamp, C, f_lo_hz, f_hi_hz, ref_freq_hz, max_delay, d_min, &f->t))
    return drop(fail(PBK_ERR_UNSUPPORTED, "state rows or shifts beyond 32-bit indices"));
  const pbk_fdmt::Tables& t = f->t;
  f->nsamp = nsamp, f->D = max_delay, f->d_min = d_min, f->C = C, f->P = P;
  const long long ndm = max_delay - d_min + 1, rows = t.rows;
  // rows of the largest state level the passes keep (levels k .. max(L - 1, 0))
  const int kmax = std::max(t.L - 1, 0);
  auto state_rows = [&](int k) {
    long long m = 0;
    for (int l = k; l <= kmax; ++l) m = std::max<long long>(m, t.row0[l].back());
    return m;
  };
  // fusion depth: 0, the leaves alone, which was fastest on every workload measured (DESIGN.md
  // 5.4h: the shared-memory merges pay a halo of the node's largest row per tile and run two CTAs
  // per SM); PBK_FDMT_FUSED=k forces k merges in the first kernel (developer knob)
  const long long spread = (long long)t.s_max - t.s_min;
  const long long wfull = std::min<long long>(nsamp, rows + spread + max_delay);
  int k = 0, T = fdmt_tile(t, 0, P, wfull);
  if (const char* e = getenv("PBK_FDMT_FUSED")) {
    k = atoi(e);
    if (k < 0 || k > kmax) return drop(fail(PBK_ERR_INVALID, "PBK_FDMT_FUSED=%d: 0..%d", k, kmax));
    T = fdmt_tile(t, k, P, wfull);
    if (!T) return drop(fail(PBK_ERR_UNSUPPORTED, "PBK_FDMT_FUSED=%d does not fit shared memory", k));
  }
  f->k = k, f->T = T;
  f->smem = fdmt_fused_smem(t, k, T, P, &f->bufB_floats);
  // time chunks: the largest J whose two state levels fit the cap (0: 1/5 of the device)
  size_t cap = (size_t)max_workspace_bytes;
  if (cap == 0) {
    size_t fr = 0, tot = 0;
    const cudaError_t ce = cudaMemGetInfo(&fr, &tot);
    if (ce != cudaSuccess)
      return drop(fail(PBK_ERR_CUDA, "FDMT plan: %s", cudaGetErrorString(ce)));
    cap = tot / 5;
  }
  const int nbuf = t.L - 1 > k ? 2 : 1;
  const long long srows = state_rows(k);
  auto bytes_of = [&](long long J) {
    const long long w = std::min<long long>(nsamp, J + spread + max_delay);
    const long long stride = (w * P + 3) & ~3LL;
    return (double)nbuf * srows * stride * sizeof(float);
  };
  long long J = std::max(rows, 1LL);
  if (bytes_of(J) > (double)cap) {
    long long lo = 0, hi = J;
    while (hi - lo > 1) {
      const long long mid = (lo + hi) / 2;
      if (bytes_of(mid) <= (double)cap) lo = mid; else hi = mid;
    }
    J = lo;
  }
  if (J < 1) return drop(fail(PBK_ERR_UNSUPPORTED, "workspace cap %zu bytes holds no chunk (%.0f bytes needed)", cap, bytes_of(1)));
  f->nchunks = rows > 0 ? (int)((rows + J - 1) / J) : 0;
  f->J = f->nchunks ? (rows + f->nchunks - 1) / f->nchunks : 0;
  {
    const long long w = std::min<long long>(nsamp, f->J + spread + max_delay);
    f->stride = (w * P + 3) & ~3LL;
    if (w * P > INT_MAX) return drop(fail(PBK_ERR_UNSUPPORTED, "a state row beyond 32-bit indices"));
  }
  // tables: int header then int4 entries
  std::vector<int> hdr;
  std::vector<int> row0_off(t.L + 1), ent_off_i(t.L + 1, 0);
  for (int l = 0; l <= t.L; ++l) {
    row0_off[l] = (int)hdr.size();
    hdr.insert(hdr.end(), t.row0[l].begin(), t.row0[l].end());
  }
  f->row0_off_at = (int)hdr.size();
  hdr.insert(hdr.end(), row0_off.begin(), row0_off.end());
  f->nnodes_at = (int)hdr.size();
  hdr.insert(hdr.end(), t.nnodes.begin(), t.nnodes.end());
  f->ent_off_at = (int)hdr.size();
  f->ent_off.assign(t.L + 1, 0);
  long long ne = 0;
  for (int l = 1; l <= t.L; ++l) f->ent_off[l] = ne, ne += (long long)t.ent[l].size();
  f->last_off = ne;
  if (ne + (long long)t.last.size() > INT_MAX) return drop(fail(PBK_ERR_UNSUPPORTED, "tables beyond 32-bit indices"));
  for (int l = 0; l <= t.L; ++l) ent_off_i[l] = (int)f->ent_off[l];
  hdr.insert(hdr.end(), ent_off_i.begin(), ent_off_i.end());
  while (hdr.size() % 4) hdr.push_back(0);
  f->ent_at = (int)hdr.size();
  std::vector<int4> ents;
  ents.reserve(ne + t.last.size());
  for (int l = 1; l <= t.L; ++l)
    for (const pbk_fdmt::Entry& e : t.ent[l]) ents.push_back(make_int4(e.l, e.u, e.h, e.s));
  for (const pbk_fdmt::Entry& e : t.last) ents.push_back(make_int4(e.l, e.u, e.h, e.s));
  f->tab_bytes = hdr.size() * sizeof(int) + ents.size() * sizeof(int4);
  pbk_plan* pl = new pbk_plan();
  pl->kind = PLAN_FDMT;
  pl->device = device;
  pl->ndm = (int)ndm;
  pl->fdmt = f;
  auto cleanup = [&](int code) { pbk_plan_destroy(pl); return code; };
  cudaError_t e = cudaMalloc(&f->d_tab, f->tab_bytes);
  if (e == cudaSuccess)
    e = cudaMemcpy(f->d_tab, hdr.data(), hdr.size() * sizeof(int), cudaMemcpyHostToDevice);
  if (e == cudaSuccess && !ents.empty())
    e = cudaMemcpy(f->d_tab + f->ent_at, ents.data(), ents.size() * sizeof(int4), cudaMemcpyHostToDevice);
  if (rows > 0) {
    f->buf_bytes = (size_t)srows * f->stride * sizeof(float);
    for (int b = 0; b < nbuf && e == cudaSuccess; ++b) e = cudaMalloc(&f->buf[b], f->buf_bytes);
  }
  if (e == cudaSuccess && f->smem)
    e = cudaFuncSetAttribute(pbk_fdmt::fdmt_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)kFdmtSmemCap);   // the cap, never less: other plans share it
  if (e != cudaSuccess)
    return cleanup(fail(e == cudaErrorMemoryAllocation ? PBK_ERR_NOMEM : PBK_ERR_CUDA,
                        "FDMT plan: %s", cudaGetErrorString(e)));
  pl->launches = f->nchunks * (1 + std::max(t.L - 1 - k, 0) + 1);
  pl->in_bytes = (size_t)nsamp * C * P * sizeof(float);
  pl->out_bytes = (size_t)ndm * rows * P * sizeof(float);
  *out = pl;
  return PBK_OK;
}

extern "C" int pbk_fdmt_plan_geometry(const pbk_plan* pl, int32_t* ndm, int64_t* rows,
                                      int64_t* t_lo) {
  if (!pl || pl->kind != PLAN_FDMT) return fail(PBK_ERR_INVALID, "not an FDMT plan");
  if (!ndm || !rows || !t_lo) return fail(PBK_ERR_INVALID, "NULL argument");
  *ndm = pl->ndm;
  *rows = pl->fdmt->t.rows;
  *t_lo = pl->fdmt->t.t_lo;
  return PBK_OK;
}

extern "C" int pbk_fdmt_exec_device(pbk_plan* pl, const void* d_in, void* d_out, void* stream) {
  if (!pl || pl->kind != PLAN_FDMT) return fail(PBK_ERR_INVALID, "not an FDMT plan");
  if (!d_in || !d_out) return fail(PBK_ERR_INVALID, "NULL data pointer");
  if (((uintptr_t)d_in | (uintptr_t)d_out) & 3)
    return fail(PBK_ERR_INVALID, "float32 arrays must be 4-byte aligned");
  const FdmtPlan& f = *pl->fdmt;
  const pbk_fdmt::Tables& t = f.t;
  if (t.rows == 0) return PBK_OK;
  CUDA_TRY(cudaSetDevice(pl->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int P = f.P, kmax = std::max(t.L - 1, 0);
  const int4* ents = reinterpret_cast<const int4*>(f.d_tab + f.ent_at);
  for (int ch = 0; ch < f.nchunks; ++ch) {
    const long long ja = ch * f.J, jn = std::min(f.J, t.rows - ja);
    // window: root times [t_lo + ja + s_min - D, t_lo + ja + jn + s_max), clipped at 0
    const long long ws = std::max(0LL, t.t_lo + ja + t.s_min - f.D);
    const long long we = t.t_lo + ja + jn + t.s_max;
    const int wlen = (int)(we - ws);
    pbk_fdmt::FusedArgs fa{};
    fa.x = reinterpret_cast<const float*>(d_in);
    fa.out = f.buf[0];
    fa.xrow = (long long)f.C * P;
    fa.ws = ws;
    fa.stride = f.stride;
    fa.wlen = wlen;
    fa.P = P, fa.k = f.k, fa.T = f.T, fa.nnodes = t.nnodes[f.k];
    fa.row0 = f.d_tab;
    fa.row0_off = f.d_tab + f.row0_off_at;
    fa.nnodes_l = f.d_tab + f.nnodes_at;
    fa.ent = ents;
    fa.ent_off = f.d_tab + f.ent_off_at;
    fa.bufB_floats = f.bufB_floats;
    const long long ntiles = (wlen + f.T - 1) / f.T;
    pbk_fdmt::fdmt_fused_kernel<<<(unsigned)(ntiles * fa.nnodes), dim3(32, pbk_fdmt::kFusedThreads / 32), f.smem, st>>>(fa);
    const int n = wlen * P;
    const unsigned gy = (unsigned)std::min<long long>((n + pbk_fdmt::kPassFloats - 1) / pbk_fdmt::kPassFloats, 65535);
    int cur = 0;
    for (int l = f.k + 1; l <= kmax; ++l) {
      pbk_fdmt::PassArgs pa{};
      pa.src = f.buf[cur];
      pa.dst = f.buf[cur ^ 1];
      pa.ent = ents + f.ent_off[l];
      pa.stride = f.stride;
      pa.n = n;
      pa.P = P;
      pbk_fdmt::fdmt_pass_kernel<<<dim3((unsigned)t.row0[l].back(), gy), pbk_fdmt::kThreads, 0, st>>>(pa);
      cur ^= 1;
    }
    pbk_fdmt::LastArgs la{};
    la.src = f.buf[cur];
    la.out = reinterpret_cast<float*>(d_out);
    la.ent = ents + f.last_off;
    la.stride = f.stride;
    la.rows = t.rows;
    la.base = t.t_lo + ja - ws;
    la.ja = ja;
    la.n = (int)(jn * P);
    la.P = P;
    const unsigned ly = (unsigned)std::min<long long>((la.n + pbk_fdmt::kThreads - 1) / pbk_fdmt::kThreads, 65535);
    pbk_fdmt::fdmt_last_kernel<<<dim3((unsigned)pl->ndm, ly), pbk_fdmt::kThreads, 0, st>>>(la);
  }
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "FDMT launch: %s", cudaGetErrorString(e));
  return PBK_OK;
}

extern "C" int pbk_fdmt_exec_host(pbk_plan* pl, const void* in, void* out) {
  if (!pl || pl->kind != PLAN_FDMT) return fail(PBK_ERR_INVALID, "not an FDMT plan");
  if (!in || !out) return fail(PBK_ERR_INVALID, "NULL data pointer");
  if (pl->fdmt->t.rows == 0) return PBK_OK;
  std::lock_guard<std::mutex> lock(pl->mu);
  CUDA_TRY(cudaSetDevice(pl->device));
  int rc;
  if ((rc = ensure_buf(&pl->h_din, pl->in_bytes)) != PBK_OK) return rc;
  if ((rc = ensure_buf(&pl->h_dout, pl->out_bytes)) != PBK_OK) return rc;
  cudaStream_t st = cudaStreamPerThread;
  CUDA_TRY(host_to_device(pl->h_din, in, pl->in_bytes, st));
  if ((rc = pbk_fdmt_exec_device(pl, pl->h_din, pl->h_dout, st)) != PBK_OK) return rc;
  CUDA_TRY(device_to_host(out, pl->h_dout, pl->out_bytes, st));
  return PBK_OK;
}

// ------------------------------------------------------------------------------------------
// detection, downsample, fold
// ------------------------------------------------------------------------------------------
struct DevBuf {  // RAII staging for the host-pointer variants
  void* p = nullptr;
  ~DevBuf() { if (p) cudaFree(p); }
};

extern "C" int pbk_detect(const void* in, void* out, int64_t nsamp, int64_t nchan, int64_t npol,
                          int32_t out_kind, int64_t downsample, int32_t on_device, int32_t device,
                          void* stream) {
  if (!in || !out) return fail(PBK_ERR_INVALID, "NULL data pointer");
  if (nsamp <= 0 || nchan <= 0 || npol <= 0 || downsample < 1)
    return fail(PBK_ERR_INVALID, "bad shape");
  if (out_kind != PBK_OUT_INTENSITY && out_kind != PBK_OUT_STOKES_I)
    return fail(PBK_ERR_INVALID, "out_kind must be INTENSITY or STOKES_I");
  if (out_kind == PBK_OUT_STOKES_I && npol != 2) return fail(PBK_ERR_INVALID, "Stokes I needs npol == 2");
  CUDA_TRY(cudaSetDevice(device));
  const long long rows = nsamp / downsample;
  const long long relems = out_kind == PBK_OUT_STOKES_I ? nchan : nchan * npol;
  if (rows == 0) return PBK_OK;
  if (on_device) {
    cudaError_t e = launch_detect(reinterpret_cast<const float2*>(in), reinterpret_cast<float*>(out),
                                  rows, nchan * npol, out_kind == PBK_OUT_STOKES_I, downsample,
                                  reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "detect launch: %s", cudaGetErrorString(e));
    return PBK_OK;
  }
  DevBuf di, dout;
  const size_t ib = (size_t)rows * downsample * nchan * npol * 8, ob = (size_t)rows * relems * 4;
  CUDA_TRY(cudaMalloc(&di.p, ib));
  CUDA_TRY(cudaMalloc(&dout.p, ob));
  cudaStream_t st = cudaStreamPerThread;
  CUDA_TRY(cudaMemcpyAsync(di.p, in, ib, cudaMemcpyHostToDevice, st));
  cudaError_t e = launch_detect(reinterpret_cast<const float2*>(di.p), reinterpret_cast<float*>(dout.p),
                                rows, nchan * npol, out_kind == PBK_OUT_STOKES_I, downsample, st);
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "detect launch: %s", cudaGetErrorString(e));
  CUDA_TRY(cudaMemcpyAsync(out, dout.p, ob, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return PBK_OK;
}

extern "C" int pbk_detect_scrunch(const void* in, void* out, int64_t nsamp, int64_t nchan,
                                  int64_t npol, int32_t out_kind, int64_t time_sum,
                                  int64_t freq_sum, int32_t on_device, int32_t device,
                                  void* stream) {
  if (!in || !out) return fail(PBK_ERR_INVALID, "NULL data pointer");
  if (nsamp <= 0 || nchan <= 0 || npol <= 0 || time_sum < 1 || freq_sum < 1)
    return fail(PBK_ERR_INVALID, "bad shape");
  if (nchan % freq_sum) return fail(PBK_ERR_INVALID, "freq_sum must divide nchan");
  if (out_kind != PBK_OUT_INTENSITY && out_kind != PBK_OUT_STOKES_I)
    return fail(PBK_ERR_INVALID, "out_kind must be INTENSITY or STOKES_I");
  if (out_kind == PBK_OUT_STOKES_I && npol != 2) return fail(PBK_ERR_INVALID, "Stokes I needs npol == 2");
  if (npol > INT_MAX) return fail(PBK_ERR_INVALID, "npol too large");
  CUDA_TRY(cudaSetDevice(device));
  const long long rows = nsamp / time_sum, cout = nchan / freq_sum;
  const bool stokes = out_kind == PBK_OUT_STOKES_I;
  if (rows == 0) return PBK_OK;
  if (on_device) {
    cudaError_t e = launch_detect_scrunch(reinterpret_cast<const float2*>(in),
                                          reinterpret_cast<float*>(out), rows, cout, (int)npol,
                                          stokes, time_sum, freq_sum,
                                          reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "detect launch: %s", cudaGetErrorString(e));
    return PBK_OK;
  }
  DevBuf di, dout;
  const size_t ib = (size_t)rows * time_sum * nchan * npol * 8;
  const size_t ob = (size_t)rows * cout * (stokes ? 1 : npol) * 4;
  CUDA_TRY(cudaMalloc(&di.p, ib));
  CUDA_TRY(cudaMalloc(&dout.p, ob));
  cudaStream_t st = cudaStreamPerThread;
  CUDA_TRY(cudaMemcpyAsync(di.p, in, ib, cudaMemcpyHostToDevice, st));
  cudaError_t e = launch_detect_scrunch(reinterpret_cast<const float2*>(di.p),
                                        reinterpret_cast<float*>(dout.p), rows, cout, (int)npol,
                                        stokes, time_sum, freq_sum, st);
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "detect launch: %s", cudaGetErrorString(e));
  CUDA_TRY(cudaMemcpyAsync(out, dout.p, ob, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return PBK_OK;
}

extern "C" int pbk_shift_channels(const void* in, void* out, int64_t nsamp_in, int64_t nsamp_out,
                                  int64_t nchan, int64_t cell_bytes, const int64_t* delays,
                                  int32_t on_device, int32_t device, void* stream) {
  if (!in || !out || !delays) return fail(PBK_ERR_INVALID, "NULL pointer");
  if (nsamp_in <= 0 || nsamp_out < 0 || nchan <= 0 || cell_bytes <= 0 || cell_bytes % 4)
    return fail(PBK_ERR_INVALID, "bad shape (cell_bytes must be a positive multiple of 4)");
  for (int64_t c = 0; c < nchan; ++c)
    if (delays[c] < 0 || delays[c] + nsamp_out > nsamp_in)
      return fail(PBK_ERR_INVALID, "delay[%lld] = %lld reads outside the input", (long long)c,
                  (long long)delays[c]);
  if (nsamp_out == 0) return PBK_OK;
  CUDA_TRY(cudaSetDevice(device));
  const long long words = cell_bytes / 4;
  DevBuf dd, di, dout;
  CUDA_TRY(cudaMalloc(&dd.p, (size_t)nchan * 8));
  cudaStream_t st = on_device ? reinterpret_cast<cudaStream_t>(stream) : cudaStreamPerThread;
  CUDA_TRY(cudaMemcpyAsync(dd.p, delays, (size_t)nchan * 8, cudaMemcpyHostToDevice, st));
  const void* src = in;
  void* dst = out;
  const size_t ib = (size_t)nsamp_in * nchan * cell_bytes, ob = (size_t)nsamp_out * nchan * cell_bytes;
  if (!on_device) {
    CUDA_TRY(cudaMalloc(&di.p, ib));
    CUDA_TRY(cudaMalloc(&dout.p, ob));
    CUDA_TRY(cudaMemcpyAsync(di.p, in, ib, cudaMemcpyHostToDevice, st));
    src = di.p;
    dst = dout.p;
  }
  cudaError_t e = launch_1d(shift_channels_kernel, nsamp_out * nchan * words, st,
                            reinterpret_cast<const unsigned*>(src),
                            reinterpret_cast<unsigned*>(dst), (long long)nsamp_out,
                            (long long)nchan, words, reinterpret_cast<const long long*>(dd.p));
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "shift launch: %s", cudaGetErrorString(e));
  if (!on_device) CUDA_TRY(cudaMemcpyAsync(out, dout.p, ob, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));   // the delay table is freed on return
  return PBK_OK;
}

extern "C" int pbk_downsample(const void* in, void* out, int64_t nsamp, int64_t row_elems,
                              int64_t factor, int32_t on_device, int32_t device, void* stream) {
  if (!in || !out) return fail(PBK_ERR_INVALID, "NULL data pointer");
  if (nsamp <= 0 || row_elems <= 0 || factor < 1) return fail(PBK_ERR_INVALID, "bad shape");
  CUDA_TRY(cudaSetDevice(device));
  const long long rows = nsamp / factor;
  if (rows == 0) return PBK_OK;
  if (on_device) {
    cudaError_t e = launch_downsample(reinterpret_cast<const float*>(in), reinterpret_cast<float*>(out),
                                      rows, row_elems, factor, reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "downsample launch: %s", cudaGetErrorString(e));
    return PBK_OK;
  }
  DevBuf di, dout;
  const size_t ib = (size_t)rows * factor * row_elems * 4, ob = (size_t)rows * row_elems * 4;
  CUDA_TRY(cudaMalloc(&di.p, ib));
  CUDA_TRY(cudaMalloc(&dout.p, ob));
  cudaStream_t st = cudaStreamPerThread;
  CUDA_TRY(cudaMemcpyAsync(di.p, in, ib, cudaMemcpyHostToDevice, st));
  cudaError_t e = launch_downsample(reinterpret_cast<const float*>(di.p), reinterpret_cast<float*>(dout.p),
                                    rows, row_elems, factor, st);
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "downsample launch: %s", cudaGetErrorString(e));
  CUDA_TRY(cudaMemcpyAsync(out, dout.p, ob, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return PBK_OK;
}

extern "C" int pbk_fold(const void* in, int64_t nsamp, int64_t row_elems, const double* coeffs,
                        int32_t ncoef, double sample_rate_hz, int64_t n0, int32_t nbin,
                        void* profile, void* counts, void* bins_out, int32_t on_device,
                        int32_t device, void* stream) {
  if (!in || !profile || !counts || !coeffs) return fail(PBK_ERR_INVALID, "NULL pointer");
  if (nsamp <= 0 || row_elems <= 0 || nbin <= 0) return fail(PBK_ERR_INVALID, "bad shape");
  if (ncoef < 1 || ncoef > kFoldMaxCoef)
    return fail(PBK_ERR_INVALID, "ncoef must be in [1, %d]", kFoldMaxCoef);
  if (!(sample_rate_hz > 0) || !std::isfinite(sample_rate_hz))
    return fail(PBK_ERR_INVALID, "sample_rate_hz must be finite and > 0");
  for (int i = 0; i < ncoef; ++i)
    if (!std::isfinite(coeffs[i]))
      return fail(PBK_ERR_INVALID, "phase coefficient %d is not finite", i);
  CUDA_TRY(cudaSetDevice(device));
  FoldArgs fa;
  memset(&fa, 0, sizeof(fa));
  for (int i = 0; i < ncoef; ++i) fa.coef[i] = coeffs[i];
  fa.ncoef = ncoef;
  fa.sample_rate = sample_rate_hz;
  fa.n0 = n0;
  fa.nbin = nbin;
  fa.nsamp = nsamp;
  fa.row_elems = row_elems;
  fold_args_finish(fa);
  if (on_device) {
    fa.in = reinterpret_cast<const float*>(in);
    fa.profile = reinterpret_cast<float*>(profile);
    fa.counts = reinterpret_cast<unsigned long long*>(counts);
    fa.bins_out = reinterpret_cast<int*>(bins_out);
    cudaError_t e = launch_fold(fa, reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "fold launch: %s", cudaGetErrorString(e));
    return PBK_OK;
  }
  DevBuf di, dp, dc, db;
  const size_t ib = (size_t)nsamp * row_elems * 4, pb = (size_t)nbin * row_elems * 4,
               cb = (size_t)nbin * 8, bb = (size_t)nsamp * 4;
  CUDA_TRY(cudaMalloc(&di.p, ib));
  CUDA_TRY(cudaMalloc(&dp.p, pb));
  CUDA_TRY(cudaMalloc(&dc.p, cb));
  if (bins_out) CUDA_TRY(cudaMalloc(&db.p, bb));
  cudaStream_t st = cudaStreamPerThread;
  CUDA_TRY(cudaMemcpyAsync(di.p, in, ib, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(dp.p, profile, pb, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(dc.p, counts, cb, cudaMemcpyHostToDevice, st));
  fa.in = reinterpret_cast<const float*>(di.p);
  fa.profile = reinterpret_cast<float*>(dp.p);
  fa.counts = reinterpret_cast<unsigned long long*>(dc.p);
  fa.bins_out = reinterpret_cast<int*>(db.p);
  cudaError_t e = launch_fold(fa, st);
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "fold launch: %s", cudaGetErrorString(e));
  CUDA_TRY(cudaMemcpyAsync(profile, dp.p, pb, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(counts, dc.p, cb, cudaMemcpyDeviceToHost, st));
  if (bins_out) CUDA_TRY(cudaMemcpyAsync(bins_out, db.p, bb, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return PBK_OK;
}

// ------------------------------------------------------------------------------------------
// single-pulse search: boxcar S/N at many widths, maximum over windows of starts (pbk_search.cuh)
// ------------------------------------------------------------------------------------------
// Shared memory of one boxcar CTA is at most this much, so that two CTAs fit an SM.
static constexpr size_t kBoxSmemCap = 112 * 1024;

extern "C" int pbk_boxcar_search(const void* in, int64_t nser, int64_t rows, int64_t ncols,
                                 const int32_t* widths, int32_t nwidths, int64_t window,
                                 void* stats, int32_t stats_given, void* snr, void* start,
                                 void* width, int32_t on_device, int32_t device, void* stream) {
  namespace ps = pbk_search;
  if (nser < 1 || ncols < 1 || rows < 0)
    return fail(PBK_ERR_INVALID, "bad shape (nser and ncols must be >= 1, rows >= 0)");
  if (!widths) return fail(PBK_ERR_INVALID, "widths is NULL");
  if (nwidths < 1 || nwidths > ps::kMaxWidths)
    return fail(PBK_ERR_INVALID, "nwidths = %d: 1 to %d widths", nwidths, ps::kMaxWidths);
  for (int k = 0; k < nwidths; ++k)
    if (widths[k] < 1 || (k > 0 && widths[k] <= widths[k - 1]))
      return fail(PBK_ERR_INVALID, "widths must be >= 1 and strictly increasing (widths[%d] = %d)",
                  k, widths[k]);
  if (window < 1) return fail(PBK_ERR_INVALID, "window must be >= 1");
  if (rows == 0) return PBK_OK;
  if (!in || !stats || !snr || !start || !width) return fail(PBK_ERR_INVALID, "NULL data pointer");
  if (on_device && ((((uintptr_t)in | (uintptr_t)snr | (uintptr_t)start | (uintptr_t)width) & 3) ||
                    ((uintptr_t)stats & 7)))
    return fail(PBK_ERR_INVALID, "device arrays must be aligned to their element size");
  const int wmax = widths[nwidths - 1];
  if (wmax > ps::kMaxWidth)
    return fail(PBK_ERR_UNSUPPORTED, "width %d: at most %d samples", wmax, ps::kMaxWidth);
  if (rows > INT_MAX || ncols > INT_MAX || nser > INT_MAX || nser * ncols > INT_MAX)
    return fail(PBK_ERR_UNSUPPORTED, "rows, ncols and nser * ncols must fit 32-bit indices");
  if (nser * rows > LLONG_MAX / 8 / ncols) return fail(PBK_ERR_UNSUPPORTED, "input too large");
  const int win = (int)std::min<int64_t>(window, rows);
  const int nwin = (int)((rows + win - 1) / win);
  // columns per CTA: the widest power of two <= min(ncols, 32) whose ring fits
  int CW = 32, lr = 0, R = 0;
  while (CW > ncols) CW /= 2;
  for (;; CW /= 2) {
    const int T = ps::kV * ps::kThreads / CW;
    lr = (wmax + T - 1) / T * T;
    for (R = 1; R < lr + T + 1; R *= 2) {}
    if (CW == 1 || ps::boxcar_smem(CW, R + 1) <= kBoxSmemCap) break;
  }
  const size_t smem = ps::boxcar_smem(CW, R + 1);
  const int ngroups = (int)((ncols + CW - 1) / CW);
  CUDA_TRY(cudaSetDevice(device));
  int nsm = 0;
  CUDA_TRY(cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, device));
  // runs of windows per series: enough CTAs for several waves, but runs of at least 4 (LR + T)
  // starts so that the LR samples re-read at the start of a run stay a small share
  const long long T = ps::kV * ps::kThreads / CW;
  const long long want = (8LL * nsm + nser * ngroups - 1) / (nser * ngroups);
  const long long by_halo = std::max<long long>(1, rows / (4 * (lr + T)));
  long long runs = std::max<long long>(1, std::min(std::min(want, by_halo), (long long)nwin));
  const long long wpr = (nwin + runs - 1) / runs;
  runs = (nwin + wpr - 1) / wpr;
  const long long grid = nser * ngroups * runs;
  const long long nchunks = (rows + (long long)ps::kThreads / CW * ps::kStatPer - 1) /
                            ((long long)ps::kThreads / CW * ps::kStatPer);
  if (grid > INT_MAX || nser * ngroups * nchunks > INT_MAX)
    return fail(PBK_ERR_UNSUPPORTED, "too many tiles for one launch");

  cudaStream_t st = on_device ? reinterpret_cast<cudaStream_t>(stream) : cudaStreamPerThread;
  const size_t ib = (size_t)nser * rows * ncols * 4, sb = (size_t)nser * ncols * 16,
               ob = (size_t)nser * nwin * ncols * 4;
  DevBuf di, ds, dsnr, dstart, dwidth;
  const void* x = in;
  void* d_stats = stats;
  void* d_snr = snr;
  void* d_start = start;
  void* d_width = width;
  if (!on_device) {
    CUDA_TRY(cudaMalloc(&di.p, ib));
    CUDA_TRY(cudaMalloc(&ds.p, sb));
    CUDA_TRY(cudaMalloc(&dsnr.p, ob));
    CUDA_TRY(cudaMalloc(&dstart.p, ob));
    CUDA_TRY(cudaMalloc(&dwidth.p, ob));
    CUDA_TRY(host_to_device(di.p, in, ib, st));
    if (stats_given) CUDA_TRY(host_to_device(ds.p, stats, sb, st));
    x = di.p, d_stats = ds.p, d_snr = dsnr.p, d_start = dstart.p, d_width = dwidth.p;
  }
  if (!stats_given) {
    // the partials live in a stream-ordered allocation, freed behind the kernels
    ps::StatArgs sa{};
    sa.x = reinterpret_cast<const float*>(x);
    sa.stats = reinterpret_cast<double*>(d_stats);
    sa.rows = rows, sa.ncols = ncols, sa.nseries = nser * ncols;
    sa.ngroups = ngroups, sa.nchunks = (int)nchunks;
    void* part = nullptr;
    CUDA_TRY(cudaMallocAsync(&part, (size_t)nser * ncols * nchunks * 24, st));
    sa.part = reinterpret_cast<double*>(part);
    cudaError_t e = ps::launch_stats(CW, sa, st);
    cudaError_t ef = cudaFreeAsync(part, st);
    if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "statistics launch: %s", cudaGetErrorString(e));
    CUDA_TRY(ef);
  }
  ps::BoxArgs a{};
  a.x = reinterpret_cast<const float*>(x);
  a.stats = reinterpret_cast<const double*>(d_stats);
  a.snr = reinterpret_cast<float*>(d_snr);
  a.start = reinterpret_cast<int*>(d_start);
  a.width = reinterpret_cast<int*>(d_width);
  a.rows = rows, a.ncols = ncols, a.window = win, a.nwin = nwin;
  a.ngroups = ngroups, a.runs = (int)runs, a.wpr = (int)wpr;
  a.nw = nwidths, a.wmax = wmax, a.lr = lr, a.mask = R - 1, a.rs = R + 1;
  for (int k = 0; k < nwidths; ++k) a.widths[k] = widths[k];
  CUDA_TRY(cudaFuncSetAttribute(ps::boxcar_kernel_of(CW), cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)kBoxSmemCap));
  cudaError_t e = ps::launch_boxcar(CW, a, (unsigned)grid, smem, st);
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "boxcar launch: %s", cudaGetErrorString(e));
  if (!on_device) {
    CUDA_TRY(device_to_host(snr, d_snr, ob, st));
    CUDA_TRY(device_to_host(start, d_start, ob, st));
    CUDA_TRY(device_to_host(width, d_width, ob, st));
    if (!stats_given) CUDA_TRY(device_to_host(stats, d_stats, sb, st));
  }
  return PBK_OK;
}

// ------------------------------------------------------------------------------------------
// spectral kurtosis: per-block estimate, flags and zeroing of flagged cells (pbk_sk.cuh)
// ------------------------------------------------------------------------------------------
extern "C" int pbk_spectral_kurtosis(const void* in, void* out, int64_t nsamp, int64_t nchan,
                                     int64_t npol, int32_t in_dtype, int64_t m, double nd,
                                     double lo, double hi, void* sk, void* mask, int32_t on_device,
                                     int32_t device, void* stream) {
  namespace pk = pbk_sk;
  if (in_dtype == PBK_U4X2 || in_dtype == PBK_U2X2)
    return fail(PBK_ERR_UNSUPPORTED, "spectral kurtosis of u4 / u2 input: a zeroed sample has no code");
  if (in_dtype != PBK_C64 && in_dtype != PBK_I8X2 && in_dtype != PBK_F32)
    return fail(PBK_ERR_INVALID, "in_dtype must be PBK_C64, PBK_I8X2 or PBK_F32");
  if (m < 2) return fail(PBK_ERR_INVALID, "m = %lld: at least 2 samples per block", (long long)m);
  if (!std::isfinite(nd) || nd <= 0.0) return fail(PBK_ERR_INVALID, "nd must be finite and > 0");
  if (std::isnan(lo) || std::isnan(hi) || lo > hi)
    return fail(PBK_ERR_INVALID, "thresholds must satisfy lo <= hi");
  if (nchan < 1 || npol < 1 || nsamp < 0)
    return fail(PBK_ERR_INVALID, "bad shape (nchan and npol must be >= 1, nsamp >= 0)");
  if (!out && !sk && !mask) return fail(PBK_ERR_INVALID, "no output: out, sk and mask are NULL");
  if (nsamp > 0 && !in) return fail(PBK_ERR_INVALID, "in is NULL");
  const int esize = in_dtype == PBK_C64 ? 8 : in_dtype == PBK_I8X2 ? 2 : 4;
  if (on_device && ((((uintptr_t)in | (uintptr_t)out) & (esize - 1)) || ((uintptr_t)sk & 3)))
    return fail(PBK_ERR_INVALID, "device arrays must be aligned to their element size");
  if (nchan > INT_MAX || npol > INT_MAX || nchan * npol > INT_MAX)
    return fail(PBK_ERR_UNSUPPORTED, "nchan * npol must be at most INT32_MAX");
  const long long W = nchan * npol;
  if (nsamp > LLONG_MAX / 8 / W) return fail(PBK_ERR_UNSUPPORTED, "input too large");
  const long long nblk = nsamp / m;
  const size_t rowb = (size_t)W * esize, ib = (size_t)nsamp * rowb;
  const bool copy = out && out != in;
  if (nblk == 0) {   // nothing to estimate: a separate output is a copy of the input
    if (copy && ib) {
      if (!on_device) {
        std::memcpy(out, in, ib);
        return PBK_OK;
      }
      CUDA_TRY(cudaSetDevice(device));
      CUDA_TRY(cudaMemcpyAsync(out, in, ib, cudaMemcpyDeviceToDevice,
                               reinterpret_cast<cudaStream_t>(stream)));
    }
    return PBK_OK;
  }
  // the estimate grid: (block, split, column group).  The lanes, the splits and so the order of
  // every sum follow from the shape alone; arrays aligned to vw elements only take wider loads.
  const int vw = pk::vector_width(esize);
  const long long vn = W % vw == 0 ? vw : 1;
  const int CW = pk::columns_per_cta(W / vn);
  const long long tpc = pk::kThreads / CW, ngn = (W / vn + CW - 1) / CW;
  const long long want = (pk::kTargetCtas + nblk * ngn - 1) / (nblk * ngn);
  const long long most = std::max<long long>(1, m / (tpc * pk::kMinRowsPerLane));
  long long nsplit = std::max<long long>(1, std::min(want, most));
  const long long chunk = (m + nsplit - 1) / nsplit;
  nsplit = (m + chunk - 1) / chunk;
  const long long ncells = nblk * nchan, fgrid = (ncells + pk::kThreads - 1) / pk::kThreads;
  if (nblk * nsplit * ((W + CW - 1) / CW) > INT_MAX || fgrid > INT_MAX)
    return fail(PBK_ERR_UNSUPPORTED, "too many blocks for one launch");

  CUDA_TRY(cudaSetDevice(device));
  cudaStream_t st = on_device ? reinterpret_cast<cudaStream_t>(stream) : cudaStreamPerThread;
  const size_t skb = (size_t)ncells * npol * 4, mb = (size_t)ncells;
  DevBuf di, dsk, dm;
  const void* x = in;
  void* d_sk = sk;
  void* d_mask = mask;
  void* zap = out;          // the array whose flagged cells are zeroed
  void* cp = copy ? out : nullptr;
  if (!on_device) {
    // host route: zero in place in a device copy of the input, then copy the whole array out
    CUDA_TRY(cudaMalloc(&di.p, ib));
    CUDA_TRY(host_to_device(di.p, in, ib, st));
    if (sk) CUDA_TRY(cudaMalloc(&dsk.p, skb));
    if (mask) CUDA_TRY(cudaMalloc(&dm.p, mb));
    x = di.p, d_sk = dsk.p, d_mask = dm.p;
    zap = out ? di.p : nullptr;
    cp = nullptr;
  } else if (copy && (size_t)nsamp > (size_t)nblk * m) {   // the tail rows are never estimated
    const size_t off = (size_t)nblk * m * rowb;
    CUDA_TRY(cudaMemcpyAsync(static_cast<char*>(out) + off, static_cast<const char*>(in) + off,
                             ib - off, cudaMemcpyDeviceToDevice, st));
  }
  const bool vec = vn > 1 && (((uintptr_t)x | (uintptr_t)zap | (uintptr_t)cp) % (vw * esize)) == 0;
  const long long ngroups = vec ? ngn : (W + CW - 1) / CW;
  const unsigned pgrid = (unsigned)(nblk * nsplit * ngroups);
  // the partial sums and the flags live in a stream-ordered allocation
  const size_t partb = (size_t)nblk * nsplit * W * 16;
  void* part = nullptr;
  CUDA_TRY(cudaMallocAsync(&part, partb + (size_t)ncells, st));
  unsigned char* flags = static_cast<unsigned char*>(part) + partb;
  pk::PartArgs pa{};
  pa.in = x, pa.out = cp, pa.part = part, pa.flags = flags;
  pa.W = W, pa.m = m, pa.chunk = chunk, pa.nchan = nchan, pa.npol = npol;
  pa.nsplit = (int)nsplit, pa.ngroups = (int)ngroups;
  pk::FinArgs fa{};
  fa.part = part;
  fa.sk = reinterpret_cast<float*>(d_sk);
  fa.mask = reinterpret_cast<unsigned char*>(d_mask);
  fa.flags = flags;
  fa.ncells = ncells, fa.nchan = nchan, fa.npol = npol, fa.W = W;
  fa.nsplit = (int)nsplit;
  fa.mf = (double)m;
  fa.f = ((double)m * nd + 1.0) / ((double)m - 1.0);
  fa.lo = lo, fa.hi = hi;
  cudaError_t e = pk::launch_pass(esize, false, vec, CW, pa, pgrid, st);
  if (e == cudaSuccess) e = pk::launch_finalize(esize, fa, (unsigned)fgrid, st);
  if (e == cudaSuccess && zap) {
    pa.out = zap;
    e = pk::launch_pass(esize, true, vec, CW, pa, pgrid, st);
  }
  cudaError_t ef = cudaFreeAsync(part, st);
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "spectral kurtosis launch: %s", cudaGetErrorString(e));
  CUDA_TRY(ef);
  if (!on_device) {
    if (sk) CUDA_TRY(device_to_host(sk, d_sk, skb, st));
    if (mask) CUDA_TRY(device_to_host(mask, d_mask, mb, st));
    if (out) CUDA_TRY(device_to_host(out, di.p, ib, st));
  }
  return PBK_OK;
}

extern "C" int pbk_phase_predict(const double* dt_s, int64_t n, double dt0_s,
                                 double sample_rate_hz, int64_t n0, const double* coeffs,
                                 int32_t ncoef, int64_t rphase, void* phase_int, void* phase_frac,
                                 int32_t on_device, int32_t device, void* stream) {
  if (!coeffs || !phase_int || !phase_frac) return fail(PBK_ERR_INVALID, "NULL pointer");
  if (n <= 0) return fail(PBK_ERR_INVALID, "n must be positive");
  if (ncoef < 1 || ncoef > kFoldMaxCoef)
    return fail(PBK_ERR_INVALID, "ncoef must be in [1, %d]", kFoldMaxCoef);
  if (!dt_s && !(sample_rate_hz > 0))
    return fail(PBK_ERR_INVALID, "sample_rate_hz must be > 0 when times are generated");
  CUDA_TRY(cudaSetDevice(device));
  PredictArgs pa;
  memset(&pa, 0, sizeof(pa));
  for (int i = 0; i < ncoef; ++i) pa.coef[i] = coeffs[i];
  pa.ncoef = ncoef;
  pa.dt0 = dt0_s;
  pa.sample_rate = sample_rate_hz;
  pa.n0 = n0;
  pa.n = n;
  pa.rphase = rphase;
  if (on_device) {
    pa.dt = dt_s;
    pa.ph_int = reinterpret_cast<long long*>(phase_int);
    pa.ph_frac = reinterpret_cast<double*>(phase_frac);
    cudaError_t e = launch_phase_predict(pa, reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "predict launch: %s", cudaGetErrorString(e));
    return PBK_OK;
  }
  DevBuf dd, di, df;
  const size_t nb = (size_t)n * 8;
  cudaStream_t st = cudaStreamPerThread;
  if (dt_s) {
    CUDA_TRY(cudaMalloc(&dd.p, nb));
    CUDA_TRY(cudaMemcpyAsync(dd.p, dt_s, nb, cudaMemcpyHostToDevice, st));
  }
  CUDA_TRY(cudaMalloc(&di.p, nb));
  CUDA_TRY(cudaMalloc(&df.p, nb));
  pa.dt = reinterpret_cast<const double*>(dd.p);
  pa.ph_int = reinterpret_cast<long long*>(di.p);
  pa.ph_frac = reinterpret_cast<double*>(df.p);
  cudaError_t e = launch_phase_predict(pa, st);
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "predict launch: %s", cudaGetErrorString(e));
  CUDA_TRY(cudaMemcpyAsync(phase_int, di.p, nb, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaMemcpyAsync(phase_frac, df.p, nb, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return PBK_OK;
}

// elementwise helper shared by the host-pointer variants below
template <typename F>
static int run_elementwise(const void* in, void* out, size_t in_bytes, size_t out_bytes,
                           int on_device, int device, void* stream, F launch) {
  if (!in || !out) return fail(PBK_ERR_INVALID, "NULL data pointer");
  CUDA_TRY(cudaSetDevice(device));
  if (on_device) {
    cudaError_t e = launch(in, out, reinterpret_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "kernel launch: %s", cudaGetErrorString(e));
    return PBK_OK;
  }
  DevBuf di, dout;
  CUDA_TRY(cudaMalloc(&di.p, in_bytes ? in_bytes : 16));
  CUDA_TRY(cudaMalloc(&dout.p, out_bytes ? out_bytes : 16));
  cudaStream_t st = cudaStreamPerThread;
  CUDA_TRY(host_to_device(di.p, in, in_bytes, st));
  cudaError_t e = launch(di.p, dout.p, st);
  if (e != cudaSuccess) return fail(PBK_ERR_CUDA, "kernel launch: %s", cudaGetErrorString(e));
  CUDA_TRY(device_to_host(out, dout.p, out_bytes, st));
  return PBK_OK;
}

extern "C" int pbk_mix(const void* in, void* out, int64_t nsamp, int64_t ncols,
                       const double* cycles_per_sample, int32_t on_device, int32_t device,
                       void* stream) {
  if (nsamp < 0 || ncols <= 0 || !cycles_per_sample) return fail(PBK_ERR_INVALID, "bad argument");
  CUDA_TRY(cudaSetDevice(device));
  DevBuf df;
  CUDA_TRY(cudaMalloc(&df.p, (size_t)ncols * 8));
  CUDA_TRY(cudaMemcpy(df.p, cycles_per_sample, (size_t)ncols * 8, cudaMemcpyHostToDevice));
  const size_t nb = (size_t)nsamp * ncols * 8;
  int rc = run_elementwise(in, out, nb, nb, on_device, device, stream,
                           [&](const void* i, void* o, cudaStream_t st) {
                             return launch_1d(mix_kernel, nsamp * ncols, st,
                                              reinterpret_cast<const float2*>(i),
                                              reinterpret_cast<float2*>(o), (long long)nsamp,
                                              (long long)ncols,
                                              reinterpret_cast<const double*>(df.p));
                           });
  if (rc == PBK_OK && on_device)
    CUDA_TRY(cudaStreamSynchronize(reinterpret_cast<cudaStream_t>(stream)));  // df is freed here
  return rc;
}

extern "C" int pbk_decimate2(const void* in, void* out, int64_t nsamp, int64_t ncols,
                             int32_t on_device, int32_t device, void* stream) {
  if (nsamp < 0 || ncols <= 0) return fail(PBK_ERR_INVALID, "bad shape");
  const long long rows_out = (nsamp + 1) / 2;
  return run_elementwise(in, out, (size_t)nsamp * ncols * 8, (size_t)rows_out * ncols * 8,
                         on_device, device, stream, [&](const void* i, void* o, cudaStream_t st) {
                           return launch_1d(decimate2_kernel, rows_out * ncols, st,
                                            reinterpret_cast<const float2*>(i),
                                            reinterpret_cast<float2*>(o), rows_out,
                                            (long long)ncols);
                         });
}

extern "C" int pbk_stokes(const void* in, void* out, int64_t npairs, int32_t circular,
                          int32_t on_device, int32_t device, void* stream) {
  if (npairs < 0) return fail(PBK_ERR_INVALID, "bad count");
  return run_elementwise(in, out, (size_t)npairs * 16, (size_t)npairs * 16, on_device, device,
                         stream, [&](const void* i, void* o, cudaStream_t st) {
                           return launch_1d(aligned16(i, o) ? stokes_kernel<true>
                                                            : stokes_kernel<false>,
                                            npairs, st, reinterpret_cast<const float2*>(i),
                                            reinterpret_cast<float*>(o), (long long)npairs,
                                            (int)circular);
                         });
}

extern "C" int pbk_pol_basis(const void* in, void* out, int64_t npairs, int32_t to_circular,
                             int32_t on_device, int32_t device, void* stream) {
  if (npairs < 0) return fail(PBK_ERR_INVALID, "bad count");
  return run_elementwise(in, out, (size_t)npairs * 16, (size_t)npairs * 16, on_device, device,
                         stream, [&](const void* i, void* o, cudaStream_t st) {
                           return launch_1d(aligned16(i, o) ? pol_basis_kernel<true>
                                                            : pol_basis_kernel<false>,
                                            npairs, st, reinterpret_cast<const float2*>(i),
                                            reinterpret_cast<float2*>(o), (long long)npairs,
                                            (int)to_circular);
                         });
}

// chirp H[k, c] (dedispersion.py:19-23) as an explicit (nsamp, nchan) complex64 array
__global__ void __launch_bounds__(256) chirp_kernel(PassArgs p, float2* out, long long nsamp,
                                                    long long nchan) {
  const long long total = nsamp * nchan;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long k = i / nchan, c = i - k * nchan;
    out[i] = chirp_value(p, p.chan_freq[c], k);
  }
}

extern "C" int pbk_chirp(int64_t nsamp, int64_t nchan, double dm, double sample_rate_hz,
                         double ref_freq_hz, const double* chan_freq_hz, void* out,
                         int32_t on_device, int32_t device, void* stream) {
  if (nsamp <= 0 || nchan <= 0 || !chan_freq_hz || !out)
    return fail(PBK_ERR_INVALID, "bad argument");
  if (!(sample_rate_hz > 0)) return fail(PBK_ERR_INVALID, "sample_rate_hz must be > 0");
  CUDA_TRY(cudaSetDevice(device));
  DevBuf df;
  CUDA_TRY(cudaMalloc(&df.p, (size_t)nchan * 8));
  CUDA_TRY(cudaMemcpy(df.p, chan_freq_hz, (size_t)nchan * 8, cudaMemcpyHostToDevice));
  PassArgs a;
  defaults(a);
  a.N = nsamp;
  a.chan_freq = reinterpret_cast<const double*>(df.p);
  a.df = 1.0 / ((double)nsamp * (1.0 / sample_rate_hz));
  if (std::isinf(ref_freq_hz)) { a.fr_sub = 0; a.inv_fr = 0; a.a0 = -1.0; }
  else { a.fr_sub = ref_freq_hz; a.inv_fr = 1.0 / ref_freq_hz; a.a0 = 0; }
  a.D = (1.0 / 2.41e-4) * dm * 1e12;
  a.scale = 1.0f;
  const size_t ob = (size_t)nsamp * nchan * 8;
  int rc = run_elementwise(out /*unused as input*/, out, 0, ob, on_device, device, stream,
                           [&](const void*, void* o, cudaStream_t st) {
                             return launch_1d(chirp_kernel, nsamp * nchan, st, a,
                                              reinterpret_cast<float2*>(o), (long long)nsamp,
                                              (long long)nchan);
                           });
  if (rc == PBK_OK && on_device)
    CUDA_TRY(cudaStreamSynchronize(reinterpret_cast<cudaStream_t>(stream)));  // df is freed here
  return rc;
}

// ------------------------------------------------------------------------------------------
// complex128 (FP64) transforms: pbk_f64.cuh.  Plan-less: two work arrays per call from the
// stream-ordered allocator; complex128 is the accuracy path, not the throughput path.
// ------------------------------------------------------------------------------------------
struct F64Work {   // stream-ordered scratch (+ staging for host pointers), freed on scope exit
  cudaStream_t st;
  std::vector<void*> ptrs;
  explicit F64Work(cudaStream_t s) : st(s) {}
  cudaError_t get(void** p, size_t bytes) {
    cudaError_t e = cudaMallocAsync(p, bytes ? bytes : 16, st);
    if (e == cudaSuccess) ptrs.push_back(*p);
    return e;
  }
  ~F64Work() { for (void* p : ptrs) cudaFreeAsync(p, st); }
};

static int f64_check_len(long long n) {
  if (n > (1ll << 28))
    return fail(PBK_ERR_UNSUPPORTED, "complex128 transform length %lld is too long", n);
  return PBK_OK;
}

extern "C" int pbk_fft_c128(const void* in, void* out, int64_t outer, int64_t n, int64_t inner,
                            int32_t inverse, int32_t on_device, int32_t device, void* stream) {
  if (!in || !out) return fail(PBK_ERR_INVALID, "NULL data pointer");
  if (outer <= 0 || n <= 0 || inner <= 0) return fail(PBK_ERR_INVALID, "shape must be positive");
  int rc = f64_check_len(n);
  if (rc != PBK_OK) return rc;
  CUDA_TRY(cudaSetDevice(device));
  cudaStream_t st = on_device ? reinterpret_cast<cudaStream_t>(stream) : cudaStreamPerThread;
  const size_t bytes = (size_t)outer * n * inner * sizeof(double2);
  F64Work w(st);
  auto alloc = [&](void** p, size_t b) { return w.get(p, b); };
  double2 *res, *din = nullptr;
  const double2* src = reinterpret_cast<const double2*>(in);
  if (!on_device) {
    CUDA_TRY(w.get((void**)&din, bytes));
    CUDA_TRY(host_to_device(din, in, bytes, st));
    src = din;
  }
  CUDA_TRY(f64_fft_any(src, alloc, outer, n, inner, inverse ? +1 : -1, st, &res));
  double2* dst = reinterpret_cast<double2*>(out);
  if (!on_device) CUDA_TRY(w.get((void**)&dst, bytes));
  f64_store_kernel<<<f64_blocks(outer * n * inner), 256, 0, st>>>(
      res, dst, 0, outer * n, inner, inverse ? 1.0 / (double)n : 1.0, 0);
  CUDA_TRY(cudaGetLastError());
  if (!on_device) {
    CUDA_TRY(device_to_host(out, dst, bytes, st));
    CUDA_TRY(cudaStreamSynchronize(st));
  }
  return PBK_OK;
}

extern "C" int pbk_stft_c128(const void* in, void* out, int64_t nseg, int64_t nperseg,
                             int64_t nchan, int64_t npol, int32_t inverse, int32_t on_device,
                             int32_t device, void* stream) {
  if (!in || !out) return fail(PBK_ERR_INVALID, "NULL data pointer");
  if (nseg <= 0 || nperseg <= 0 || nchan <= 0 || npol <= 0)
    return fail(PBK_ERR_INVALID, "shape must be positive");
  int rc = f64_check_len(nperseg);
  if (rc != PBK_OK) return rc;
  CUDA_TRY(cudaSetDevice(device));
  cudaStream_t st = on_device ? reinterpret_cast<cudaStream_t>(stream) : cudaStreamPerThread;
  const long long n = nperseg, I = nchan * npol, total = nseg * n * I;
  const size_t bytes = (size_t)total * sizeof(double2);
  F64Work w(st);
  auto alloc = [&](void** p, size_t b) { return w.get(p, b); };
  double2 *c, *res, *din = nullptr;
  const double2* src = reinterpret_cast<const double2*>(in);
  if (!on_device) {
    CUDA_TRY(w.get((void**)&din, bytes));
    CUDA_TRY(host_to_device(din, in, bytes, st));
    src = din;
  }
  double2* dst = reinterpret_cast<double2*>(out);
  if (!on_device) CUDA_TRY(w.get((void**)&dst, bytes));
  if (!inverse) {   // segments are (n, C P) blocks: transform, then shift / scale / regroup
    CUDA_TRY(f64_fft_any(src, alloc, nseg, n, I, -1, st, &res));
    f64_stft_permute_kernel<<<f64_blocks(total), 256, 0, st>>>(res, dst, nseg, n, nchan, npol, 0,
                                                                1.0 / (double)n);
  } else {          // (x * n) then ifft (misc.py:82-87): ungroup / ifftshift, unscaled inverse
    CUDA_TRY(w.get((void**)&c, bytes));
    f64_stft_permute_kernel<<<f64_blocks(total), 256, 0, st>>>(src, c, nseg, n, nchan, npol, 1, 1.0);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(f64_fft_any(c, alloc, nseg, n, I, +1, st, &res));
    f64_store_kernel<<<f64_blocks(total), 256, 0, st>>>(res, dst, 0, nseg * n, I, 1.0, 0);
  }
  CUDA_TRY(cudaGetLastError());
  if (!on_device) {
    CUDA_TRY(device_to_host(out, dst, bytes, st));
    CUDA_TRY(cudaStreamSynchronize(st));
  }
  return PBK_OK;
}

extern "C" int pbk_dedisp_c128(const void* in, void* out, int64_t nsamp, int64_t nchan,
                               int64_t npol, int32_t out_kind, double dm, double sample_rate_hz,
                               double ref_freq_hz, const double* chan_freq_hz, int64_t crop_start,
                               int64_t crop_stop, const void* chirp, int32_t on_device,
                               int32_t device, void* stream) {
  if (!in || !chan_freq_hz) return fail(PBK_ERR_INVALID, "NULL pointer");
  if (nsamp <= 0 || nchan <= 0 || npol <= 0) return fail(PBK_ERR_INVALID, "shape must be positive");
  if (!(sample_rate_hz > 0)) return fail(PBK_ERR_INVALID, "sample_rate_hz must be > 0");
  if (out_kind < PBK_OUT_C64 || out_kind > PBK_OUT_STOKES_I)
    return fail(PBK_ERR_INVALID, "unknown out_kind %d", out_kind);
  if (out_kind == PBK_OUT_STOKES_I && npol != 2) return fail(PBK_ERR_INVALID, "Stokes I needs npol == 2");
  if (crop_start < 0 || crop_stop > nsamp) return fail(PBK_ERR_INVALID, "crop outside the signal");
  int rc = f64_check_len(nsamp);
  if (rc != PBK_OK) return rc;
  const long long rows = std::max<long long>(0, crop_stop - crop_start);
  if (rows == 0) return PBK_OK;
  if (!out) return fail(PBK_ERR_INVALID, "output pointer is NULL");
  CUDA_TRY(cudaSetDevice(device));
  cudaStream_t st = on_device ? reinterpret_cast<cudaStream_t>(stream) : cudaStreamPerThread;
  const long long N = nsamp, I = nchan * npol;
  const size_t bytes = (size_t)N * I * sizeof(double2);
  const long long E = out_kind == PBK_OUT_STOKES_I ? nchan : I;
  const size_t obytes = (size_t)rows * E * (out_kind == PBK_OUT_C64 ? 16 : 8);
  F64Work w(st);
  auto alloc = [&](void** p, size_t b) { return w.get(p, b); };
  double2 *res, *din = nullptr;
  double* dfreq;
  float2* dchirp = nullptr;
  CUDA_TRY(w.get((void**)&dfreq, (size_t)nchan * 8));
  CUDA_TRY(cudaMemcpyAsync(dfreq, chan_freq_hz, (size_t)nchan * 8, cudaMemcpyHostToDevice, st));
  const double2* src = reinterpret_cast<const double2*>(in);
  if (!on_device) {
    CUDA_TRY(w.get((void**)&din, bytes));
    CUDA_TRY(host_to_device(din, in, bytes, st));
    src = din;
    if (chirp) {
      CUDA_TRY(w.get((void**)&dchirp, (size_t)N * nchan * 8));
      CUDA_TRY(host_to_device(dchirp, chirp, (size_t)N * nchan * 8, st));
    }
  } else {
    dchirp = const_cast<float2*>(reinterpret_cast<const float2*>(chirp));
  }
  CUDA_TRY(f64_fft_any(src, alloc, 1, N, I, -1, st, &res));
  F64Chirp c;
  c.N = N; c.nchan = nchan; c.npol = npol;
  c.df = 1.0 / ((double)N * (1.0 / sample_rate_hz));
  if (std::isinf(ref_freq_hz)) { c.fr_sub = 0; c.inv_fr = 0; c.a0 = -1.0; }
  else { c.fr_sub = ref_freq_hz; c.inv_fr = 1.0 / ref_freq_hz; c.a0 = 0; }
  c.D = (1.0 / 2.41e-4) * dm * 1e12;
  c.chan_freq = dfreq;
  c.chirp_arr = dchirp;
  f64_chirp_kernel<<<f64_blocks(N * I), 256, 0, st>>>(res, c);
  CUDA_TRY(cudaGetLastError());
  double2* spec = res;
  CUDA_TRY(f64_fft_any(spec, alloc, 1, N, I, +1, st, &res));
  void* dst = out;
  if (!on_device) CUDA_TRY(w.get(&dst, obytes));
  f64_store_kernel<<<f64_blocks(rows * E), 256, 0, st>>>(res, dst, crop_start, crop_stop, I,
                                                         1.0 / (double)N, out_kind);
  CUDA_TRY(cudaGetLastError());
  if (!on_device) {
    CUDA_TRY(device_to_host(out, dst, obytes, st));
    CUDA_TRY(cudaStreamSynchronize(st));
  } else {
    // the host array of channel frequencies was copied asynchronously: it must stay valid until
    // the copy has run, so wait for it here (a few KB; the kernels stay queued)
    CUDA_TRY(cudaStreamSynchronize(st));
  }
  return PBK_OK;
}

// power detection of complex128 voltages in FP64 (core.py:766-774 keeps float64 for complex128)
extern "C" int pbk_detect_c128(const void* in, void* out, int64_t nsamp, int64_t nchan,
                               int64_t npol, int32_t out_kind, int32_t on_device, int32_t device,
                               void* stream) {
  if (!in || !out) return fail(PBK_ERR_INVALID, "NULL data pointer");
  if (nsamp <= 0 || nchan <= 0 || npol <= 0) return fail(PBK_ERR_INVALID, "bad shape");
  if (out_kind != PBK_OUT_INTENSITY && out_kind != PBK_OUT_STOKES_I)
    return fail(PBK_ERR_INVALID, "out_kind must be INTENSITY or STOKES_I");
  if (out_kind == PBK_OUT_STOKES_I && npol != 2) return fail(PBK_ERR_INVALID, "Stokes I needs npol == 2");
  CUDA_TRY(cudaSetDevice(device));
  cudaStream_t st = on_device ? reinterpret_cast<cudaStream_t>(stream) : cudaStreamPerThread;
  const long long I = nchan * npol, E = out_kind == PBK_OUT_STOKES_I ? nchan : I;
  const size_t ib = (size_t)nsamp * I * 16, ob = (size_t)nsamp * E * 8;
  F64Work w(st);
  const double2* src = reinterpret_cast<const double2*>(in);
  void* dst = out;
  if (!on_device) {
    double2* din;
    CUDA_TRY(w.get((void**)&din, ib));
    CUDA_TRY(w.get(&dst, ob));
    CUDA_TRY(host_to_device(din, in, ib, st));
    src = din;
  }
  f64_store_kernel<<<f64_blocks(nsamp * E), 256, 0, st>>>(src, dst, 0, nsamp, I, 1.0, out_kind);
  CUDA_TRY(cudaGetLastError());
  if (!on_device) {
    CUDA_TRY(device_to_host(out, dst, ob, st));
    CUDA_TRY(cudaStreamSynchronize(st));
  }
  return PBK_OK;
}

// ------------------------------------------------------------------------------------------
// raw memory helpers
// ------------------------------------------------------------------------------------------
extern "C" int pbk_malloc(void** dptr, size_t bytes, int32_t device) {
  if (!dptr) return fail(PBK_ERR_INVALID, "dptr is NULL");
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(cudaMalloc(dptr, bytes ? bytes : 1));
  return PBK_OK;
}
extern "C" int pbk_free(void* dptr, int32_t device) {
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(cudaFree(dptr));
  return PBK_OK;
}
extern "C" int pbk_memcpy_h2d(void* dst, const void* src, size_t bytes, int32_t device) {
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice));
  return PBK_OK;
}
extern "C" int pbk_memcpy_d2h(void* dst, const void* src, size_t bytes, int32_t device) {
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost));
  return PBK_OK;
}
extern "C" int pbk_memcpy_async(void* dst, const void* src, size_t bytes, int32_t to_device,
                                int32_t device, void* stream) {
  CUDA_TRY(cudaSetDevice(device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // large PAGEABLE sources go through the bounce pipeline, which has read src when it returns; a
  // page-locked source (and any copy under 32 MiB) is one plain cudaMemcpyAsync, so the caller
  // must keep src valid until the stream has reached the copy
  if (to_device)
    CUDA_TRY(host_to_device(dst, src, bytes, st));
  else
    CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st));
  return PBK_OK;
}
extern "C" int pbk_device_sync(int32_t device) {
  CUDA_TRY(cudaSetDevice(device));
  CUDA_TRY(cudaDeviceSynchronize());
  return PBK_OK;
}
