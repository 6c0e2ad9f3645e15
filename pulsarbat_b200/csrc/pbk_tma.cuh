// pbk_tma.cuh -- TMA-staged, software-pipelined variant of the compile-time-shaped pass kernels.
//
// The kernels of pbk_fast.cuh load a tile with synchronous LDG -> register -> shared-memory
// traffic, so a CTA alternates between a load phase (warps parked on the long scoreboard) and a
// compute phase, and only the second resident CTA hides either.  Here one CTA per SM owns a RING of
// tile buffers in shared memory; tiles are brought in by the tensor-memory accelerator
// (cp.async.bulk.tensor: one instruction per 256-row box, completion on an mbarrier) while the
// warps only ever compute:
//
//   * the CTA is NG thread GROUPS of C::NT threads (the unit that owned a CTA in pbk_fast.cuh); a
//     group works on one tile at a time, synchronises with a named barrier, and keeps the same
//     per-tile code (stage functions, level twiddle, chirp, epilogues, TSUM accumulators);
//   * NBUF = NG + NG/2 buffers: NG being computed in place, the rest in flight.  The tiles of the
//     CTA form ONE sequence (round k of group 0, of group 1, ...; groups that have run out of
//     tiles are skipped); the tile of rank k lives in buffer k % NBUF.  The group that finishes
//     rank k issues the TMA load of rank k + NBUF into the buffer it just released -- no "empty"
//     barrier, and a load has a whole tile time to land.  A consumer first waits (a shared-memory
//     word per buffer) until ITS load has been issued, then on the buffer's mbarrier: without the
//     first wait a group that runs more than one use of a buffer ahead would see the barrier's
//     parity of the use before last and walk into a tile another group has not consumed yet;
//   * a tile is a dense box of the 4-D view (lane, inner time offset, tile row, outer block) of
//     the pass input -- the tensor map is encoded by the host per pass (pbk_api.cu: tma_encode).
//
// The tile arrives in natural row order.  Forward / middle passes run their first stage in place
// from shared memory.  An inverse pass reads the rows its first radix-R stage needs (a digit
// reversal) into registers, waits for the group, and writes the stage output back in the
// last-stage order -- one extra barrier instead of a second buffer.
//
// Preconditions (host: setup_tma): wide tiles (I % W == 0), complex64 or pair-planar input, plain
// pass-after-pass schedule.  Tiles of 2^6 .. 2^9 points have rows of >= 128 B (full DRAM bursts, no
// XOR swizzle in shared memory); the 2^10-point tile (64-byte rows) exists for the MID pass only.
#pragma once
#include <cuda.h>
#include <cstdio>

#include "pbk_fast.cuh"

namespace pbk {

// ------------------------------------------------------------------------------------------
// PTX wrappers: mbarrier, bulk tensor copy, proxy fence, named barrier
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok = 0;
  while (!ok) {
    asm volatile(
        "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        " selp.u32 %0, 1, 0, p;\n}\n"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
  }
}
// box (c0.., c1, c2.., c3) of a rank-4 tensor -> dense shared-memory tile; completes on `bar`
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, int c0, int c1,
                                            int c2, int c3, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, "
      "{%2, %3, %4, %5}], [%6];" ::"r"(smem_u32(dst)),
      "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(smem_u32(bar))
      : "memory");
}
// orders this thread's earlier generic-proxy accesses to shared memory before later async-proxy
// (TMA) accesses to the same addresses
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
template <int NT>
struct GroupSync {   // named barrier 1 + group (barrier 0 is __syncthreads)
  int id;
  __device__ __forceinline__ void operator()() const {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(NT) : "memory");
  }
};

template <class C>
struct TmaCfg {
  static constexpr int CTA_THREADS = 512;
  static constexpr int NG = CTA_THREADS / C::NT;          // thread groups per CTA
  static constexpr int NBUF = NG + NG / 2;                // tile buffers in the ring
  static constexpr int BOX_ROWS = C::L < 256 ? C::L : 256;
  static constexpr int BOXES = C::L / BOX_ROWS;           // TMA instructions per tile
  static constexpr size_t TILE_BYTES = C::TILE_BYTES;
  static constexpr size_t OFF_TW = (size_t)NBUF * TILE_BYTES;
  static constexpr size_t OFF_G = OFF_TW + (size_t)C::TW_PAD * sizeof(float2);
  static constexpr size_t OFF_INFO = OFF_G + (size_t)NG * C::RL * sizeof(float4);
  static constexpr size_t OFF_BAR = OFF_INFO + (size_t)NG * 64;
  static constexpr size_t OFF_ISSUED = OFF_BAR + (size_t)NBUF * 8;   // rank last issued per buffer
  static constexpr size_t OFF_SEQ = OFF_ISSUED + (size_t)NBUF * 8;     // t0[NG], cnt[NG] (issuer's copy)
  static constexpr size_t SMEM_BYTES = OFF_SEQ + (size_t)NG * 16 + 64;
  // rows of 64 B (PW = 4): the tile arrives row-major and the first stage writes the swizzled
  // layout the later stages expect (fwd_first_smem); only the MID kernel is instantiated there
  static_assert(C::PW >= 4, "TMA tiles are row-major boxes of at least 64-byte rows");
  static_assert(C::NT * NG == CTA_THREADS && NG >= 2, "thread groups tile the CTA");
  static_assert(sizeof(TileInfo) <= 64, "tile record slot");
  static_assert(SMEM_BYTES <= 227 * 1024, "ring of tile buffers exceeds shared memory");
};

// first forward stage on a tile that is already in shared memory in natural row order: in place
// (a DIF butterfly reads and writes the same R rows); complex64 input is de-interleaved here.
// Tiles with rows shorter than 128 B keep the XOR swizzle of pbk_fast.cuh (phys_pt) from the
// first stage's OUTPUT on: the stage then writes row b ^ 1 for some b, i.e. the rows its
// neighbour four lanes away has read -- same warp, same iteration, so a __syncwarp between the
// loads and the stores is all the ordering that needs.
template <class C, int LOADK, bool SIGNINV>
__device__ __forceinline__ void fwd_first_smem(float4* tile, const float2* tws, int tid) {
  constexpr int R = C::radix(0), S = C::stride(0);
  constexpr int TASKS = S * C::PW;
  constexpr int ITERS = (TASKS + C::NT - 1) / C::NT;
  static_assert(C::PPB == 1 || (S % (C::RL * C::PPB) == 0 && C::PW * C::PPB <= 32 &&
                                TASKS % C::NT == 0),
                "swizzled first stage: partner rows are exchanged inside a warp");
  const int pr = tid & (C::PW - 1);
#pragma unroll
  for (int it = 0; it < ITERS; ++it) {
    const int tau = tid + it * C::NT;
    if (TASKS % C::NT != 0 && tau >= TASKS) break;
    const int b = tau >> C::LOG2PW;
    c2 v[R];
#pragma unroll
    for (int i = 0; i < R; ++i) {
      const float4 t = tile[((b + i * S) << C::LOG2PW) + pr];
      if (LOADK == LK_PLANAR) {
        v[i].re = make_float2(t.x, t.y);
        v[i].im = make_float2(t.z, t.w);
      } else {   // LK_C64: {re0, im0, re1, im1}
        v[i].re = make_float2(t.x, t.z);
        v[i].im = make_float2(t.y, t.w);
      }
    }
    if constexpr (C::PPB > 1) __syncwarp();
    Butterfly<R, SIGNINV>::run(v);
    stage_twiddle<R, S, SIGNINV>(v, tws + C::tw_off(0), b);
#pragma unroll
    for (int i = 0; i < R; ++i) sts_c2(tile, (phys_pt<C, S>(b, i) << C::LOG2PW) + pr, v[i]);
  }
}

// ------------------------------------------------------------------------------------------
// kernel
// ------------------------------------------------------------------------------------------
template <int MODE, class C, int LOADK, int EPI, bool TWOCH = false, bool TSUM = false>
__global__ void __launch_bounds__(TmaCfg<C>::CTA_THREADS, 1)
tma_pass_kernel(const __grid_constant__ PassArgs p, const __grid_constant__ CUtensorMap tmap,
                const float2* __restrict__ tables, long long ntiles) {
  using T_ = TmaCfg<C>;
  constexpr int NG = T_::NG, NBUF = T_::NBUF, NT = C::NT;
  static_assert(C::NS >= 2, "at least two stages");
  static_assert(LOADK == LK_PLANAR || LOADK == LK_C64, "TMA tiles hold complex64 pairs");
  static_assert(!TSUM || (MODE == MODE_INV && (EPI == EPI_INTENSITY || EPI == EPI_STOKES_I)),
                "TSUM is a final INV pass");
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  float4* ring = reinterpret_cast<float4*>(smem_raw);
  float2* tws = reinterpret_cast<float2*>(smem_raw + T_::OFF_TW);
  const int g = threadIdx.x / NT;          // warp-uniform: NT is a multiple of 32
  const int tid = threadIdx.x - g * NT;
  const int pr = tid & (C::PW - 1);
  float4* G4 = reinterpret_cast<float4*>(smem_raw + T_::OFF_G) + g * C::RL;
  TileInfo* sinfo = reinterpret_cast<TileInfo*>(smem_raw + T_::OFF_INFO + (size_t)g * 64);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + T_::OFF_BAR);
  volatile long long* issued = reinterpret_cast<volatile long long*>(smem_raw + T_::OFF_ISSUED);
  const GroupSync<NT> gsync{1 + g};

  constexpr int in_bits = 64;
  constexpr int out_eb = (EPI == EPI_INTENSITY || EPI == EPI_STOKES_I) ? 4 : 8;
  const unsigned rb_out = (unsigned)(p.mout.a_row * out_eb);

  // ---- tile sequences of the NG groups (a group is a "virtual CTA" of the plain kernels) ------
  const long long vgrid = (long long)gridDim.x * NG;
  const int ncg = TSUM ? p.I / C::W : 1;
  const int tq = TSUM ? p.tsum_q : 1;
  const unsigned ts_off = TSUM ? (unsigned)(p.crop_start & ((1ll << p.tsum_log2) - 1)) : 0u;
  auto ts_snap = [&](long long u) -> long long {
    if (!TSUM || ts_off == 0) return u;
    const long long nr = u & ((1ll << p.log2nmul) - 1);
    const long long tail = (1ll << p.log2nmul) - ((1ll << p.tsum_log2) - ts_off);
    if (nr > 0 && nr < ts_off) return u - nr + ts_off;
    if (nr > tail) return u - nr + tail;
    return u;
  };
  // Runs of the NG groups (start, count).  Every thread needs its own group's run, rank_of all
  // counts once per tile, and the issuing thread walks all runs with a run-time group index.
  // Two ways to hold them, chosen per kind of pass on measurements (cfg2 / 2^24 x 64 lanes):
  //   RUNS_LOCAL  per-thread arrays; the run-time index puts them in local memory, and the loop
  //               bound is a local load per tile.  The HBM-bound forward / inverse passes are
  //               4-6 % faster this way (2^8: 1.43 vs 1.49 ms): anything that lets the loads run
  //               further ahead of the stores costs them DRAM efficiency.
  //   otherwise   own run in registers, all runs in shared memory for rank_of and the issuer.
  //               The passes that are not HBM-bound gain: 2^10-point MID 4.85 -> 4.25 ms, fused
  //               time sum 1.09 -> 1.04 ms.
  constexpr bool RUNS_LOCAL = MODE != MODE_MID && !TSUM;
  long long l_t0[RUNS_LOCAL ? NG : 1];
  int l_cnt[RUNS_LOCAL ? NG : 1];
  long long my_t0 = 0;
  int my_cnt = 0;
  long long* s_t0 = reinterpret_cast<long long*>(smem_raw + T_::OFF_SEQ);
  int* s_cnt = reinterpret_cast<int*>(s_t0 + NG);
#pragma unroll
  for (int gg = 0; gg < NG; ++gg) {
    const long long vb = (long long)blockIdx.x * NG + gg;
    long long start;
    int c;
    if (TSUM) {
      const long long total = ntiles / tq, r = vb / tq, nr = vgrid / tq;
      start = ts_snap(total * r / nr);
      c = (int)(ts_snap(total * (r + 1) / nr) - start);
    } else {
      start = vb;
      c = vb < ntiles ? (int)((ntiles - vb + vgrid - 1) / vgrid) : 0;
    }
    if constexpr (RUNS_LOCAL) {
      l_t0[gg] = start;
      l_cnt[gg] = c;
    } else {
      if (gg == g) { my_t0 = start; my_cnt = c; }
      if (threadIdx.x == 0) { s_t0[gg] = start; s_cnt[gg] = c; }
    }
  }
  auto run_cnt = [&](int gg) -> int { return RUNS_LOCAL ? l_cnt[RUNS_LOCAL ? gg : 0] : s_cnt[gg]; };
  auto run_t0 = [&](int gg) -> long long { return RUNS_LOCAL ? l_t0[RUNS_LOCAL ? gg : 0] : s_t0[gg]; };
  auto own_cnt = [&]() -> int { return RUNS_LOCAL ? l_cnt[RUNS_LOCAL ? g : 0] : my_cnt; };
  auto own_t0 = [&]() -> long long { return RUNS_LOCAL ? l_t0[RUNS_LOCAL ? g : 0] : my_t0; };
  // rank of tile j of group gg in the CTA's sequence (rounds of the groups, exhausted ones skipped)
  auto rank_of = [&](int gg, long long j) -> long long {
    long long k = 0;
#pragma unroll
    for (int h = 0; h < NG; ++h) {
      const long long upto = j + (h < gg ? 1 : 0), ch = run_cnt(h);
      k += ch < upto ? ch : upto;
    }
    return k;
  };
  // j-th tile of group gg whose run starts at start
  auto tile_of = [&](int gg, long long start, long long j) -> long long {
    if (!TSUM) return start + j * vgrid;
    const long long i = start + j;
    const long long cb = i >> p.log2nmul, nr = i & ((1ll << p.log2nmul) - 1);
    const int cgq = (int)(((long long)blockIdx.x * NG + gg) % tq);
    return nr * ncg + cb * tq + cgq;
  };
  // one thread: arm the buffer's barrier, start the tile's box(es), publish the rank
  auto issue = [&](long long tile, long long rank) {
    const int buf = (int)(rank % NBUF);
    const long long q0 = tile * C::W;
    const long long o = q0 / p.RI;
    const long long r0 = q0 - o * p.RI;
    const long long nrest = r0 / p.I;
    const int col0 = (int)(r0 - nrest * p.I);
    mbar_expect_tx(&full[buf], (uint32_t)T_::TILE_BYTES);
#pragma unroll
    for (int bx = 0; bx < T_::BOXES; ++bx)
      tma_load_4d(reinterpret_cast<unsigned char*>(ring) + (size_t)buf * T_::TILE_BYTES +
                      (size_t)bx * T_::BOX_ROWS * C::PW * sizeof(float4),
                  &tmap, 2 * col0, (int)nrest, bx * T_::BOX_ROWS, (int)o, &full[buf]);
    __threadfence_block();
    issued[buf] = rank;
  };
  // one thread: issue the tile that comes `ahead` places after tile j of group gg, if there is one
  auto issue_ahead = [&](int gg, long long j, long long rank, int ahead) {
    int h = gg;
    long long jj = j;
    for (int found = 0;;) {
      if (++h == NG) { h = 0; ++jj; }
      bool any = false;                 // is any group still alive in this or a later round?
#pragma unroll
      for (int q = 0; q < NG; ++q) any = any || jj < run_cnt(q);
      if (!any) return;
      if (jj < run_cnt(h) && ++found == ahead) break;
    }
    issue(tile_of(h, run_t0(h), jj), rank + ahead);
  };

  pdl_trigger();
  for (int i = threadIdx.x; i < C::TW_TOTAL; i += T_::CTA_THREADS) tws[i] = tables[i];
  if (threadIdx.x == 0) {
    for (int b = 0; b < NBUF; ++b) {
      mbar_init(&full[b], 1);
      issued[b] = -1;
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (tid == 0 && own_cnt() > 0)
    fast_tile_info<C, EPI>(p, tile_of(g, own_t0(), 0), *sinfo, in_bits, out_eb);
  __syncthreads();
  pdl_wait();   // the first TMA loads read the previous pass's output
  if (threadIdx.x == 0) {     // ranks 0 .. NBUF-1: "ahead of the tile before the first"
    for (int a = 1; a <= NBUF; ++a) issue_ahead(NG - 1, -1, -1, a);
  }

  // per-thread part of the output address (wide tiles: the tile sits inside one row of lanes)
  const int colt = 2 * pr;
  const long long off_out =
      ((long long)(colt / p.P) * p.mout.a_c + (colt % p.P) * p.mout.a_p) * out_eb;
  const int chant = colt / p.P;

  constexpr int RL = C::RL;
  constexpr int LTASKS = (C::L / RL) * C::PW;
  constexpr int LITERS = (LTASKS + NT - 1) / NT;
  static_assert(MODE != MODE_INV || LTASKS % NT == 0, "whole first-stage tasks per thread");

  TsumAcc<C, TSUM ? EPI : EPI_STOKES_I> tacc;
  char* ts_colbase = nullptr;
  unsigned ts_nrest = 0;
  const long long ts_rowbytes = p.mout.a_n * out_eb;
  if (TSUM) tacc.clear();

  for (long long j = 0; j < own_cnt(); ++j) {
    const long long rank = rank_of(g, j);
    const int buf = (int)(rank % NBUF);
    {
      float4* tile = ring + (size_t)buf * (C::L * C::PW);
      FastTile T;
      unsigned nrest0;
      {
        const TileInfo ti = *sinfo;
        T.gin = nullptr;
        T.gout = reinterpret_cast<char*>(p.out) + ti.bo + off_out;
        if constexpr (TSUM) {
          char* colbase = T.gout - ((long long)ti.nrest - p.crop_start) * ts_rowbytes;
          if (ts_colbase != nullptr &&
              (colbase != ts_colbase || ((ti.nrest - ts_off) & ((1u << p.tsum_log2) - 1)) == 0))
            tsum_flush<C, EPI>(p, tacc, ts_colbase, ts_nrest, tid, ts_rowbytes);
          ts_colbase = colbase;
          ts_nrest = ti.nrest;
        }
        nrest0 = ti.nrest;
        T.nrest = ti.nrest;
        T.klow = ti.klow;
        T.chan = ti.chan0 + chant;
        T.row_lo = ti.row_lo;
        T.row_cnt = ti.row_cnt;
          }
      if (MODE != MODE_MID && tid < RL) {
        const float2 gv = unit_root((unsigned long long)nrest0 * (unsigned)(C::KS * tid), p.log2M);
        G4[tid] = make_float4(gv.x, gv.y, gv.y, gv.x);
      }
#define PBK_TMA_NEXT_INFO()                                                      \
  if (tid == 0 && j + 1 < own_cnt())                                             \
    fast_tile_info<C, EPI>(p, tile_of(g, own_t0(), j + 1), *sinfo, in_bits, out_eb)

      while (issued[buf] < rank) {}                               // our load has been issued ...
      mbar_wait(&full[buf], (uint32_t)((rank / NBUF) & 1));       // ... and has landed

      if (MODE == MODE_FWD) {
        fwd_first_smem<C, LOADK, false>(tile, tws, tid);
        gsync();
        PBK_TMA_NEXT_INFO();
        mid_stages<C, false, false>(tile, tws, tid, gsync);
#pragma unroll
        for (int it = 0; it < LITERS; ++it) {
          const int tau = tid + it * NT;
          if (LTASKS % NT != 0 && tau >= LTASKS) break;
          const int b = tau >> C::LOG2PW;
          c2 v[RL];
#pragma unroll
          for (int i = 0; i < RL; ++i) v[i] = lds_c2(tile, last_idx<C>(b, i, pr));
          Butterfly<RL, false>::run(v);
          const int klo = klo_of<C>(b);
          level_twiddle<RL, false>(p, v, T.nrest, (unsigned)klo, G4);
#pragma unroll
          for (int i = 0; i < RL; ++i) fast_store_c64(T, (unsigned)(klo + i * C::KS), rb_out, v[i]);
        }
      } else if (MODE == MODE_MID) {
        fwd_first_smem<C, LOADK, false>(tile, tws, tid);
        gsync();
        PBK_TMA_NEXT_INFO();
        mid_stages<C, false, false>(tile, tws, tid, gsync);
#pragma unroll
        for (int it = 0; it < LITERS; ++it) {
          const int tau = tid + it * NT;
          if (LTASKS % NT != 0 && tau >= LTASKS) break;
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
        gsync();
        mid_stages<C, true, false>(tile, tws, tid, gsync);
        inv_last<C, EPI>(T, tile, tws, tid, rb_out);
      } else {   // MODE_INV: natural-order rows -> registers, barrier, first DIT stage in place
        c2 v[LITERS][RL];
#pragma unroll
        for (int it = 0; it < LITERS; ++it) {
          const int b = (tid + it * NT) >> C::LOG2PW;
          const int klo = klo_of<C>(b);
#pragma unroll
          for (int i = 0; i < RL; ++i) v[it][i] = lds_c2(tile, ((klo + i * C::KS) << C::LOG2PW) + pr);
        }
        gsync();   // every thread holds its rows (and G is written): the tile can be overwritten
        PBK_TMA_NEXT_INFO();
#pragma unroll
        for (int it = 0; it < LITERS; ++it) {
          const int b = (tid + it * NT) >> C::LOG2PW;
          level_twiddle<RL, true>(p, v[it], T.nrest, (unsigned)klo_of<C>(b), G4);
          Butterfly<RL, true>::run(v[it]);
#pragma unroll
          for (int i = 0; i < RL; ++i) sts_c2(tile, last_idx<C>(b, i, pr), v[it][i]);
        }
        gsync();
        mid_stages<C, true, false>(tile, tws, tid, gsync);
        if constexpr (TSUM) inv_last_sum<C, EPI>(T, tile, tws, tid, tacc);
        else inv_last<C, EPI>(T, tile, tws, tid, rb_out);
      }
#undef PBK_TMA_NEXT_INFO
    }
    // the buffer is released: generic-proxy accesses of this group are ordered before the TMA
    // write that refills it, then one thread starts the load of rank + NBUF (same buffer)
    fence_proxy_async();
    gsync();
    if (tid == 0) issue_ahead(g, j, rank, NBUF);
  }
  if constexpr (TSUM) {
    if (ts_colbase != nullptr) tsum_flush<C, EPI>(p, tacc, ts_colbase, ts_nrest, tid, ts_rowbytes);
  }
}

}  // namespace pbk
