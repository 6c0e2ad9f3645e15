// pbk_tsumw.cuh -- the time-summing last pass (INV 2^8 + detection + time sum, pbk_fast.cuh TSUM)
// with WARP-PRIVATE columns: no thread-group barrier anywhere in the tile loop.
//
// In the group kernels (pbk_fast.cuh, pbk_tma.cuh) thread t of a 256-thread group owns lane pair
// t & 15 and stage task t >> 4, so the rows a second-stage task reads were written by sixteen
// threads in eight different warps, and every stage ends in a barrier of the whole group.  With
// the loads hidden by TMA that barrier is where the pass waits (ncu: 2.4 of 4 warps per scheduler
// parked on it, issue slots 46 % busy).  Here a warp owns TWO lane-pair columns of the tile, all
// 256 rows of them: lane = 16 * (column & 1) + task.  Both radix-16 stages of a column then run
// inside one warp and exchange through shared memory under __syncwarp alone; the eight warps of a
// group only meet at the buffer hand-off, which is a counter (the warp that finishes a tile last
// starts the TMA load that refills its buffer) -- nobody waits there either.
//
// Shared-memory layout of a tile: rows of 256 B = 16 columns of 16 B, written by ONE TMA box of a
// rank-5 view of the pass input whose lane axis is split into 128-byte chunks (box = 32 floats x 2
// chunks x 1 x 256 rows x 1), so that the box can carry CU_TENSOR_MAP_SWIZZLE_128B (which spans
// at most 128 B) while a tile row stays ONE contiguous 256-byte run in global memory -- two
// separate 128-byte boxes doubled the number of row chunks and ran into the ~48 G chunks/s limit
// of strided rows (DESIGN.md 5.1), 1.13 ms.  The swizzle is address-based: the 16-byte slot of
// column c in row r is c ^ (((2 r + (c >> 3)) & 7)) within its 128-byte half, i.e. it varies with
// r & 3 only.  A quarter-warp is therefore 4 consecutive tasks x the warp's 2 columns
// (lane = 8 (task >> 2) + 4 (column & 1) + (task & 3)); it reads / writes rows whose r & 3 differ:
//   * first stage input   rows b + 16 i               (task b, register i)
//   * exchange            rows 16 b + ((i + b) & 15)  (the rotation by b makes r & 3 distinct)
//   * second stage input  the same slots, seen as 16 i + ((b + i) & 15) for task b, register i
// so every LDS.128 / STS.128 is conflict-free.
//
// The tile sequence of a CTA, the ring of buffers, the "issued rank" word and the run bookkeeping of
// the time sum are those of tma_pass_kernel<.., TSUM = true>; the tile record (addresses, inner
// offset, crop rows) is computed by the thread that issues the load and travels with the buffer.
// Read-only passes only: the columns of a warp are 32 bytes wide, which would not do for stores.
//
// MEASURED (B200, cfg2's last pass, profiles/r02_tsum_warp_private.log): bit-identical output, the
// barrier stall is gone (2.4 -> 0.002 warps per issue) -- and the pass is SLOWER, 1.13-1.18 ms
// against 0.95-0.97 ms for the thread-group kernels.  The warps now wait for DATA instead
// (16 % of the warp-state samples sit in the mbarrier wait or behind the "issued" poll): a buffer
// is refilled only when the last of eight free-running warps has left it, and a ring of three
// 64 KiB buffers for two groups has one tile of slack, which lock-stepped groups use better than
// drifting warps.  More buffers do not fit (3 x 64 KiB + tables = 201 KiB).  Opt-in: PBK_TSUMW=1.
#pragma once
#include "pbk_tma.cuh"

namespace pbk {

template <class C>
struct TsumwCfg {
  static constexpr int CTA_THREADS = 512;
  static constexpr int NG = 2;                 // groups (tile sequences) per CTA
  static constexpr int WPG = 8;                // warps per group: 2 of the 16 columns each
  static constexpr int NBUF = 3;
  static constexpr size_t TILE_BYTES = (size_t)C::L * 16 * sizeof(float4);   // 256 rows x 256 B
  static constexpr size_t OFF_TW = (size_t)NBUF * TILE_BYTES;
  static constexpr size_t OFF_G = OFF_TW + (size_t)C::TW_PAD * sizeof(float2);
  static constexpr size_t OFF_INFO = OFF_G + (size_t)(CTA_THREADS / 32) * 16 * sizeof(float4);
  static constexpr size_t OFF_BAR = OFF_INFO + (size_t)NBUF * 64;
  static constexpr size_t OFF_ISSUED = OFF_BAR + (size_t)NBUF * 8;
  static constexpr size_t OFF_DONE = OFF_ISSUED + (size_t)NBUF * 8;
  static constexpr size_t OFF_SEQ = OFF_DONE + (size_t)NBUF * 8;
  static constexpr size_t SMEM_BYTES = OFF_SEQ + (size_t)NG * 16 + 64;
  static_assert(C::NS == 2 && C::radix(0) == 16 && C::radix(1) == 16 && C::PW == 16,
                "warp-private columns: 2^8-point tiles of 16 x 16, 16 lane pairs wide");
  static_assert(sizeof(TileInfo) <= 64, "tile record slot");
  static_assert(SMEM_BYTES <= 227 * 1024, "ring of tile buffers exceeds shared memory");
};

template <class C, int EPI>
__global__ void __launch_bounds__(TsumwCfg<C>::CTA_THREADS, 1)
tsum_warp_kernel(const __grid_constant__ PassArgs p, const __grid_constant__ CUtensorMap tmap,
                 const float2* __restrict__ tables, long long ntiles) {
  using T_ = TsumwCfg<C>;
  constexpr int NG = T_::NG, NBUF = T_::NBUF, WPG = T_::WPG;
  static_assert(EPI == EPI_INTENSITY || EPI == EPI_STOKES_I, "a detected, time-summed output");
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  float2* tws = reinterpret_cast<float2*>(smem_raw + T_::OFF_TW);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = warp / WPG, w = warp % WPG;
  const int b = ((lane >> 3) << 2) | (lane & 3);   // stage task of this lane
  const int col = 2 * w + ((lane >> 2) & 1);       // lane pair (column of the tile) of this lane
  const int half = col >> 3, chunk = col & 7;
  float4* G4 = reinterpret_cast<float4*>(smem_raw + T_::OFF_G) + warp * 16;
  TileInfo* info_ring = reinterpret_cast<TileInfo*>(smem_raw + T_::OFF_INFO);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + T_::OFF_BAR);
  volatile long long* issued = reinterpret_cast<volatile long long*>(smem_raw + T_::OFF_ISSUED);
  int* done = reinterpret_cast<int*>(smem_raw + T_::OFF_DONE);
  long long* s_t0 = reinterpret_cast<long long*>(smem_raw + T_::OFF_SEQ);
  int* s_cnt = reinterpret_cast<int*>(s_t0 + NG);

  constexpr int out_eb = 4;
  // ---- tile sequences of the groups: as in tma_pass_kernel<.., TSUM> ---------------------------
  const long long vgrid = (long long)gridDim.x * NG;
  const int ncg = p.I / C::W;
  const int tq = p.tsum_q;
  const unsigned ts_off = (unsigned)(p.crop_start & ((1ll << p.tsum_log2) - 1));
  auto ts_snap = [&](long long u) -> long long {
    if (ts_off == 0) return u;
    const long long nr = u & ((1ll << p.log2nmul) - 1);
    const long long tail = (1ll << p.log2nmul) - ((1ll << p.tsum_log2) - ts_off);
    if (nr > 0 && nr < ts_off) return u - nr + ts_off;
    if (nr > tail) return u - nr + tail;
    return u;
  };
  long long my_t0 = 0;
  int my_cnt = 0;
#pragma unroll
  for (int gg = 0; gg < NG; ++gg) {
    const long long vb = (long long)blockIdx.x * NG + gg;
    const long long total = ntiles / tq, r = vb / tq, nr = vgrid / tq;
    const long long start = ts_snap(total * r / nr);
    const int c = (int)(ts_snap(total * (r + 1) / nr) - start);
    if (gg == g) { my_t0 = start; my_cnt = c; }
    if (threadIdx.x == 0) { s_t0[gg] = start; s_cnt[gg] = c; }
  }
  auto rank_of = [&](int gg, long long j) -> long long {
    long long k = 0;
#pragma unroll
    for (int h = 0; h < NG; ++h) {
      const long long upto = j + (h < gg ? 1 : 0), ch = s_cnt[h];
      k += ch < upto ? ch : upto;
    }
    return k;
  };
  auto tile_of = [&](int gg, long long start, long long j) -> long long {
    const long long i = start + j;
    const long long cb = i >> p.log2nmul, nr = i & ((1ll << p.log2nmul) - 1);
    const int cgq = (int)(((long long)blockIdx.x * NG + gg) % tq);
    return nr * ncg + cb * tq + cgq;
  };
  // one thread: tile record into the buffer's slot, arm the barrier, start the two half-tile
  // boxes, publish the rank
  auto issue = [&](long long tile, long long rank) {
    const int buf = (int)(rank % NBUF);
    fast_tile_info<C, EPI>(p, tile, info_ring[buf], 64, out_eb);
    const long long q0 = tile * C::W;
    const long long o = q0 / p.RI;
    const long long r0 = q0 - o * p.RI;
    const long long nrest = r0 / p.I;
    const int col0 = (int)(r0 - nrest * p.I);
    mbar_expect_tx(&full[buf], (uint32_t)T_::TILE_BYTES);
    tma_load_5d(smem_raw + (size_t)buf * T_::TILE_BYTES, &tmap, 0, col0 / 16, (int)nrest, 0, (int)o,
                &full[buf]);
    __threadfence_block();
    issued[buf] = rank;
  };
  auto issue_ahead = [&](int gg, long long j, long long rank, int ahead) {
    int h = gg;
    long long jj = j;
    for (int found = 0;;) {
      if (++h == NG) { h = 0; ++jj; }
      bool any = false;
#pragma unroll
      for (int q = 0; q < NG; ++q) any = any || jj < s_cnt[q];
      if (!any) return;
      if (jj < s_cnt[h] && ++found == ahead) break;
    }
    issue(tile_of(h, s_t0[h], jj), rank + ahead);
  };

  pdl_trigger();
  for (int i = threadIdx.x; i < C::TW_TOTAL; i += T_::CTA_THREADS) tws[i] = tables[i];
  if (threadIdx.x == 0) {
    for (int q = 0; q < NBUF; ++q) {
      mbar_init(&full[q], 1);
      issued[q] = -1;
      done[q] = 0;
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  pdl_wait();
  if (threadIdx.x == 0) {
    for (int a = 1; a <= NBUF; ++a) issue_ahead(NG - 1, -1, -1, a);
  }

  // this lane's columns of the output (bytes from the tile's first column)
  const int colt = 2 * col;
  const long long off_out =
      ((long long)(colt / p.P) * p.mout.a_c + (colt % p.P) * p.mout.a_p) * out_eb;
  const long long ts_rowbytes = p.mout.a_n * out_eb;
  using acc_t = typename std::conditional<EPI == EPI_STOKES_I, float, float2>::type;
  acc_t acc[16];
  auto acc_clear = [&]() {
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      if constexpr (EPI == EPI_STOKES_I) acc[i] = 0.f;
      else acc[i] = make_float2(0.f, 0.f);
    }
  };
  // tile row b + 16 i at inner offset nrest is time n = (row << log2nmul) + nrest and lands in
  // output row (n - crop_start) >> tsum_log2, or its phase bin (see tsum_flush in pbk_fast.cuh)
  auto flush = [&](char* colbase, unsigned nrest) {
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      const long long n = ((long long)(b + 16 * i) << p.log2nmul) + nrest;
      if constexpr (EPI == EPI_STOKES_I) {
        if (acc[i] != 0.f)
          atomicAdd(reinterpret_cast<float*>(tsum_row(p, colbase, n, ts_rowbytes)), acc[i]);
      } else {
        if (acc[i].x != 0.f || acc[i].y != 0.f) {
          float* a = reinterpret_cast<float*>(tsum_row(p, colbase, n, ts_rowbytes));
          if (acc[i].x != 0.f) atomicAdd(a, acc[i].x);
          if (acc[i].y != 0.f) atomicAdd(a + 1, acc[i].y);
        }
      }
    }
    acc_clear();
  };
  acc_clear();
  char* ts_colbase = nullptr;
  unsigned ts_nrest = 0;

  // float4 index of (row, this lane's column) inside a tile buffer
  auto slot = [&](int row) -> int { return row * 16 + half * 8 + (chunk ^ ((2 * row + half) & 7)); };

  for (long long j = 0; j < my_cnt; ++j) {
    const long long rank = rank_of(g, j);
    const int buf = (int)(rank % NBUF);
    const float4* tile = reinterpret_cast<const float4*>(smem_raw + (size_t)buf * T_::TILE_BYTES);
    float4* tilew = reinterpret_cast<float4*>(smem_raw + (size_t)buf * T_::TILE_BYTES);
    // our load has been issued (one lane polls, sleeping in between: sixteen warps spinning on a
    // shared-memory word would take the issue slots and the LSU from the warps that compute) ...
    if (lane == 0)
      while (issued[buf] < rank) __nanosleep(64);
    __syncwarp();
    mbar_wait(&full[buf], (uint32_t)((rank / NBUF) & 1));       // ... and has landed
    const TileInfo ti = info_ring[buf];
    {
      char* colbase = reinterpret_cast<char*>(p.out) + ti.bo + off_out -
                      ((long long)ti.nrest - p.crop_start) * ts_rowbytes;
      if (ts_colbase != nullptr &&
          (colbase != ts_colbase || ((ti.nrest - ts_off) & ((1u << p.tsum_log2) - 1)) == 0))
        flush(ts_colbase, ts_nrest);
      ts_colbase = colbase;
      ts_nrest = ti.nrest;
    }
    if (lane < 16) {     // (any 16 lanes: the table is indexed by the register number)
      const float2 gv = unit_root((unsigned long long)ti.nrest * (unsigned)(C::KS * lane), p.log2M);
      G4[lane] = make_float4(gv.x, gv.y, gv.y, gv.x);
    }
    c2 v[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = lds_c2(tile, slot(b + 16 * i));
    __syncwarp();          // G is written; every lane holds its rows: the columns can be overwritten
    level_twiddle<16, true>(p, v, ti.nrest, (unsigned)b, G4);
    Butterfly<16, true>::run(v);
#pragma unroll
    for (int i = 0; i < 16; ++i) sts_c2(tilew, slot(16 * b + ((i + b) & 15)), v[i]);
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = lds_c2(tile, slot(16 * i + ((b + i) & 15)));
    // the buffer is free as far as this warp goes: order its generic-proxy accesses before the TMA
    // write that refills it, count the warp, and let the last of the group's warps start the load
    // of rank + NBUF into it
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) {
      __threadfence_block();
      if (atomicAdd(&done[buf], 1) == WPG - 1) {
        done[buf] = 0;
        __threadfence_block();
        issue_ahead(g, j, rank, NBUF);
      }
    }
    stage_twiddle<16, 16, true>(v, tws + C::tw_off(0), b);
    Butterfly<16, true>::run(v);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      if ((unsigned)(b + 16 * i) - ti.row_lo >= ti.row_cnt) continue;
      if constexpr (EPI == EPI_STOKES_I) {
        float s = acc[i];
        s = fmaf(v[i].re.x, v[i].re.x, s);
        s = fmaf(v[i].im.x, v[i].im.x, s);
        s = fmaf(v[i].re.y, v[i].re.y, s);
        s = fmaf(v[i].im.y, v[i].im.y, s);
        acc[i] = s;
      } else {
        acc[i] = p_fma(v[i].re, v[i].re, p_fma(v[i].im, v[i].im, acc[i]));
      }
    }
  }
  if (ts_colbase != nullptr) flush(ts_colbase, ts_nrest);
}

}  // namespace pbk
