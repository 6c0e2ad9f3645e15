// pbk_fast_inst.cuh -- shared body of the per-family instantiation units.
#pragma once
#include <algorithm>

#include "pbk_fast.cuh"
#include "pbk_fast_launch.h"

namespace pbk {

template <class C>
static void cfg_info(FastInfo* info) {
  info->log2pw = C::LOG2PW;
  info->tw_count = C::TW_TOTAL;
  info->threads = C::NT;
  info->minb = C::MINB;
  info->smem = C::SMEM_BYTES;
  info->tsum_ok = (C::stride(0) * C::PW) % C::NT == 0;
}

template <int MODE, class C, int LOADK, int EPI, bool TWOCH, bool NARROW, bool SIGNINV = false,
          bool TSUM = false>
static cudaError_t cfg_launch_variant(const PassArgs& a, const float2* d_tables, long long ntiles,
                                      int num_sms, cudaStream_t st) {
  auto kern = fast_pass_kernel<MODE, C, LOADK, EPI, TWOCH, NARROW, SIGNINV, TSUM>;
  constexpr size_t smem = C::smem_bytes(NARROW);
  static bool attr_done[16] = {};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 16 && !attr_done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess) return e;
    attr_done[dev] = true;
  }
  const long long resident = (long long)num_sms * C::MINB;
  unsigned grid = (unsigned)std::min<long long>(ntiles - a.tile0, resident);
  // a TSUM CTA's contiguous run of tiles must span at least two whole groups of summed rows
  if (TSUM) {
    const long long q = a.tsum_q;
    grid = (unsigned)(q * std::max<long long>(1, std::min<long long>(resident / q,
                                                                      (ntiles / q) >> (a.tsum_log2 + 1))));
  }
  if (MODE == MODE_FWD && EPI == EPI_INTENSITY)   // whole groups of 2^fsum_g_log2 tiles per CTA
    grid = (unsigned)std::min<long long>(std::max<long long>(1, ntiles >> a.fsum_g_log2), resident);
  return pdl_launch(kern, dim3(grid, std::max(1, a.trials)), dim3(C::NT), smem, st, a, d_tables,
                    ntiles);
}

// NARROW (arrays with fewer lanes per row than the tile is wide) is a separate instantiation so
// that the common wide case keeps tile-uniform bookkeeping
template <int MODE, class C, int LOADK, int EPI, bool TWOCH = false, bool SIGNINV = false>
static cudaError_t cfg_launch_mode(const PassArgs& a, const float2* d_tables, long long ntiles,
                                   int num_sms, cudaStream_t st) {
  if (a.I < C::W)
    return cfg_launch_variant<MODE, C, LOADK, EPI, TWOCH, true, SIGNINV>(a, d_tables, ntiles,
                                                                         num_sms, st);
  return cfg_launch_variant<MODE, C, LOADK, EPI, TWOCH, false, SIGNINV>(a, d_tables, ntiles,
                                                                        num_sms, st);
}

// inverse passes always read the scratch array; a MID pass reads the user's complex64 input only
// when it is the whole plan (then it is also final)
template <class C>
static cudaError_t cfg_launch(int mode, const PassArgs& a, const float2* d_tables,
                              long long ntiles, int num_sms, cudaStream_t st) {
  switch (mode) {
    case MODE_FWD:
      if (a.sign > 0) {    // inverse exponent (ifft / ISTFT plans): conjugated butterflies and twiddles
        if (a.final_epi) {
          if (a.load_kind == LOAD_PLANAR)
            return cfg_launch_mode<MODE_FWD, C, LK_PLANAR, EPI_C64, false, true>(a, d_tables, ntiles,
                                                                                 num_sms, st);
          if (a.load_kind == LOAD_TRANSP)
            return cfg_launch_mode<MODE_FWD, C, LK_TRANSP, EPI_C64, false, true>(a, d_tables, ntiles,
                                                                                 num_sms, st);
          return cfg_launch_mode<MODE_FWD, C, LK_C64, EPI_C64, false, true>(a, d_tables, ntiles,
                                                                            num_sms, st);
        }
        if (a.load_kind == LOAD_PLANAR)
          return cfg_launch_mode<MODE_FWD, C, LK_PLANAR, EPI_SCRATCH, false, true>(a, d_tables,
                                                                                   ntiles, num_sms, st);
        return cfg_launch_mode<MODE_FWD, C, LK_C64, EPI_SCRATCH, false, true>(a, d_tables, ntiles,
                                                                              num_sms, st);
      }
      if (a.final_epi && a.fsum_log2 > 0) {  // channelizer with a detected, frequency-summed output
        // one lane pair per row: every lane row of the tile is a contiguous run of L rows in the
        // scratch array, read coalesced and transposed through shared memory
        if (a.load_kind == LOAD_TRANSP_PLANAR)
          return cfg_launch_variant<MODE_FWD, C, LK_TRANSP_PLANAR, EPI_INTENSITY, false, true>(
              a, d_tables, ntiles, num_sms, st);
        return cfg_launch_variant<MODE_FWD, C, LK_PLANAR, EPI_INTENSITY, false, true>(
            a, d_tables, ntiles, num_sms, st);
      }
      if (a.final_epi) {   // last pass of a forward FFT / STFT plan: scaled natural-order output
        if (a.load_kind == LOAD_PLANAR)
          return cfg_launch_mode<MODE_FWD, C, LK_PLANAR, EPI_C64>(a, d_tables, ntiles, num_sms, st);
        return cfg_launch_mode<MODE_FWD, C, LK_C64, EPI_C64>(a, d_tables, ntiles, num_sms, st);
      }
      if (a.load_kind == LOAD_I8X2)
        return cfg_launch_mode<MODE_FWD, C, LK_I8, EPI_SCRATCH>(a, d_tables, ntiles, num_sms, st);
      if (a.load_kind == LOAD_U4X2)
        return cfg_launch_mode<MODE_FWD, C, LK_U4, EPI_SCRATCH>(a, d_tables, ntiles, num_sms, st);
      if (a.load_kind == LOAD_U2X2)
        return cfg_launch_mode<MODE_FWD, C, LK_U2, EPI_SCRATCH>(a, d_tables, ntiles, num_sms, st);
      if (a.load_kind == LOAD_PLANAR)
        return cfg_launch_mode<MODE_FWD, C, LK_PLANAR, EPI_SCRATCH>(a, d_tables, ntiles, num_sms,
                                                                    st);
      return cfg_launch_mode<MODE_FWD, C, LK_C64, EPI_SCRATCH>(a, d_tables, ntiles, num_sms, st);
    case MODE_MID:
      if (a.P == 1) {   // single-polarisation data: a lane pair is two channels
        if (!a.final_epi)
          return cfg_launch_mode<MODE_MID, C, LK_PLANAR, EPI_SCRATCH, true>(a, d_tables, ntiles,
                                                                            num_sms, st);
        if (a.epi_kind == EPI_C64)
          return cfg_launch_mode<MODE_MID, C, LK_C64, EPI_C64, true>(a, d_tables, ntiles, num_sms,
                                                                     st);
        return cfg_launch_mode<MODE_MID, C, LK_C64, EPI_INTENSITY, true>(a, d_tables, ntiles,
                                                                         num_sms, st);
      }
      if (!a.final_epi)
        return cfg_launch_mode<MODE_MID, C, LK_PLANAR, EPI_SCRATCH>(a, d_tables, ntiles, num_sms,
                                                                    st);
      switch (a.epi_kind) {
        case EPI_C64:
          return cfg_launch_mode<MODE_MID, C, LK_C64, EPI_C64>(a, d_tables, ntiles, num_sms, st);
        case EPI_INTENSITY:
          return cfg_launch_mode<MODE_MID, C, LK_C64, EPI_INTENSITY>(a, d_tables, ntiles, num_sms,
                                                                     st);
        default:
          return cfg_launch_mode<MODE_MID, C, LK_C64, EPI_STOKES_I>(a, d_tables, ntiles, num_sms,
                                                                    st);
      }
    default:
      if (!a.final_epi)
        return cfg_launch_mode<MODE_INV, C, LK_PLANAR, EPI_SCRATCH>(a, d_tables, ntiles, num_sms,
                                                                    st);
      if (a.tsum_log2 > 0) {   // detected output with the time sum fused into the epilogue
        if (a.epi_kind == EPI_INTENSITY)
          return cfg_launch_variant<MODE_INV, C, LK_PLANAR, EPI_INTENSITY, false, false, false, true>(
              a, d_tables, ntiles, num_sms, st);
        return cfg_launch_variant<MODE_INV, C, LK_PLANAR, EPI_STOKES_I, false, false, false, true>(
            a, d_tables, ntiles, num_sms, st);
      }
      switch (a.epi_kind) {
        case EPI_C64:
          return cfg_launch_mode<MODE_INV, C, LK_PLANAR, EPI_C64>(a, d_tables, ntiles, num_sms, st);
        case EPI_INTENSITY:
          return cfg_launch_mode<MODE_INV, C, LK_PLANAR, EPI_INTENSITY>(a, d_tables, ntiles,
                                                                        num_sms, st);
        default:
          return cfg_launch_mode<MODE_INV, C, LK_PLANAR, EPI_STOKES_I>(a, d_tables, ntiles,
                                                                       num_sms, st);
      }
  }
}

}  // namespace pbk
