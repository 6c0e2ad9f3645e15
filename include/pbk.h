/* pbk.h -- C ABI of libpbk.so: B200 (sm_100a) kernels for pulsarbat's FFT baseband hot path.
 *
 * The reference (theXYZT/pulsarbat) is pure Python and has no FFI of its own (SURVEY.md 8b);
 * the seams it offers are function-level.  Every entry point below names the reference
 * interface it stands in for (paths relative to /root/reference/pulsarbat).  INTEGRATION.md
 * shows the ctypes stub a pulsarbat maintainer would add at each seam.
 *
 * Conventions
 *  - Every function returns 0 (PBK_OK) or a negative pbk_status; nothing throws or aborts.
 *    pbk_last_error() returns a thread-local message for the last failure on this thread.
 *  - Arrays are C-ordered with time slowest: (nsamp, nchan, npol) complex64 = float pairs
 *    (core.py:36-39, 392-394, 786-787).  npol is the product of all axes after frequency.
 *  - The caller owns every data pointer.  The library owns plans and their workspaces.
 *  - *_host entry points take HOST pointers (pageable or pinned), copy in, run, copy out and
 *    synchronise before returning; they may be called concurrently from several threads (a
 *    plan serialises its own executions).  *_device entry points take DEVICE pointers on the
 *    plan's device, enqueue on `stream` (a cudaStream_t cast to void*, NULL = legacy default
 *    stream) and do not synchronise.  A plan owns its scratch arrays (one, or two of N*C*P*8
 *    bytes each when that is at most 1/5 of the device memory; pbk_plan_info reports the total):
 *    executions of the same plan must be ordered on the device (same stream, or events between
 *    streams).  A *_device execution only enqueues kernels (and a memset of a summed output,
 *    and the device-to-device copies of a staged array, below): it can be captured into a CUDA
 *    graph once the plan's lazily allocated buffers exist.  The passes of one execution are chained with
 *    programmatic dependent launch (PBK_PDL=0 switches it off); the first pass waits for the
 *    previous kernel of the stream to complete like any kernel, and kernels the caller enqueues
 *    afterwards wait for the last pass.
 *  - Device pointers need only the alignment of their element type: 8 bytes for complex64 and
 *    int64, 4 for float32 and int32, 2 for int8 (re, im) pairs, 1 for packed u4 / u2 rows.
 *    16-byte aligned arrays take the vectorised kernels.  Other arrays give the same result on a
 *    scalar path, or through a plan-owned 16-byte aligned staging buffer and a device-to-device
 *    copy where the work needs the vectorised kernels: the output of a plan whose last pass sums
 *    time, detects or recombines even / odd samples, and the profile of
 *    pbk_stft_fold_exec_device.  The staging buffer is allocated at the first execution that
 *    needs it and counted in pbk_plan_info's workspace bytes.
 *  - There is no CPU fallback: without a CUDA device every call fails with PBK_ERR_CUDA.
 */
#ifndef PBK_H_
#define PBK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PBK_VERSION 100

typedef struct pbk_plan pbk_plan;

enum pbk_status {
  PBK_OK = 0,
  PBK_ERR_INVALID = -1,     /* bad argument */
  PBK_ERR_UNSUPPORTED = -2, /* valid request this build cannot run (e.g. a transform too long) */
  PBK_ERR_CUDA = -3,        /* CUDA runtime error / no device */
  PBK_ERR_NOMEM = -4
};

enum pbk_dtype {
  PBK_C64 = 0,
  PBK_I8X2 = 1, /* interleaved (re, im) int8 pairs */
  PBK_F32 = 2,  /* real float32 (imaginary part zero); ramp plans only */
  /* packed raw baseband, decoded in the load of the first pass (builder-defined like PBK_I8X2,
   * SURVEY 8a row U: the reference receives decoded samples from `baseband`,
   * readers/_baseband_readers.py:139-153).  Elements are packed in array order, first element in
   * the least significant bits; nchan * npol must be even. */
  PBK_U4X2 = 3, /* one byte per complex sample: low nibble re, high nibble im, offset binary
                   (value = code - 8) */
  PBK_U2X2 = 4  /* four bits per complex sample: bits 1:0 re, bits 3:2 im; two complex samples
                   per byte; codes 0..3 -> -3.3359, -1, +1, +3.3359 (the usual 2-bit levels) */
};

enum pbk_out_kind {
  PBK_OUT_C64 = 0,       /* dedispersed voltages, complex64                              */
  PBK_OUT_INTENSITY = 1, /* re^2+im^2 per pol, float32      (core.py:766-774)            */
  PBK_OUT_STOKES_I = 2   /* |A|^2+|B|^2, float32, npol == 2 (core.py:944-948, 956-960)   */
};

int pbk_version(void);
const char* pbk_last_error(void);
const char* pbk_status_string(int status);
int pbk_device_count(int* count);
/* PCI bus id of a CUDA device ("0000:1b:00.0"), for binding the host process to the GPU's NUMA
 * node (one process per GPU, SURVEY 8e); no reference counterpart */
int pbk_device_pci_bus_id(int device, char* buf, int n);
/* free / total bytes of device memory (the host mirror caps its plan cache by workspace bytes);
 * no reference counterpart */
int pbk_device_mem_info(int device, size_t* free_bytes, size_t* total_bytes);

/* ---- coherent dedispersion ---------------------------------------------------------------
 * Replaces transforms/dedispersion.py:81-133 `coherent_dedispersion` for numpy/dask blocks and
 * device buffers, including the chirp of dedispersion.py:19-23/59-75, which is generated inside
 * the kernel (FP64 phase) and never stored.  crop_start/crop_stop are computed by the CALLER
 * exactly as dedispersion.py:127-131 so that the integer crop is bit-identical to the reference;
 * pass (0, nsamp) for the uncropped circular result.
 *   out_kind C64:        out is (crop_stop-crop_start, nchan, npol) complex64
 *   out_kind INTENSITY:  out is (rows, nchan, npol) float32
 *   out_kind STOKES_I:   out is (rows, nchan) float32
 * with rows = (crop_stop-crop_start) / downsample when downsample > 1 (time sum of `downsample`
 * consecutive samples, tail dropped; builder-defined, SURVEY 8a row R; only for float outputs).
 */
typedef struct pbk_dedisp_desc {
  int64_t nsamp;              /* N >= 2; powers of two >= 16 run on the tile-FFT passes, any other
                                 length through Bluestein on top of them (pbk_blue.cuh) */
  int64_t nchan;              /* C */
  int64_t npol;               /* P */
  int32_t in_dtype;           /* pbk_dtype */
  int32_t out_kind;           /* pbk_out_kind */
  double dm;                  /* pc / cm^3 */
  double sample_rate_hz;      /* per-channel sample rate == channel bandwidth (core.py:761) */
  double ref_freq_hz;         /* may be +inf */
  const double* chan_freq_hz; /* [nchan] channel centre frequencies (core.py:569-574) */
  int64_t crop_start;
  int64_t crop_stop;
  int64_t downsample;         /* 1 = none */
  int32_t explicit_chirp;     /* 1: a (nsamp, nchan) complex64 chirp is passed at execution
                                 (dedispersion.py:121-124, `chirp=` argument) */
  int32_t device;             /* CUDA device ordinal */
} pbk_dedisp_desc;

int pbk_dedisp_plan_create(const pbk_dedisp_desc* desc, pbk_plan** plan);
/* rows of the output, elements per row, bytes per element */
int pbk_dedisp_out_shape(const pbk_plan* plan, int64_t* rows, int64_t* row_elems,
                         int64_t* elem_bytes);
int pbk_dedisp_exec_host(pbk_plan* plan, const void* in, void* out, const void* chirp);
int pbk_dedisp_exec_device(pbk_plan* plan, const void* d_in, void* d_out, const void* d_chirp,
                           void* stream);
/* coherent dedispersion -> detection -> time sum -> fold (row F) as one execution of a dedispersion
 * plan whose out_kind is INTENSITY or STOKES_I (and no explicit chirp): the time-summed power of
 * output row j is ADDED to profile[bin(j), :] (float32 (nbin, row_elems), caller-zeroed or carrying
 * earlier blocks) and counts[bin(j)] += 1 (int64 (nbin,)), bin(j) from the phase polynomial at
 * t = (n0 + j) / sample_rate_hz exactly as pbk_fold, where sample_rate_hz is the OUTPUT-ROW rate
 * (input rate / downsample).  Device pointers, enqueued on `stream`; nothing is written to a
 * voltage or intensity array of the caller.
 * When the plan sums time in the epilogue of its last inverse pass (pbk_plan_describe shows
 * ":timesum"), the intensity (out_rows x row_elems floats) is at least 256 MiB, there are at
 * most 512 rows per bin and d_profile is 16-byte aligned, the bins are computed first and that pass adds its group sums straight
 * into the profile, so the intensity never reaches HBM; otherwise (smaller intensities stay in L2
 * between two steps, and many rows per bin serialise the atomics) the plan's normal execution
 * writes a plan-owned float32 buffer of out_rows x row_elems (allocated at the first such
 * execution and counted in pbk_plan_info's workspace bytes), which is then folded.  Bins and counts are exact on both
 * routes; the fused profile collects many float atomics per row in any order, so it is
 * reproducible to rounding, not bit for bit.  ncoef in [1, 16], finite coefficients, finite
 * sample_rate_hz > 0, nbin > 0; a C64 plan returns PBK_ERR_INVALID; an empty crop returns PBK_OK
 * and touches nothing.  A later pbk_dedisp_exec_device of the same plan is unaffected. */
int pbk_dedisp_fold_exec_device(pbk_plan* plan, const void* d_in, void* d_profile, void* d_counts,
                                const double* coeffs, int32_t ncoef, double sample_rate_hz,
                                int64_t n0, int32_t nbin, void* stream);

/* Coherent dedispersion of one block at ndm trial DMs (a coherent DM search, or refining the DM of
 * a known pulsar): the forward transform of the input runs once per execution, and the chirp pass
 * and every pass after it run once per trial.  `desc` means what it means for
 * pbk_dedisp_plan_create, except that desc->dm is ignored: trial k uses dms[k] (any finite value,
 * 0 and negative DMs included).  All trials share one crop, one downsample and one out_kind; raw
 * int8 / u4 / u2 input works.  explicit_chirp, ndm < 1, a NULL dms and a non-finite DM return
 * PBK_ERR_INVALID.  Each trial computes bit for bit what a pbk_dedisp_plan_create plan with the
 * same desc and dm = dms[k] computes.
 * Execute with pbk_dedisp_exec_device / pbk_dedisp_exec_host: out is a contiguous
 * (ndm, rows, row_elems) array, trial k at out + k * rows * row_elems * elem_bytes, where
 * pbk_dedisp_out_shape reports the shape of ONE trial.  A trial slab that is not 16-byte aligned
 * is written through the plan's staging buffer.  The plan keeps a second scratch array for the
 * shared forward result; the per-trial inverse passes run in place in the other one.  When every
 * per-trial pass runs on the LDG fast kernels and has fewer tiles than the GPU holds CTAs, T > 1
 * trials run as one launch (gridDim.y = T; the other array then holds T slabs), with T chosen by the
 * plan for about two waves of CTAs and bounded by the memory of the slabs; otherwise T = 1.
 * Lengths that are not powers of two (Bluestein) run their whole execution once per trial.  pbk_dedisp_fold_exec_device on a
 * trial plan returns PBK_ERR_UNSUPPORTED.  pbk_plan_describe lists the shared passes, then
 * "TRIALS:ndm=<ndm>:per_launch=<T>" and the passes run per batch of T trials; pbk_plan_info and
 * pbk_plan_segments count the shared passes once and the per-trial launches once per batch, so
 * launches = shared passes + ceil(ndm / T) x per-trial passes.  The last timed segment of a batch
 * ends where the next batch's first launch starts, so it includes the zeroing of a time-summed
 * output and the copy out of a staged output between them. */
int pbk_dedisp_trials_plan_create(const pbk_dedisp_desc* desc, const double* dms, int32_t ndm,
                                  pbk_plan** plan);
/* number of trial DMs of a plan: ndm for a trial plan, 1 for every other plan */
int pbk_plan_trials(const pbk_plan* plan, int32_t* ndm);

/* Overlap-save execution of a pbk_dedisp_plan_create plan over nblocks blocks of one
 * device-resident stream (builder-defined, SURVEY 8a row O).  With advance = crop_stop - crop_start
 * and an input row of nchan * npol elements of in_dtype (row bytes = nchan * npol * bits / 8, so
 * int8, u4 and u2 rows work), block b reads the plan's nsamp rows starting at row b * advance of
 * d_in and writes the plan's normal output at d_out + b * rows * row_elems * elem_bytes
 * (pbk_dedisp_out_shape): d_in must hold (nblocks - 1) * advance + nsamp rows and d_out nblocks
 * output slabs.  Block b is bit for bit what pbk_dedisp_exec_device writes into a 16-byte aligned
 * buffer from d_in + b * advance * row bytes.  Enqueue only, like pbk_dedisp_exec_device.
 * nblocks == 0 or an empty crop returns PBK_OK and touches nothing; nblocks < 0 or a NULL pointer
 * returns PBK_ERR_INVALID; a trial plan or an explicit-chirp plan returns PBK_ERR_UNSUPPORTED.
 * When d_in, d_out and the block stride (advance * row bytes) are 16-byte aligned and the plan can
 * batch (pbk_plan_blocks_per_launch > 1), T blocks run as one launch per pass (gridDim.y = T) and
 * a time-summed output is zeroed once per batch; the last batch may be partial.  The T scratch
 * slabs of each scratch array are allocated at the first batched execution and counted in
 * pbk_plan_info's workspace bytes.  Otherwise each block runs the single execution at its pointers,
 * with an output slab that is not 16-byte aligned written through the staging buffer.
 * pbk_plan_profile does not time block executions. */
int pbk_dedisp_exec_blocks_device(pbk_plan* plan, const void* d_in, int64_t nblocks, void* d_out,
                                  void* stream);
/* Blocks batched per launch (T) by pbk_dedisp_exec_blocks_device on a 16-byte aligned stream: about
 * two waves of resident CTAs in every pass, bounded by the memory of T slabs in each scratch array;
 * 1 when the plan cannot batch (a pass on the generic or TMA kernels, a Bluestein length, a
 * one-level plan, an output through the float buffer or a slab that is not a multiple of 16 bytes),
 * and for trial and ramp plans. */
int pbk_plan_blocks_per_launch(const pbk_plan* plan, int32_t* T);

/* ---- FFT-domain phase ramp / band mask ("next" rows: time_shift, freq_shift) ------------------
 * Replaces the core of transforms/transforms.py:268-271 (time_shift) and :348-361 (freq_shift):
 *   out[:, col] = ifft(fft(in[:, col]) * H_col),
 *   H_col[k] = 0 if lo_col <= fftshift_position(k) < hi_col, else exp(-2 pi i s_col fftfreq(N,1)[k])
 * in/out are (nsamp, ncols) complex64.  Execute with pbk_dedisp_exec_host / _device (chirp NULL).
 * zero_lo / zero_hi may be NULL (no zeroed band), shift_samples may be NULL (no ramp). */
enum pbk_ramp_flags {
  PBK_RAMP_HILBERT = 1,    /* multiply by the analytic-signal weights h = 1,2,..,2,1,0,..,0
                              (utils.py:50-54 real_to_complex) */
  PBK_RAMP_REAL_INPUT = 2  /* in is (nsamp, ncols) float32 */
};
int pbk_ramp_plan_create(int64_t nsamp, int64_t ncols, const double* shift_samples,
                         const int64_t* zero_lo, const int64_t* zero_hi, int32_t flags,
                         int32_t device, pbk_plan** plan);
/* out[m, col] = (-1)^m in[2m, col]: the exp(-i pi n/2) mix + decimation by 2 that ends
 * utils.py:56-61 real_to_complex; out is (ceil(nsamp/2), ncols) complex64 */
int pbk_decimate2(const void* in, void* out, int64_t nsamp, int64_t ncols, int32_t on_device,
                  int32_t device, void* stream);
/* out[n, col] = in[n, col] * exp(+2 pi i cycles_per_sample[col] * n)   (transforms.py:346) */
int pbk_mix(const void* in, void* out, int64_t nsamp, int64_t ncols,
            const double* cycles_per_sample, int32_t on_device, int32_t device, void* stream);

/* ---- axis-0 complex FFT --------------------------------------------------------------------
 * Replaces fft.py:30-48 `pb.fft.fft` / `pb.fft.ifft` with axis=0 for complex64 data (scipy
 * "backward" normalisation: forward unscaled, inverse 1/n), natural-order output.
 * Data is (outer, n, inner) complex64, transform along n; any n >= 2 (powers of two run on the
 * tile-FFT passes directly, other lengths through Bluestein on top of them).
 */
int pbk_fft_plan_create(int64_t outer, int64_t n, int64_t inner, int32_t inverse, int32_t device,
                        pbk_plan** plan);

/* ---- channelize / unchannelize -------------------------------------------------------------
 * Replaces contrib/misc.py:17-55 `stft` and :58-93 `istft` (boxcar, no overlap):
 *   forward:  in (nseg*nperseg, nchan, npol) -> out (nseg, nchan*nperseg, npol),
 *             out[s, c*n + ((k + n/2) mod n), p] = (1/n) sum_t in[s*n+t, c, p] e^{-2 pi i k t/n}
 *   inverse:  in (nseg, nchan_out*nperseg, npol) -> out (nseg*nperseg, nchan_out, npol)
 * Any nperseg >= 2 (the reference's tests use 33).  The input is never modified (the reference's
 * istft scales its input in place, misc.py:82-83).  A forward plan for ONE single-polarisation
 * channel whose nperseg is a power of two with a two-level half-length plan (2^14 .. 2^22 and
 * possibly longer; 2 .. 2^13 have a one-level half) is built on the (nperseg/2, 2) even / odd view
 * of the stream and recombined in the last pass (pbk_plan_describe shows ":evenodd"; PBK_NO_SPLIT=1
 * disables it) -- same input, same output, the compile-time-shaped kernels instead of the
 * run-time-shaped ones.  Every other nperseg runs the full-length plan (Bluestein when it is not a
 * power of two).
 */
int pbk_stft_plan_create(int64_t nseg, int64_t nperseg, int64_t nchan, int64_t npol,
                         int32_t inverse, int32_t device, pbk_plan** plan);
/* Channelizer with a DETECTED, frequency-summed output (BASELINE configs[3]: channelize, then
 * power per fine channel, then sum over `freq_sum` adjacent fine channels -- misc.py:41-52 followed
 * by core.py:766-774 / :948 and the builder-defined channel sum of pbk_detect_scrunch) as ONE plan:
 * the detection runs in the epilogue of the last FFT pass, so the channelized voltages never
 * reach HBM.
 *   in  (nseg*nperseg, 1, npol) complex64
 *   out (nseg, nperseg/freq_sum, npol) float32   out_kind INTENSITY, npol 1 or 2
 *       (nseg, nperseg/freq_sum)       float32   out_kind STOKES_I (npol 2)
 * with out[s, c', p] = sum_{f < freq_sum} |stft(in)[s, c'*freq_sum + f, p]|^2, fftshift and 1/n
 * scale of the reference's stft included.  One channel only, a power-of-two segment length that
 * the plan splits into two levels (of the lengths tested: npol 2 from 2^13 to 2^20, npol 1 --
 * planned at half length -- from 2^14 to 2^22; not 2^22 with npol 2, not 2^24) and a power-of-two
 * freq_sum that divides the first level in whole
 * last-pass tiles; other shapes, any length that is not a power of two among them, return
 * PBK_ERR_UNSUPPORTED (use pbk_stft_plan_create + pbk_detect_scrunch).
 * Executed with pbk_fft_exec_device / pbk_fft_exec_host. */
int pbk_stft_detect_plan_create(int64_t nseg, int64_t nperseg, int64_t nchan, int64_t npol,
                                int32_t out_kind, int64_t freq_sum, int32_t device,
                                pbk_plan** plan);
/* ... and the fold behind it (row F) in the same launches: the power sums of segment s are ADDED
 * to profile[bin(s), :, :] (float32 (nbin, nperseg/freq_sum[, npol]), caller-zeroed or carrying
 * earlier blocks) and counts[bin(s)] += 1 (int64 (nbin,)), bin(s) from the phase polynomial at
 * t = (n0 + s) / sample_rate_hz exactly as pbk_fold (sample_rate_hz is the SEGMENT rate).  `plan`
 * comes from pbk_stft_detect_plan_create; device pointers, enqueued on `stream`.  A profile that
 * is not 16-byte aligned is copied into the plan's staging buffer, accumulated there by the same
 * launches and copied back. */
int pbk_stft_fold_exec_device(pbk_plan* plan, const void* d_in, void* d_profile, void* d_counts,
                              const double* coeffs, int32_t ncoef, double sample_rate_hz,
                              int64_t n0, int32_t nbin, void* stream);
/* the channelizer fed with raw baseband (PBK_I8X2 / PBK_U4X2 / PBK_U2X2, decoded in the load of the
 * first pass; forward transform only): what readers/_baseband_readers.py:139-153 + misc.py:17-55
 * do in two steps on the host */
int pbk_stft_plan_create_raw(int64_t nseg, int64_t nperseg, int64_t nchan, int64_t npol,
                             int32_t in_dtype, int32_t device, pbk_plan** plan);

/* execution for FFT and STFT plans */
int pbk_fft_exec_host(pbk_plan* plan, const void* in, void* out);
int pbk_fft_exec_device(pbk_plan* plan, const void* d_in, void* d_out, void* stream);

/* ---- complex128 -----------------------------------------------------------------------------
 * The reference keeps complex128 through its transforms (scipy preserves the dtype:
 * dedispersion.py:125, fft.py:34, misc.py:47,87; core.py:766-774 returns float64 power), and its
 * own test of +-DM reversibility asserts atol 3e-8 (tests/test_dedispersion.py:73-98).  These entry
 * points compute in FP64 (Stockham radix-4 passes, csrc/pbk_f64.cuh; any other length through
 * Bluestein's chirp-z identity on top of them): complex128 is never narrowed to complex64.
 * Plan-less; host pointers (synchronous) or device pointers (`on_device`, enqueued on `stream`).
 *   pbk_dedisp_c128: in (nsamp, nchan, npol) complex128 -> out rows [crop_start, crop_stop) as
 *                    complex128 (C64 kind), float64 per-pol power or float64 Stokes I; the chirp
 *                    is generated in FP64 and rounded to complex64 exactly as dedispersion.py:23
 *                    does, or taken from `chirp` ((nsamp, nchan) complex64) when non-NULL
 *   pbk_fft_c128:    (outer, n, inner) complex128, axis 1, scipy "backward" normalisation
 *   pbk_stft_c128:   stft / istft of (nseg*nperseg, nchan, npol) complex128
 *   pbk_detect_c128: float64 |z|^2 per element, or Stokes I over pol pairs */
int pbk_dedisp_c128(const void* in, void* out, int64_t nsamp, int64_t nchan, int64_t npol,
                    int32_t out_kind, double dm, double sample_rate_hz, double ref_freq_hz,
                    const double* chan_freq_hz, int64_t crop_start, int64_t crop_stop,
                    const void* chirp, int32_t on_device, int32_t device, void* stream);
int pbk_fft_c128(const void* in, void* out, int64_t outer, int64_t n, int64_t inner,
                 int32_t inverse, int32_t on_device, int32_t device, void* stream);
int pbk_stft_c128(const void* in, void* out, int64_t nseg, int64_t nperseg, int64_t nchan,
                  int64_t npol, int32_t inverse, int32_t on_device, int32_t device, void* stream);
int pbk_detect_c128(const void* in, void* out, int64_t nsamp, int64_t nchan, int64_t npol,
                    int32_t out_kind, int32_t on_device, int32_t device, void* stream);

/* ---- detection / integration ---------------------------------------------------------------
 * pbk_detect:     float32 power from complex64 voltages (core.py:766-774; Stokes I core.py:948).
 *                 in (nsamp, nchan, npol) c64 -> out (nsamp/downsample, nchan[, npol]) f32
 * pbk_downsample: out[j] = sum_{m<M} in[j*M+m] over time on float32 (builder-defined, row R).
 * Both take device pointers when `on_device` != 0, host pointers otherwise.
 */
int pbk_detect(const void* in, void* out, int64_t nsamp, int64_t nchan, int64_t npol,
               int32_t out_kind, int64_t downsample, int32_t on_device, int32_t device,
               void* stream);
/* pbk_detect with an additional sum over `freq_sum` adjacent channels (frequency scrunching
 * after channelize; builder-defined like row R):
 *   out[j, c', (p)] = sum_{m<time_sum} sum_{f<freq_sum} |in[j*time_sum+m, c'*freq_sum+f, p]|^2 */
int pbk_detect_scrunch(const void* in, void* out, int64_t nsamp, int64_t nchan, int64_t npol,
                       int32_t out_kind, int64_t time_sum, int64_t freq_sum, int32_t on_device,
                       int32_t device, void* stream);
/* Incoherent dedispersion (transforms/dedispersion.py:136-177): per-channel integer roll + crop,
 *   out[n, c, :] = in[n + delays[c], c, :],  n < nsamp_out,  0 <= delays[c] <= nsamp_in - nsamp_out
 * for any element type; cell_bytes = bytes per (sample, channel) cell (multiple of 4).  The delays
 * (host array) are computed by the caller exactly as dedispersion.py:164-169. */
int pbk_shift_channels(const void* in, void* out, int64_t nsamp_in, int64_t nsamp_out,
                       int64_t nchan, int64_t cell_bytes, const int64_t* delays,
                       int32_t on_device, int32_t device, void* stream);
int pbk_downsample(const void* in, void* out, int64_t nsamp, int64_t row_elems,
                   int64_t factor, int32_t on_device, int32_t device, void* stream);

/* Incoherent dedispersion at ndm trial DMs summed over frequency: a DM x time plane (builder-defined;
 * trial k is pbk_shift_channels with that trial's delays, summed over channels):
 *   out[k, j, p] = sum_{c < nchan} in[j + delays[k * nchan + c], c, p],  j < rows,
 * in (nsamp_in, nchan, npol) float32, out a contiguous (ndm, rows, npol) float32 array.  Channels
 * are added in ascending order in float32 with no atomics: executions are bit for bit
 * reproducible, and integer-valued data within float32's exact range sum exactly.  The delays
 * (host array [ndm * nchan]) are any non-negative values with delay + rows <= nsamp_in; trials may
 * come in any order and repeat.  pb.incoherent_dedispersion_trials builds them from the reference's
 * rounded delays (dedispersion.py:164-169) and the intersection of every trial's valid rows.
 * The plan sorts the trials by sweep, groups them in blocks of KD <= 8 and uploads its tables once
 * (counted in pbk_plan_info's workspace bytes); one execution is one kernel launch.
 * ndm < 1, nchan < 1, npol < 1, rows < 0, a NULL pointer, a negative delay or delay + rows >
 * nsamp_in return PBK_ERR_INVALID; rows, nsamp_in or nchan above INT32_MAX and npol > 256 return
 * PBK_ERR_UNSUPPORTED.  rows == 0 executes as a no-op.  pbk_plan_describe shows
 * "INCOH:ndm=..:C=..:P=..:rows=.." and the tile (KD, TT rows, CC channels per staged chunk, shared
 * bytes, CTAs); pbk_plan_trials reports ndm, pbk_plan_blocks_per_launch 1, pbk_plan_segments 0:
 * pbk_plan_profile does not time these plans (time them with events around the call).
 * Execution: device pointers need 4-byte alignment (PBK_ERR_INVALID otherwise); _exec_device only
 * enqueues one kernel on `stream` and can be captured into a graph; _exec_host copies in, runs,
 * copies out and synchronises.  The input is never written. */
int pbk_incoh_trials_plan_create(int64_t nsamp_in, int64_t nchan, int64_t npol, int64_t rows,
                                 const int64_t* delays, int32_t ndm, int32_t device,
                                 pbk_plan** plan);
int pbk_incoh_trials_exec_device(pbk_plan* plan, const void* d_in, void* d_out, void* stream);
int pbk_incoh_trials_exec_host(pbk_plan* plan, const void* in, void* out);

/* Fast dispersion measure transform (FDMT; builder-defined, DESIGN.md 5.4h, numpy statement in
 * tests/fdmt_oracle.py): every integer delay trial d in [d_min, max_delay] of a (nsamp, nchan,
 * npol) float32 filterbank with ascending channels over [f_lo_hz, f_hi_hz), in about
 * ceil(log2 nchan) passes.  Trial d sums exactly d + nchan samples per column along a track of
 * d samples of sweep from f_hi to f_lo; out is a contiguous (ndm, rows, npol) float32 array with
 * ndm = max_delay - d_min + 1, and out[k, j, :] is trial d_min + k arriving at ref_freq_hz
 * t_lo + j samples after the input starts (pbk_fdmt_plan_geometry).  Every output is a fixed
 * tree of float32 adds: executions are bit for bit reproducible, integer-valued input sums
 * exactly, and a chunked plan equals an unchunked one.
 * The plan builds the tree and its index tables once in float64 (uploaded, counted in
 * pbk_plan_info's workspace bytes with the two state buffers).  The state is about
 * (max_delay + nchan) * nsamp * npol floats per level; when two levels exceed
 * max_workspace_bytes (0: a fifth of the device's memory) the output rows are split into chunks,
 * each an independent transform of its input slice.  pbk_plan_describe shows
 * "FDMT:C=..:P=..:D=..:levels=..:fused=k:T=..:smem=..:chunks=..:rows=..", where k merges run
 * inside the first kernel (PBK_FDMT_FUSED=k forces it).
 * nsamp, nchan or npol < 1, f_lo_hz <= 0, f_hi_hz <= f_lo_hz, ref_freq_hz <= 0, max_delay < 0,
 * d_min < 0 or > max_delay, and a NULL pointer return PBK_ERR_INVALID; nsamp, nchan, npol or
 * nsamp + max_delay beyond INT32_MAX, state rows beyond 32-bit indices and a workspace cap that
 * holds no chunk return PBK_ERR_UNSUPPORTED.  rows == 0 (nsamp too short for the sweep) is a valid
 * plan whose executions are no-ops, as for pbk_incoh_trials.
 * Execution: device pointers need 4-byte alignment (PBK_ERR_INVALID otherwise); _exec_device only
 * enqueues kernels on `stream` (no synchronisation, no atomics) and can be captured into a graph;
 * _exec_host copies in, runs, copies out and synchronises.  The input is never written. */
int pbk_fdmt_plan_create(int64_t nsamp, int64_t nchan, int64_t npol, double f_lo_hz,
                         double f_hi_hz, double ref_freq_hz, int64_t max_delay, int64_t d_min,
                         int64_t max_workspace_bytes, int32_t device, pbk_plan** plan);
int pbk_fdmt_plan_geometry(const pbk_plan* plan, int32_t* ndm, int64_t* rows, int64_t* t_lo);
int pbk_fdmt_exec_device(pbk_plan* plan, const void* d_in, void* d_out, void* stream);
int pbk_fdmt_exec_host(pbk_plan* plan, const void* in, void* out);

/* Single-pulse search of a stack of time series (builder-defined): x (nser, rows, ncols) float32,
 * C-contiguous, series (s, c) = x[s, :, c] -- e.g. the (ndm, rows, 1[*P]) plane of
 * pbk_incoh_trials_* or the (ndm, rows, nchan[*P]) output of a trial plan.
 *   stats[s, c] = (mean, std) of the series in float64, population std (ddof 0), (nser, ncols, 2)
 *       float64: computed (fixed-order partials per chunk of rows, merged in a fixed order) and
 *       written when stats_given == 0, read when it is 1;
 *   snr(s, c, t, w) = (sum_{i<w} x[s, t+i, c] - w mean) / (std sqrt(w)) for every t with
 *       t + w <= rows, at the widths[0 .. nwidths) (host array, strictly increasing, >= 1, at most
 *       4096 samples); every snr of a series whose std is not > 0 (zero, negative, NaN) is 0;
 *   window j holds the starts [j window, min((j+1) window, rows)), nwin = ceil(rows / window):
 *       snr[s, j, c] (float32), start[s, j, c] and width[s, j, c] (int32), each (nser, nwin, ncols),
 *       are the maximum over the (t, w) of the window, ties to the smallest t, then the smallest w,
 *       compared in float64; a window with no valid (t, w) gets -inf, -1, -1.
 * window = 1 gives the best-S/N plane; window = max(widths) a compact per-window maximum.  No
 * atomics: executions are bit for bit reproducible, and integer-valued data give exact boxcar sums.
 * nser < 1, ncols < 1, rows < 0, nwidths outside 1..32, widths not strictly increasing or < 1,
 * window < 1, a NULL pointer when rows > 0, and device arrays not aligned to their element size
 * (4 bytes, 8 for stats) return PBK_ERR_INVALID; a width above 4096, rows, ncols or nser * ncols
 * above INT32_MAX and grids beyond one launch return PBK_ERR_UNSUPPORTED.  rows == 0 is a no-op.
 * on_device = 1 only enqueues on `stream` (the statistics partials are a stream-ordered
 * allocation); 0 copies in, runs, copies out and synchronises.  The input is never written. */
int pbk_boxcar_search(const void* in, int64_t nser, int64_t rows, int64_t ncols,
                      const int32_t* widths, int32_t nwidths, int64_t window, void* stats,
                      int32_t stats_given, void* snr, void* start, void* width, int32_t on_device,
                      int32_t device, void* stream);

/* Spectral kurtosis RFI flagging (builder-defined; Nita & Gary 2010): in (nsamp, nchan, npol) of
 * in_dtype PBK_C64, PBK_I8X2 or PBK_F32 (detected power, a filterbank), C-contiguous; column
 * (c, p) is one series.  Per block b of the m rows [b m, (b+1) m), nblk = floor(nsamp / m), and
 * per column, with p = re^2 + im^2 (voltages) or p = x (float32), widened to float64:
 *   S1 = sum p, S2 = sum p^2 -- int64 for int8 input (exact), float64 in a fixed order otherwise;
 *   SK = F (m S2 / (S1 S1) - 1) in float64 in exactly this order without contraction,
 *       F = (m nd + 1) / (m - 1), NaN when S1 == 0 (an all-zero block);
 *   sk[b, c, p] = (float)SK, float32 (nblk, nchan, npol);
 *   mask[b, c] = 1 when the SK of any p is not inside [lo, hi] (NaN is flagged), uint8 (nblk, nchan).
 * nd is the number of raw voltage powers summed into each value of in: 1 for voltages, e.g. 2 for
 * Stokes I or downsample * freq_sum for pbk_detect output.  The int8 route is bit for bit the
 * float64 definition; no atomics, so every execution is bit for bit reproducible.
 * out: NULL (estimate only), == in (the m x npol elements of every flagged cell are set to zero in
 * place and nothing else is written), or a separate array of in's type and shape (a copy of in with
 * the flagged cells zeroed; the estimate pass writes the copy as it reads).  The tail rows
 * nblk m .. nsamp - 1 are never estimated, flagged or zeroed; they are copied when out != in.
 * A zero is 0 + 0i, (0, 0) or 0.0f.  sk and mask may each be NULL.
 * u4 / u2 input returns PBK_ERR_UNSUPPORTED: a 2-bit code has no zero, and a u4 zero is code 8,
 * so zeroing would need a decoded output.  m < 2, nd not finite or <= 0, lo or hi NaN, lo > hi,
 * nchan or npol < 1, nsamp < 0, a NULL in when nsamp > 0, all three outputs NULL, another in_dtype,
 * and device arrays not aligned to their element size (8, 2 or 4 bytes for in and out, 4 for sk)
 * return PBK_ERR_INVALID.  Element offsets are 64-bit; nchan * npol above INT32_MAX, and more than
 * INT32_MAX CTAs in either launch (nblk * splits * ceil(nchan npol / 32) or nblk * nchan / 256)
 * return PBK_ERR_UNSUPPORTED.  nblk == 0 estimates nothing and copies in to a separate out.
 * on_device = 1 only enqueues on `stream` (the partial sums are a stream-ordered allocation, the
 * tail a device-to-device copy) and can be captured into a graph; 0 copies in, runs, copies out
 * and synchronises. */
int pbk_spectral_kurtosis(const void* in, void* out, int64_t nsamp, int64_t nchan, int64_t npol,
                          int32_t in_dtype, int64_t m, double nd, double lo, double hi, void* sk,
                          void* mask, int32_t on_device, int32_t device, void* stream);

/* ---- polarisation -------------------------------------------------------------------------
 * pbk_stokes:    (A, B) complex64 pol pairs -> [I, Q, U, V] float32 (core.py:930-966; basis
 *                linear when circular == 0).  npairs = nsamp * nchan.
 * pbk_pol_basis: linear <-> circular basis change (core.py:882-928).
 * pbk_chirp:     the chirp of dedispersion.py:19-23 / 59-75 as an explicit (nsamp, nchan)
 *                complex64 array (DispersionMeasure.chirp_from_signal).
 */
int pbk_stokes(const void* in, void* out, int64_t npairs, int32_t circular, int32_t on_device,
               int32_t device, void* stream);
int pbk_pol_basis(const void* in, void* out, int64_t npairs, int32_t to_circular,
                  int32_t on_device, int32_t device, void* stream);
int pbk_chirp(int64_t nsamp, int64_t nchan, double dm, double sample_rate_hz,
              double ref_freq_hz, const double* chan_freq_hz, void* out, int32_t on_device,
              int32_t device, void* stream);

/* ---- folding (builder-defined, SURVEY 8a row F; phase model = pulsar/predictor.py:149-160) --
 * ph_n = polyval((n0+n)/sample_rate_hz) with numpy's Horner order in FP64 without FMA
 * contraction; bin = floor((ph - floor(ph)) * nbin) mod nbin;
 * profile[bin, j] += in[n, j] (float32 atomics), counts[bin] += 1 (exact).
 * profile (nbin, row_elems) float32 and counts (nbin) int64 are ACCUMULATED into (zero them
 * first); bins_out, if non-NULL, receives the int32 bin of every sample (for bit-exact checks).
 */
int pbk_fold(const void* in, int64_t nsamp, int64_t row_elems, const double* coeffs,
             int32_t ncoef, double sample_rate_hz, int64_t n0, int32_t nbin, void* profile,
             void* counts, void* bins_out, int32_t on_device, int32_t device, void* stream);

/* ---- phase prediction on the device (pulsar/predictor.py:121-147 `PhasePredictor.__call__`
 * for the samples of one polyco entry) --------------------------------------------------------
 * ph = polyval(dt) with numpy's Horner order in FP64 (no FMA contraction), split as
 * pulsar/phase.py:28-78: phase_int = rphase + rint(ph) (int64), phase_frac = ph - rint(ph) (FP64).
 * dt_s: n offsets in seconds from the entry's tmid, or NULL to generate
 * dt = dt0_s + (n0 + i) / sample_rate_hz.  The host mirror picks the entry (searchsorted on the
 * span ends, predictor.py:108-119) and raises the reference's ValueError for times out of range. */
int pbk_phase_predict(const double* dt_s, int64_t n, double dt0_s, double sample_rate_hz,
                      int64_t n0, const double* coeffs, int32_t ncoef, int64_t rphase,
                      void* phase_int, void* phase_frac, int32_t on_device, int32_t device,
                      void* stream);

void pbk_plan_destroy(pbk_plan* plan);

/* plan introspection for benchmarks: number of kernel launches per execution, workspace bytes */
int pbk_plan_info(const pbk_plan* plan, int32_t* launches, int64_t* workspace_bytes,
                  int32_t* levels, int32_t* level_log2 /* [3] */);

/* human-readable list of the passes of a plan: "FWD:L=2^11:fast-r8:W=4:tiles=65536:threads=512;..." */
int pbk_plan_describe(const pbk_plan* plan, char* buf, size_t n);

/* Per-launch device timing for benchmarks.  pbk_plan_profile(plan, nslots) makes every later
 * execution record a CUDA event before each kernel launch and after the last one, on the
 * execution stream, into slot (execution count mod nslots); nslots = 0 switches it off.
 * After synchronising, pbk_plan_profile_read returns the duration in ms of each timed segment of
 * one slot.  A segment is one kernel launch; pbk_plan_segments gives their number and
 * pbk_plan_describe lists them separated by ';' (a trailing time-sum kernel is not listed). */
int pbk_plan_segments(const pbk_plan* plan, int32_t* segments);
int pbk_plan_profile(pbk_plan* plan, int32_t nslots);
int pbk_plan_profile_read(pbk_plan* plan, int32_t slot, float* ms, int32_t n);

/* raw device-memory helpers so a ctypes caller needs no other CUDA binding */
int pbk_malloc(void** dptr, size_t bytes, int32_t device);
int pbk_free(void* dptr, int32_t device);
int pbk_memcpy_h2d(void* dst, const void* src, size_t bytes, int32_t device);
int pbk_memcpy_d2h(void* dst, const void* src, size_t bytes, int32_t device);
/* cudaMemcpyAsync on `stream` (to_device != 0: host -> device, else device -> host); truly
 * asynchronous only for pinned host memory */
int pbk_memcpy_async(void* dst, const void* src, size_t bytes, int32_t to_device, int32_t device,
                     void* stream);
int pbk_device_sync(int32_t device);

#ifdef __cplusplus
}
#endif
#endif /* PBK_H_ */
