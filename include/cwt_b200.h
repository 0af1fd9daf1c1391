/*
 * cwt_b200.h -- C ABI of the B200-native continuous-wavelet-transform engine.
 *
 * Drop-in boundary for the hot path of regeirk/pycwt.  The reference has no FFI
 * layer (it is pure Python); its "interface" for this path is the array math
 * inside pycwt/wavelet.py and pycwt/mothers.py.  Each entry point below names
 * the reference lines it replaces.  A host in any language binds these symbols
 * (ctypes / cffi / cgo / JNI); no torch or C++ types cross the boundary.
 *
 * Conventions
 *   - every function returns 0 on success, a negative cwtb_status otherwise,
 *     and never throws; cwtb_last_error(ctx) gives the message;
 *   - the caller owns every host buffer it passes; device buffers are owned by
 *     the context and addressed through opaque handles or raw device pointers
 *     obtained from cwtb_* accessors;
 *   - a context is bound to one device and one stream; calls on one context
 *     must be serialised by the caller (ctypes releases the GIL, so one context
 *     per host thread / per GPU);
 *   - complex numbers are interleaved (re, im) pairs of double (fp64 engine) or
 *     float (fp32 engine), C order, rows = scales.
 */
#ifndef CWT_B200_H
#define CWT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cwtb_ctx cwtb_ctx;

enum cwtb_status {
  CWTB_OK = 0,
  CWTB_ERR_ARG = -1,       /* bad argument (size, enum, NULL)            */
  CWTB_ERR_CUDA = -2,      /* CUDA runtime error (see cwtb_last_error)   */
  CWTB_ERR_NOMEM = -3,     /* device / pinned allocation failed          */
  CWTB_ERR_STATE = -4,     /* call sequence error (no transform resident) */
  CWTB_ERR_UNSUPPORTED = -5,
  CWTB_ERR_COMM = -6       /* NCCL error / libnccl not loadable           */
};

/* Mother-wavelet families, pycwt/mothers.py:13-233.  MexicanHat == DOG m=2. */
enum cwtb_family {
  CWTB_MORLET = 0,  /* param = f0 (mothers.py:26-28)  */
  CWTB_PAUL = 1,    /* param = m  (mothers.py:118-122) */
  CWTB_DOG = 2,     /* param = m  (mothers.py:170-173) */
  CWTB_TABLE = 3    /* caller supplies psi_ft on the [S, Np] grid (duck-typed wavelets) */
};

enum cwtb_precision { CWTB_F64 = 0, CWTB_F32 = 1 };

/* ---- lifecycle ---------------------------------------------------------- */
int cwtb_device_count(void);
int cwtb_create(int device, cwtb_ctx **out);
void cwtb_destroy(cwtb_ctx *ctx);
const char *cwtb_last_error(cwtb_ctx *ctx);
const char *cwtb_version(void);

/* Relative cut-off below which the analytic frequency response is treated as
 * zero when the per-scale band is pruned (default 1e-16: at the level of the fp64
 * rounding of the transform itself -- parity against the reference fixtures is the
 * same 5e-16 as with 1e-20, profiles/r1/eps_parity_r1.txt).  eps = 0 keeps every bin whose response
 * is representable (the reference's own underflow-to-zero set). */
int cwtb_set_band_eps(cwtb_ctx *ctx, double eps);
/* Tolerance of the band-limited expansion path (replaces the per-scale inverse FFT of
 * pycwt/wavelet.py:105-106 for scales whose band is at most 1/32 of the transform length): such a
 * scale is transformed on a coarse grid of Nc >= 2 * (band width) points and expanded to the
 * output points by a polyphase Kaiser-Bessel interpolation; (Nc, taps) are chosen so that the
 * relative aliasing error bound max sum_l |phi^(xi+l)|/|phi^(xi)| stays <= eps.  Defaults:
 * 5e-13 for the fp64 engine (measured error vs the reference ~1e-13), 2e-7 for the fp32 engine.
 * eps = 0 switches the path off: every scale runs the exact pruned transforms. */
int cwtb_set_expand_eps(cwtb_ctx *ctx, double eps_fp64, double eps_fp32);
/* Transform-length policy of pycwt/helpers.py:7-30.  pad_to_pow2 != 0 (default): the signal is
 * zero-padded to the next power of two (the reference's scipy branch, :27-30).  0: transforms
 * run at the signal's own length (what the reference does when pyfftw is installed, :15-19) --
 * Bluestein's algorithm on the power-of-two kernels, fp64 only, single-channel calls, n0 <= 2^24;
 * the smoothing filter of wct / smooth / wct_mc then is circular at the rows' own length, as in
 * the reference.  Power-of-two lengths are unaffected. */
int cwtb_set_padding(cwtb_ctx *ctx, int pad_to_pow2);
/* Time-smoothing filter of cwtb_smooth / cwtb_wct / cwtb_wct_mc.  Default (table == NULL): the
 * Gaussian exp(-0.5 (s/dt)^2 k^2) of Morlet.smooth (pycwt/mothers.py:83-91).  With a table
 * [n_rows][n] of real frequency responses (n = the transform length of the rows: next power of
 * two, or the rows' own length in un-padded mode) the following calls multiply the transforms of
 * their rows by it instead -- the smoothing operator of wavelets the reference has none for
 * (Paul, DOG: SURVEY 8f rank 4; pycwt_b200.mothers.enable_generic_smoothing).  The table stays in
 * force until replaced or cleared; calls whose rows / length differ fail with CWTB_ERR_STATE. */
int cwtb_set_smooth_filter(cwtb_ctx *ctx, const double *table, int n_rows, int64_t n);

/* Pinned host memory (so D2H of multi-GiB results runs at PCIe speed and can
 * overlap with compute).  numpy wraps the returned pointer. */
int cwtb_host_alloc(cwtb_ctx *ctx, size_t bytes, void **out);
int cwtb_host_free(cwtb_ctx *ctx, void *p);

/* ---- cwt: pycwt/wavelet.py:91-106 (+ :123 trim to n0) -------------------- */
/*
 * Computes, for every scale s_j (j < n_scales),
 *   W[j, n] = ifft_k( fft(signal, Np)[k] * sqrt(s_j*w1*Np) * conj(psi_ft(s_j*w_k)) )[n],
 *   n < n0,  w_k = 2*pi*fftfreq(Np, dt)[k],
 * with Np = next power of two >= n0 (pycwt/helpers.py:27-30).
 *
 * signal      host pointer, n0 reals (double if signal_is_f32 == 0, else float)
 * scales      host pointer, n_scales doubles (resolved by the caller exactly as
 *             wavelet.py:75-88 does)
 * family/param  mother wavelet; for CWTB_TABLE `table` is a host [n_scales, Np]
 *             complex128 array holding sqrt(s*w1*Np)*conj(psi_ft) already
 * precision   arithmetic of the engine (fp64 or fp32)
 * The result stays resident on the device until the next cwtb_cwt* call on
 * this context; fetch it with cwtb_get_* or post-process it with cwtb_icwt...
 */
int cwtb_cwt(cwtb_ctx *ctx, const void *signal, int signal_is_f32, int64_t n0,
             double dt, const double *scales, int n_scales, int family,
             double param, int precision, const void *table);

/* Same, but the signal is already on the device (double or float, n0 reals);
 * used by benchmarks (`value` leg) and by the batched path. */
int cwtb_cwt_dev(cwtb_ctx *ctx, const void *d_signal, int signal_is_f32,
                 int64_t n0, double dt, const double *scales, int n_scales,
                 int family, double param, int precision);

/* Copy W (n_scales x n0, complex of the engine precision, or converted to
 * complex128 when out_f64 != 0) to host memory.  rows [row0, row0+nrows). */
int cwtb_get_w(cwtb_ctx *ctx, void *out, int out_f64, int row0, int nrows);
/* Forward spectrum of the zero-padded signal, bins [1, Np/2), divided by
 * sqrt(Np): the `fft` return value of wavelet.py:123.  Np/2-1 complex128. */
int cwtb_get_signal_fft(cwtb_ctx *ctx, void *out);
int64_t cwtb_padded_length(cwtb_ctx *ctx);
/* Number of transforms this context has started: a handle to a device-resident result stays
 * valid while this value is unchanged. */
int64_t cwtb_job_serial(cwtb_ctx *ctx);
/* Raw device pointer of the resident W (engine precision), for zero-copy
 * consumers (DLPack / __cuda_array_interface__ wrappers). */
void *cwtb_w_device_ptr(cwtb_ctx *ctx);

/* Whole call for host callers: H2D signal, transform, one D2H of W into `out`
 * (page-locked memory from cwtb_host_alloc makes the copy run at PCIe speed; the
 * kernels take ~2 % of the copy time at the north-star size, so there is nothing
 * to overlap).  Equivalent to cwtb_cwt + cwtb_get_w. */
int cwtb_cwt_to_host(cwtb_ctx *ctx, const void *signal, int signal_is_f32,
                     int64_t n0, double dt, const double *scales, int n_scales,
                     int family, double param, int precision, void *out,
                     int out_f64);

/* ---- icwt: pycwt/wavelet.py:169-170 -------------------------------------- */
/* out[n] = sum_j Re(W[j,n]) / sqrt(s_j) for the resident W (the caller applies
 * dj*sqrt(dt)/(cdelta*psi(0))).  out: n0 doubles. */
int cwtb_icwt_sum(cwtb_ctx *ctx, double *out);
/* Same reduction for a caller-supplied host W (n_scales x n complex128). */
int cwtb_icwt_sum_host(cwtb_ctx *ctx, const void *W, const double *scales,
                       int n_scales, int64_t n, double *out);

/* ---- derived products of the resident W (SURVEY 8f rank 2) ---------------- */
/* power[j,n] = |W[j,n]|^2 (doubles, n_scales x n0). */
int cwtb_get_power(cwtb_ctx *ctx, double *out);
/* global wavelet spectrum: mean_n |W[j,n]|^2, n_scales doubles
 * (`power.mean(axis=1)`, pycwt/sample/simple_sample.py:79). */
int cwtb_global_power(cwtb_ctx *ctx, double *out);
/* power[j,n] = row_scale[j] * |W[j,n]|^2; row_scale (one factor per row, NULL = 1) carries the
 * rectification 1/s_j of Liu et al. 2007 (`power /= scales[:, None]`, docs/tutorial/cwt.md:49-53)
 * and/or a variance normalisation. */
int cwtb_get_power_scaled(cwtb_ctx *ctx, const double *row_scale, double *out);
/* mean of |W[j,n]|^2 over the columns lo[j] <= n < hi[j] of every row (NaN for an empty range):
 * the global spectrum restricted to the inside of the cone of influence, whose columns form one
 * centred range per scale. */
int cwtb_global_power_ranges(cwtb_ctx *ctx, const int64_t *lo, const int64_t *hi, double *out);
/* scale-averaged power out[n] = sum_j weights[j] * |W[j,n]|^2, n0 doubles (Torrence & Compo 1998
 * eq. 24; `scale_avg`, pycwt/sample/simple_sample.py:88-91: weights[j] = dj*dt/Cdelta/s_j inside
 * the period band, 0 outside).  Rows with weight 0 are not read. */
int cwtb_scale_avg_power(cwtb_ctx *ctx, const double *weights, double *out);

/* ---- xwt / wct: pycwt/wavelet.py:394-399, 498-514; mothers.py:61-104 ------ */
/* Two signals of equal length -> W12 = W1*conj(W2) (n_scales x n0 complex128). */
int cwtb_xwt(cwtb_ctx *ctx, const double *y1, const double *y2, int64_t n0,
             double dt, const double *scales, int n_scales, int family,
             double param, void *W12_out);
/* Wavelet coherence of two signals (Morlet smoothing operator):
 *   WCT = |S(W12/s)|^2 / (S(|W1|^2/s) * S(|W2|^2/s)),  aWCT = angle(W12),
 * S = Gaussian time filter exp(-0.5*(s/dt)^2*k^2) (FFT, zero-pad to Np) followed
 * by a boxcar of `boxcar_len` taps with half-weight ends along the scale axis
 * (helpers.py:176-191, scipy convolve2d 'same' alignment).
 * WCT_out, aWCT_out: n_scales x n0 doubles (either may be NULL). */
int cwtb_wct(cwtb_ctx *ctx, const double *y1, const double *y2, int64_t n0,
             double dt, double dj, const double *scales, int n_scales, int family,
             double param, int boxcar_len, double *WCT_out, double *aWCT_out);
/* Morlet.smooth on a caller-supplied host array (mothers.py:61-104).
 * in: n_scales x n (complex128 if is_complex else float64); out same type. */
int cwtb_smooth(cwtb_ctx *ctx, const void *in, int is_complex, int n_scales,
                int64_t n, double dt, const double *scales, int boxcar_len,
                void *out);

/* ---- Monte-Carlo coherence significance: pycwt/wavelet.py:609-630 --------- */
/* Accumulates, over `n_pairs` surrogate pairs of length n0, the histogram
 * hist[s, floor(R2*nbins)] += 1 for rows s < maxscale and points with
 * mask[s, n] != 0 (period <= coi).  `noise` is a host array
 * [n_pairs, 2, n0] of doubles drawn by the caller (exact-parity mode: the caller
 * uses numpy's RNG exactly as the reference does).  hist: n_scales x nbins int64,
 * accumulated into (not cleared). */
int cwtb_wct_mc(cwtb_ctx *ctx, const double *noise, int n_pairs, int64_t n0,
                double dt, double dj, const double *scales, int n_scales,
                int family, double param, int boxcar_len, const uint8_t *mask,
                int maxscale, int nbins, int64_t *hist);
/* The same accumulation with the surrogates drawn ON THE DEVICE (SURVEY 8b vi "seed"): pair number
 * first_pair + i is standard-normal white noise from the counter-based Philox4x32-10 stream keyed
 * by (seed, pair number), so a run does not depend on how the pairs are split over calls, ranks
 * or GPUs.  Statistically equivalent to the reference's surrogates (which are white noise too,
 * helpers.py:146-173), not bit-identical to numpy's stream; no host RNG and no H2D of noise. */
int cwtb_wct_mc_seeded(cwtb_ctx *ctx, uint64_t seed, int64_t first_pair, int n_pairs, int64_t n0,
                       double dt, const double *scales, int n_scales, int family, double param,
                       int boxcar_len, const uint8_t *mask, int maxscale, int nbins, int64_t *hist);
/* Test hook: the surrogates of the seeded mode, out[n_pairs][2][n0]. */
int cwtb_mc_surrogates(cwtb_ctx *ctx, uint64_t seed, int64_t first_pair, int n_pairs, int64_t n0,
                       double *out);

/* ---- batched transform of independent channels (SURVEY 8d config 5) ------- */
/* X: host [n_chan, n0] (float or double).  The per-channel transforms stay on
 * the device; `power_out` (may be NULL) receives the per-channel global wavelet
 * spectra [n_chan, n_scales] (doubles); `W_out` (may be NULL) receives all
 * coefficients [n_chan, n_scales, n0] in the engine precision.  The channels are
 * processed in chunks (CWTB_BATCH_MB of coefficients each).  With `power_out` only,
 * the chunks are pipelined: the input copy of chunk k+1 (straight from the caller's
 * array, pageable memory is fine) overlaps the kernels of chunk k, the spectra are
 * accumulated on the device and copied back once; the call returns when
 * `power_out` is complete. */
int cwtb_cwt_batch(cwtb_ctx *ctx, const void *X, int x_is_f32, int n_chan,
                   int64_t n0, double dt, const double *scales, int n_scales,
                   int family, double param, int precision, double *power_out,
                   void *W_out);

/* Batched transform with per-channel products reduced on the device while each chunk of W is
 * resident (W itself never leaves the device).  Arguments as cwtb_cwt_batch, plus:
 *   coi_lo, coi_hi  int64[n_scales], both or neither: columns lo_j <= n < hi_j inside the cone of
 *                   influence (the same for every channel);
 *   n_bands (0..8), band_weights [n_bands][n_scales];  chan_scale [n_chan] (NULL: 1);
 *   icwt_re, icwt_im: the icwt factor dj*sqrt(dt)/(Cdelta*psi(0));  want_icwt: 0 none,
 *                   1 real output, 2 complex output.
 * Outputs (doubles, per channel c; pycwt/sample/simple_sample.py lines each restates):
 *   power_out     [n_chan][n_scales]  mean_n |W|^2                          (glbl_power, :79; required)
 *   power_coi_out [n_chan][n_scales]  mean of |W|^2 over [lo_j, hi_j), NaN if empty (with the ranges)
 *   band_out      [n_chan][n_bands][n0]  chan_scale[c] * sum_j wt[b][j] |W[c,j,n]|^2
 *                                     (scale_avg, :88-91, with wt = dj*dt/Cdelta/s_j in the band)
 *   icwt_out      [n_chan][n0] (want_icwt 1) or [n_chan][n0][2] (want_icwt 2):
 *                 factor * sum_j Re(W[c,j,n]) / sqrt(s_j)                  (iwave, :60)
 * Every coefficient is read once, by one kernel per chunk.  With the default pipeline the column
 * outputs of chunk k are copied to the host while chunk k+1 is transformed; page-locked output
 * arrays (cwtb_host_alloc) make that copy asynchronous.  CWTB_ERR_UNSUPPORTED for CWTB_TABLE and
 * for an un-padded (cwtb_set_padding(0)) length that is not a power of two. */
int cwtb_cwt_batch_products(cwtb_ctx *ctx, const void *X, int x_is_f32, int n_chan,
                            int64_t n0, double dt, const double *scales, int n_scales,
                            int family, double param, int precision,
                            const int64_t *coi_lo, const int64_t *coi_hi,
                            int n_bands, const double *band_weights, const double *chan_scale,
                            double icwt_re, double icwt_im, int want_icwt,
                            double *power_out, double *power_coi_out, double *band_out,
                            double *icwt_out);

/* Device-resident variant: d_X [n_chan][n0] already on the device in the engine's real type;
 * one chunk (n_chan * n_scales rows <= 60000); W [n_chan][n_scales][n0] stays resident
 * (cwtb_w_device_ptr); power_out (may be NULL): host [n_chan][n_scales] mean |W|^2. */
int cwtb_cwt_batch_dev(cwtb_ctx *ctx, const void *d_X, int n_chan, int64_t n0, double dt,
                       const double *scales, int n_scales, int family, double param,
                       int precision, double *power_out);

/* ---- timing / introspection (bench.py, tests) ----------------------------- */
/* Device time (ms, CUDA events on the context's stream) of the kernels of the
 * last cwtb_cwt* / cwtb_xwt / cwtb_wct / cwtb_wct_mc call, excluding H2D/D2H; and the number
 * of kernel launches. */
double cwtb_last_kernel_ms(cwtb_ctx *ctx);
int cwtb_last_launch_count(cwtb_ctx *ctx);
/* Fills `out` (capacity n) with one int per scale of the last call:
 * log2 of the pruned transform length K' (0 if the scale used the direct small-N
 * kernel), or -log2(Nc) if the scale ran on the expansion path with a coarse grid of Nc points.
 * Returns the number written. */
int cwtb_last_plan(cwtb_ctx *ctx, int *out, int n);
/* Re-run the kernels of the last cwtb_cwt_dev call `iters` times and return the
 * mean device time per iteration in ms (events on the launching stream). */
int cwtb_bench_last(cwtb_ctx *ctx, int iters, double *ms_out);
/* One pass of the last cwtb_cwt_dev transform with a CUDA event pair around every kernel
 * launch, on a single stream (the normal run overlaps independent kernel chains on three
 * streams); writes "name|launches|total_ms|rows" lines (rows = scale rows processed) to out. */
int cwtb_profile_last(cwtb_ctx *ctx, char *out, size_t cap);
/* The same table for ANY sequence of calls (xwt, wct, wct_mc, smooth, batches): every kernel
 * launched between begin and end is bracketed by an event pair, on one stream. */
int cwtb_profile_begin(cwtb_ctx *ctx);
int cwtb_profile_end(cwtb_ctx *ctx, char *out, size_t cap);
/* Device memory helpers for benchmarks (inputs resident in HBM). */
int cwtb_dev_alloc(cwtb_ctx *ctx, size_t bytes, void **out);
int cwtb_dev_free(cwtb_ctx *ctx, void *p);
int cwtb_memcpy_h2d(cwtb_ctx *ctx, void *dst, const void *src, size_t bytes);
int cwtb_memcpy_d2h(cwtb_ctx *ctx, void *dst, const void *src, size_t bytes);
int cwtb_sync(cwtb_ctx *ctx);

/* Test hook: plain batched complex DFT of `batch` rows of length n through the engine's own
 * kernels (any n >= 2; lengths other than 2^k go through Bluestein's algorithm, fp64 only);
 * sign = -1 forward, +1 inverse (unnormalised).
 * in/out: host complex128 (precision selects the arithmetic). */
int cwtb_fft_c2c(cwtb_ctx *ctx, const void *in, void *out, int64_t n, int batch,
                 int sign, int precision);

/* ---- multi-GPU (SURVEY.md 8b vii, 8e) ------------------------------------------------------
 * One context per GPU (one process per GPU, or one host thread per context).  The transform
 * itself needs no collective: channels (pycwt.cwt per channel, wavelet.py:13-124), scales and
 * Monte-Carlo surrogate pairs (wavelet.py:609-630) are independent units that the caller
 * block-partitions over the ranks.  These entry points move the REDUCED products over
 * NVLink / NVSwitch with NCCL (bound at run time from libnccl.so.2; CWTB_ERR_COMM if absent):
 * per-channel spectra (all-gather), surrogate histograms (all-reduce), timings (max).
 * Buffers are host arrays, staged through device memory owned by the context.
 *   rank 0:  cwtb_comm_unique_id(id);  the host program hands the 128 bytes to every rank
 *   all:     cwtb_comm_init(ctx, world, rank, id);  ...collectives...;  cwtb_comm_destroy(ctx)
 * world == 1 needs no NCCL: the collectives are copies / no-ops. */
int cwtb_comm_unique_id(void *id128);
int cwtb_comm_init(cwtb_ctx *ctx, int world, int rank, const void *id128);
int cwtb_comm_destroy(cwtb_ctx *ctx);
int cwtb_comm_world(cwtb_ctx *ctx);
int cwtb_comm_rank(cwtb_ctx *ctx);
/* recv[r*bytes .. (r+1)*bytes) = rank r's `send` (bytes per rank, equal on all ranks) */
int cwtb_comm_allgather(cwtb_ctx *ctx, const void *send, void *recv, size_t bytes);
/* in place, every rank gets the result */
int cwtb_comm_allreduce_sum_i64(cwtb_ctx *ctx, int64_t *buf, size_t count);
int cwtb_comm_allreduce_max_f64(cwtb_ctx *ctx, double *buf, size_t count);
int cwtb_comm_broadcast(cwtb_ctx *ctx, void *buf, size_t bytes, int root);

#ifdef __cplusplus
}
#endif
#endif /* CWT_B200_H */
