/*
 * wtb.h -- C ABI of libwavelet_sm100a.so, the B200-native wavelet engine.
 *
 * The reference (o-nate/wavelet-transformer) is pure Python and has no FFI
 * layer; its seam is the `import pycwt as wavelet` / `import pywt` lines of
 * src/cwt.py:19, src/wct.py:14, src/xwt.py:12, src/dwt.py:14, src/modwt.py:14.
 * Each entry point below replaces one library call made through that seam and
 * cites it.  Host side: NumPy -> ctypes (wavelet_transformer_b200/_shim.py).
 *
 * Conventions
 *  - every function returns 0 on success, a negative WTB_E* code on failure;
 *    wtb_last_error() returns a thread-local message for the last failure.
 *  - all arrays are C-contiguous; "real" is float (default) or double (WTB_F64).
 *  - complex planes are interleaved (re, im) pairs of "real".
 *  - the caller owns every buffer; the library keeps no caller pointer past
 *    return.  Without WTB_DEVICE_PTRS buffers are host memory and the call is
 *    synchronous (copies inside).  With WTB_DEVICE_PTRS buffers are device
 *    memory (the call runs on the device that owns them) and the call only enqueues
 *    work on `stream` (a cudaStream_t of that device, NULL = default stream).
 *  - there is no CPU fallback: without a usable sm_100 device calls fail.
 */
#ifndef WTB_H
#define WTB_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define WTB_OK            0
#define WTB_EINVAL       -1   /* bad argument */
#define WTB_ECUDA        -2   /* CUDA runtime error (message has the detail) */
#define WTB_EUNSUPPORTED -3   /* size / mode outside what the kernels cover */
#define WTB_ENODEVICE    -4   /* no CUDA device, or not sm_100 */

#define WTB_F64          (1 << 0)  /* compute and I/O in double precision */
#define WTB_DEVICE_PTRS  (1 << 1)  /* data pointers are device pointers; async on stream */
#define WTB_COI_MASK     (1 << 2)  /* cwt power: write NaN outside the cone of influence */
#define WTB_NOISE_WHITE  (1 << 3)  /* Monte Carlo surrogates: white instead of AR(1) */
#define WTB_GENERIC_ONLY (1 << 4)  /* force the generic (any pow2 N) kernels; testing */
#define WTB_PLANE_COMPLEX (1 << 5) /* wtb_ratio_planes: the input plane is complex (|z|^2 is formed first) */
#define WTB_FFT_NO_PAD   (1 << 6)  /* Monte Carlo: transform the surrogates at their own length (pycwt with
                                      mkl_fft, the reference's conda install) instead of the next power of two */

/* mother wavelets of wtb_cwt / wtb_cwt_axes_mother (pycwt.mothers) */
#define WTB_MORLET 0   /* param = f0 */
#define WTB_PAUL   1   /* param = order m */
#define WTB_DOG    2   /* param = derivative m (m = 2: Mexican hat) */

#define WTB_NBINS 1000             /* pycwt wct_significance: nbins = 1000 */

/* ---- runtime ------------------------------------------------------------ */
int  wtb_version(void);
int  wtb_device_count(void);
/* Which device a call runs on: (1) with WTB_DEVICE_PTRS the device that owns the data pointer;
 * (2) else the device given to wtb_init() (one process per GPU, e.g. under torchrun) or named by
 * the environment variable WTB_DEVICE; (3) else the calling thread's current CUDA device.  The
 * device must be compute capability 10.x.  A call that has to switch devices puts the caller's
 * current device back before it returns. */
int  wtb_init(int device);
/* One process, several GPUs (the reference's call sites are single-process: src/wct.py:106-118).
 * Starts one worker thread and stream per device 0 .. n_gpus-1 (n_gpus <= 0: WTB_GPUS, else all
 * visible devices).  From then on host-buffer calls of wtb_cwt / wtb_cwt_morlet / wtb_xwt_wct and
 * of the filterbank entry points (wtb_modwt .. wtb_waverec) split their batch into contiguous
 * blocks, one per device, and wtb_wct_significance splits its realisations; results do not
 * depend on the number of devices.  WTB_DEVICE_PTRS calls are never
 * split.  wtb_gpu_count() is the number of devices in use (1 without a pool). */
int  wtb_init_multi(int n_gpus);
int  wtb_gpu_count(void);
/* Frees every device buffer the library holds and stops the worker threads.  No call may be in
 * flight.  The library can be used again afterwards. */
void wtb_shutdown(void);
const char *wtb_last_error(void);
/* Number of CUDA kernels this library has launched in this process (bench.py's
 * gpu_launches is the difference across the timed region). */
uint64_t wtb_kernel_launches(void);
/* Bytes of device scratch the library holds right now.  Scratch is keyed by (host thread,
 * device, stream): calls share intermediates only when they are ordered on one stream of one
 * thread, so two WTB_DEVICE_PTRS calls on different streams never touch each other's scratch.
 * It is allocated stream-ordered (no device-wide synchronisation when it grows), released when
 * its host thread exits, and by wtb_shutdown(). */
uint64_t wtb_scratch_bytes(void);

/* ---- CWT: replaces pycwt.cwt (src/cwt.py:110) + |W|^2 (src/cwt.py:114) ---- */
/* Scales, Fourier frequencies and cone of influence exactly as pycwt.cwt
 * forms them.  s0 == -1 and J == -1 select pycwt's defaults; *J_out gets the
 * resolved J (S = J+1 scales).  Any output pointer may be NULL. */
int wtb_cwt_axes(int n0, double dt, double dj, double s0, int J, double f0,
                 int *J_out, double *scales, double *freqs, double *coi);

/* Batched Morlet CWT.  x: [batch, n0] real.  nfft: FFT length >= n0.  pycwt's scipy.fftpack
 * path (the reference's pip / uv install) pads to 2^ceil(log2 n0); its mkl_fft path (the conda
 * install, environment.yml:126) transforms at nfft = n0.  Powers of two run the FFT kernels
 * (fused FP32 fast paths at 512 / 1024 / 2048 / 4096; one CTA per transform up to 8192 in FP32,
 * 4096 in FP64; longer powers of two return WTB_EUNSUPPORTED here and run in wtb_cwt, below); any other
 * length runs Bluestein's chirp-z
 * transform over the next power of two >= 2 nfft - 1 in the generic kernels (nfft <= 2048 in
 * FP64, <= 4096 in FP32).  Outputs (either
 * may be NULL): power_out [batch, S, n0] real = |W|^2; coef_out [batch, S, n0]
 * complex = W.  S = J+1 with scales s0*2^(j*dj).  No normalisation of x. */
int wtb_cwt_morlet(const void *x, int64_t batch, int n0, int nfft,
                   double dt, double dj, double s0, int J, double f0, int flags,
                   void *power_out, void *coef_out, void *stream);

/* The same two calls for any pycwt mother wavelet (constants/results_configs.py:53-58 builds
 * Paul and DOG objects next to Morlet): psi_ft is pi^-1/4 exp(-(sw-f0)^2/2) for Morlet,
 * 2^m/sqrt(m (2m-1)!) (sw)^m exp(-sw) H(sw) for Paul, -i^m/sqrt(Gamma(m+1/2)) (sw)^m exp(-(sw)^2/2)
 * for DOG; flambda = 4pi/(f0+sqrt(2+f0^2)), 4pi/(2m+1), 2pi/sqrt(m+1/2).  Morlet goes through the
 * same code as wtb_cwt_morlet (including its fused FP32 kernel).  wtb_cwt also takes the powers of two
 * past one CTA's shared memory: nfft from 16384 in FP32, 8192 in FP64, up to 2^22 = 4194304, as
 * four-step transforms over several CTAs; larger powers of two return WTB_EUNSUPPORTED. */
int wtb_cwt_axes_mother(int n0, double dt, double dj, double s0, int J, int mother, double param,
                        int *J_out, double *scales, double *freqs, double *coi);
int wtb_cwt(const void *x, int64_t batch, int n0, int nfft, double dt, double dj, double s0, int J,
            int mother, double param, int flags, void *power_out, void *coef_out, void *stream);
/* Inverse transform, replaces pycwt.icwt (Torrence & Compo eq. 11):
 * x_out[b,t] = factor * sum_s Re(W[b,s,t]) / sqrt(scales[s]) with factor =
 * dj sqrt(dt) / (C_delta psi_0(0)) formed by the caller.  coef: [batch, S, n0] complex. */
int wtb_icwt(const void *coef, int64_t batch, int S, int n0, const double *scales, double factor,
             int flags, void *x_out, void *stream);
/* Time- and scale-averaged wavelet power (Torrence & Compo 1998 eqs. 22 and 24; the pycwt sample's
 * glbl_power and scale_avg) of a batch, without the [batch, S, n0] plane leaving the device.
 * Transform arguments and kernel dispatch as wtb_cwt (any mother, FP32/FP64, any nfft wtb_cwt takes).
 * global_out (may be NULL): [batch, S] real, (1/n0) sum_{t<n0} |W[b,s,t]|^2.
 * band_out   (may be NULL): [batch, n0] real, band_factor * sum_{s=band_lo..band_hi} |W[b,s,t]|^2 / scales[s]
 *   (band_factor = dj dt / C_delta formed by the caller, as wtb_icwt's factor; the caller may fold a variance in).
 * Sums are accumulated in double in a fixed order; results do not depend on batch chunking or on
 * the number of devices wherever wtb_cwt's power plane does not.
 * WTB_EINVAL: no output requested, band_out given without 0 <= band_lo <= band_hi < S, band_factor not
 * finite, or WTB_COI_MASK (a masked plane would make every average NaN).  batch == 0 is a no-op. */
int wtb_cwt_averages(const void *x, int64_t batch, int n0, int nfft, double dt, double dj, double s0, int J,
                     int mother, double param, int band_lo, int band_hi, double band_factor, int flags,
                     void *global_out, void *band_out, void *stream);

/* ---- batched pre-processing: replaces standardize_series (src/utils/wavelet_helpers.py:22-57)
 * and pycwt.ar1 (src/cwt.py:106) for batches of series ------------------------------------ */
/* x: [batch, n] real.  y_out (may be NULL): [batch, n] = optional degree-1 detrend or mean
 * removal, then division by the RAW series' population standard deviation.  ar1_out (may be
 * NULL): [batch] lag-1 autocorrelation of the INPUT series (Allen & Smith), NaN where pycwt
 * raises "Cannot place an upperbound on the unbiased AR(1)". */
int wtb_series_prep(const void *x, int64_t batch, int n, int detrend, int remove_mean, int standardize,
                    int flags, void *y_out, double *ar1_out, void *stream);

/* ---- batched post-processing: the NumPy steps the reference runs right after the library calls --- */
/* Ratio planes: src/cwt.py:118-133 (power / signif[:, None]), src/wct.py:120-125 (|coherence| /
 * signif[:, None]) and, with WTB_PLANE_COMPLEX, normalize_xwt_results of
 * src/utils/wavelet_helpers.py:60-78 (power = |W12|^2, then power / signif[:, None]).
 * plane: [batch, S, n0] real, or complex with WTB_PLANE_COMPLEX.  signif: [sig_rows, S] doubles with
 * sig_rows = batch (one threshold row per series) or 1 (shared); a device pointer with
 * WTB_DEVICE_PTRS.  power_out (WTB_PLANE_COMPLEX only, may be NULL) and ratio_out (may be NULL with
 * power_out given): [batch, S, n0] real. */
int wtb_ratio_planes(const void *plane, int64_t batch, int S, int n0, const double *signif, int64_t sig_rows,
                     int flags, void *power_out, void *ratio_out, void *stream);
/* Phase arrows of src/wct.py:143-158 / src/xwt.py:142-154: u = cos(pi/2 - phase), v = sin(pi/2 -
 * phase) for `count` angles; either output may be NULL. */
int wtb_phase_arrows(const void *phase, int64_t count, int flags, void *u_out, void *v_out, void *stream);

/* ---- XWT / WCT: replaces pycwt.xwt (src/xwt.py:93) and pycwt.wct
 * (src/wct.py:106, src/xwt.py:122) minus the host-side normalisation ------- */
/* y1, y2: [batch, n0] real (already normalised by the caller).  Outputs (any
 * may be NULL): wct_out [batch,S,n0] real = |S12|^2/(S1*S2); phase_out
 * [batch,S,n0] real = angle(W1*conj(W2)); w12_out [batch,S,n0] complex.
 * nfft: one CTA per transform up to 8192 in FP32 / 4096 in FP64 (any length up to 4096 / 2048 with
 * WTB_FFT_NO_PAD-style unpadded nfft); longer powers of two, up to 2^22 = 4194304, take four-step
 * transforms over several CTAs (same arithmetic per row); larger nfft returns WTB_EUNSUPPORTED. */
int wtb_xwt_wct(const void *y1, const void *y2, int64_t batch, int n0, int nfft,
                double dt, double dj, double s0, int J, double f0, int flags,
                void *wct_out, void *phase_out, void *w12_out, void *stream);

/* ---- partial and multiple wavelet coherence of three series (Aguiar-Conraria & Soares 2014;
 * Ng & Chan 2012), built from pycwt's Morlet CWT and Morlet.smooth as pycwt.wct builds its spectra -- */
/* y, x1, x2: [batch, n0] real (already normalised by the caller).  With the smoothed spectra
 * S_ij = smooth(W_i conj(W_j) / s) of the three CWTs, outputs (any may be NULL, not all):
 * pwc_out [batch,S,n0] real = |S_y1 S_22 - S_y2 conj(S_12)|^2 / ((S_yy S_22 - |S_y2|^2)(S_11 S_22 - |S_12|^2)),
 * the partial coherence of y and x1 given x2; pphase_out [batch,S,n0] real = angle(S_y1 S_22 - S_y2 conj(S_12));
 * mwc_out [batch,S,n0] real = (|S_y1|^2 S_22 + |S_y2|^2 S_11 - 2 Re(S_y1 conj(S_y2) S_12)) / (S_yy (S_11 S_22 -
 * |S_12|^2)), the multiple coherence of y on x1 and x2.  The ratios are formed in double in both precisions and
 * not clamped (0/0 gives NaN).  Morlet(f0) only; scales as wtb_cwt_axes.  nfft: one CTA per transform, a power
 * of two up to 8192 in FP32 / 4096 in FP64, any other length up to 4096 / 2048; longer ones return
 * WTB_EUNSUPPORTED before any work.  batch == 0 is a no-op. */
int wtb_partial_wct(const void *y, const void *x1, const void *x2, int64_t batch, int n0, int nfft,
                    double dt, double dj, double s0, int J, double f0, int flags,
                    void *pwc_out, void *pphase_out, void *mwc_out, void *stream);

/* ---- Monte Carlo coherence significance: replaces pycwt.wct_significance -- */
/* Surrogate length N = ceil(6*s0*2^(J*dj)/dt) and the largest scale index
 * with any point inside the reliable region (pycwt's `maxscale`). */
int wtb_wct_mc_geometry(double dt, double dj, double s0, int J, double f0,
                        int *nsurr, int *maxscale);

/* Accumulate per-scale coherence histograms of `mc_count` realisations whose
 * GLOBAL indices are mc_first .. mc_first+mc_count-1 (the Philox stream is
 * keyed by the global index, so any partition over GPUs sums to the same
 * histogram).  surrogates: NULL -> AR(1) (or white) noise generated on device
 * from `seed`; else [mc_count, 2, nsurr] real ready-made series (host-injected
 * parity mode).  hist: [S, WTB_NBINS] uint64, ADDED to (caller zeroes).  The surrogates are padded to
 * the next power of two up to 2^22 (nsurr past 8192 in FP32 / 4096 in FP64 takes the four-step rows of
 * wtb_xwt_wct); with WTB_FFT_NO_PAD the one-CTA limits of wtb_xwt_wct apply. */
int wtb_wct_mc_hist(double a1, double a2, double dt, double dj, double s0, int J,
                    double f0, int64_t mc_first, int64_t mc_count, uint64_t seed,
                    const void *surrogates, int flags, uint64_t *hist, void *stream);

/* Percentile step (host arithmetic, tiny): sig95[s] for s < maxscale from the
 * histogram, NaN for the remaining rows that have reliable points. */
int wtb_wct_sig_from_hist(const uint64_t *hist, int S, int maxscale, double level,
                          const uint8_t *row_has_points, double *sig95);

/* The same percentile step with hist [S, WTB_NBINS] and sig95 [S] in DEVICE memory, enqueued on
 * `stream` (bit-identical arithmetic); row_has_points stays a host array. */
int wtb_wct_sig_from_hist_device(const uint64_t *hist, int S, int maxscale, double level,
                                 const uint8_t *row_has_points, double *sig95, void *stream);

/* pycwt.wct_significance in ONE call (src/wct.py:106 reaches it through wct(sig=True)): the
 * realisations 0 .. mc_count-1 are split over the devices of wtb_init_multi (or run on the one
 * current device), each device bins its block, device 0 sums the histograms by reading its peers'
 * memory over NVLink, and the percentile step gives sig95 [J+1].  surrogates: NULL (device Philox
 * AR(1) noise keyed by the global realisation index: the result does not depend on the number of
 * GPUs) or a HOST array [mc_count, 2, nsurr].  hist_out (may be NULL): [J+1, WTB_NBINS] summed
 * histogram.  Host buffers only.  Surrogate lengths as wtb_wct_mc_hist (padded: up to 2^22). */
int wtb_wct_significance(double a1, double a2, double dt, double dj, double s0, int J, double f0,
                         double level, int64_t mc_count, uint64_t seed, const void *surrogates,
                         int flags, double *sig95, uint64_t *hist_out);

/* Device AR(1) surrogates only (for distribution tests): out [count, 2, nsurr]. */
int wtb_rednoise(double a1, double a2, int nsurr, int64_t first, int64_t count,
                 uint64_t seed, int flags, void *out, void *stream);

/* The surrogate triples of wtb_partial_wct_mc_hist: out [count, 3, nsurr], series 0, 1, 2 with coefficients ay, a1,
 * a2 (each its own burn-in).  Series `which` of realisation m draws Philox counter (t >> 2, which, m lo, m hi), so
 * series 0 and 1 of a triple are wtb_rednoise(ay, a1)'s pair. */
int wtb_rednoise_triples(double ay, double a1, double a2, int nsurr, int64_t first, int64_t count,
                         uint64_t seed, int flags, void *out, void *stream);

/* ---- Monte Carlo significance of partial and multiple coherence (Ng & Chan 2012): the recipe of
 * wtb_wct_mc_hist applied to three independent AR(1) series -- */
/* hist: [2, J+1, WTB_NBINS] uint64 (PWC rows, then MWC rows), ADDED to.  surrogates: NULL -> device
 * Philox AR(1) triples (wtb_rednoise_triples), else [mc_count, 3, nsurr] real.  Geometry (nsurr, maxscale) as
 * wtb_wct_mc_geometry; rows s < maxscale, columns inside the reliable region, bins as wtb_wct_mc_hist (NaN and
 * negative values skipped).  Flags: WTB_F64, WTB_DEVICE_PTRS (hist and surrogates in device memory),
 * WTB_NOISE_WHITE, WTB_FFT_NO_PAD (surrogates transformed at their own length, else padded to a power of two),
 * WTB_GENERIC_ONLY.  One CTA per transform only: nfft up to 8192 in FP32 / 4096 in FP64 padded (series of about
 * 1365 / 680 samples with s0 = 2 dt), any other length up to 4096 / 2048; longer ones, |a| >= 1, NaN coefficients
 * and J < 0 are refused before any copy or launch.  mc_count == 0 is a no-op. */
int wtb_partial_wct_mc_hist(double ay, double a1, double a2, double dt, double dj, double s0, int J, double f0,
                            int64_t mc_first, int64_t mc_count, uint64_t seed, const void *surrogates,
                            int flags, uint64_t *hist, void *stream);
/* One call over the pool (realisations 0 .. mc_count-1 split by global index; the result does not depend on the
 * number of GPUs): sig_pwc, sig_mwc [J+1] (NaN / 0 rows as wtb_wct_sig_from_hist); hist_out may be NULL.  Host
 * buffers only; limits and refusals as wtb_partial_wct_mc_hist. */
int wtb_partial_wct_significance(double ay, double a1, double a2, double dt, double dj, double s0, int J,
                                 double f0, double level, int64_t mc_count, uint64_t seed,
                                 const void *surrogates, int flags, double *sig_pwc, double *sig_mwc,
                                 uint64_t *hist_out);

/* ---- MODWT: replaces src/modwt.py:126 modwt, :147 imodwt, :163 modwtmra --- */
/* Every filterbank entry point below (wtb_modwt .. wtb_waverec) takes any n.
 * One CTA holds a series in shared memory while its buffers fit 227 KB: up to
 * n = 14484 in FP64 / 29004 in FP32 for wtb_modwt, 9656 / 19336 for wtb_imodwt,
 * 14524 / 29052 for wtb_modwtmra, wtb_modwtmra_taps and wtb_wavedec, about
 * 14520 / 29050 output samples for wtb_waverec.  Longer series run level by
 * level, one launch per level, with their intermediates in device scratch (the
 * long path, which WTB_GENERIC_ONLY does not change).  The choice is made from
 * the shape.
 * g = dec_lo, h = dec_hi (pywt.Wavelet taps, length L, NOT yet divided by
 * sqrt 2).  x: [batch, n]; w: [batch, J+1, n] rows w_1..w_J, v_J. */
int wtb_modwt(const void *x, int64_t batch, int n, const double *g, const double *h,
              int L, int J, int flags, void *w_out, void *stream);
int wtb_imodwt(const void *w, int64_t batch, int n, const double *g, const double *h,
               int L, int J, int flags, void *x_out, void *stream);
/* filt: [J+1, n] periodised equivalent filters (host-built, see
 * modwt.py:56-83); out[b,j,t] = sum_l filt[j,l] * w[b,j,(t+l) mod n]. */
int wtb_modwtmra(const void *w, int64_t batch, int n, const double *filt, int J,
                 int flags, void *out, void *stream);
/* Same details D_1..D_J and smooth S_J from the taps alone (modwt.py:163-194):
 * each row runs the synthesis cascade G_1'..G_{j-1}' H_j' w_j, which equals the
 * correlation with the periodised equivalent filter.  Shapes the cascade
 * kernel does not cover (L not in {2,4,6,8}, dilated filter longer than n)
 * are served by building those filters on the host and correlating, up to
 * the one-CTA length; longer rows run the cascade one level per launch for
 * every row at once, without building the filters.  wtb_modwtmra past that
 * length correlates over each row's non-zero taps only. */
int wtb_modwtmra_taps(const void *w, int64_t batch, int n, const double *g,
                      const double *h, int L, int J, int flags, void *out,
                      void *stream);

/* ---- MODWT wavelet variance, covariance and cross-correlation by level (Percival & Walden 2000, ch. 8;
 * Whitcher, Guttorp & Percival 2000): the time_scale_regression companion, reduced on the device --------- */
/* The MODWT is wtb_modwt's (same kernels, same bits): W_j[t] = sum_l h~_l V_{j-1}[(t - 2^(j-1) l) mod n] with
 * h~ = h / sqrt 2, g~ = g / sqrt 2.  For a filter of length L, L_j = (2^j - 1)(L - 1) + 1; W_j[t] is free of
 * the circular wrap exactly for t >= L_j - 1, and M_j = n - L_j + 1 coefficients are.  For j = 1..J (the
 * scaling row V_J is not included):
 *   var_x_out [batch, J]          nu2_X(j) = (1/M_j) sum_{t=L_j-1}^{n-1} W_{X,j}[t]^2 (var_y_out likewise for y)
 *   xcov_out  [batch, J, 2K+1]    gamma_XY(j, tau) = (1/M_j) sum_t W_{X,j}[t] W_{Y,j}[t+tau], lags tau = -K..K,
 *                                 over the t with t and t+tau in [L_j-1, n-1]; divisor M_j at every lag
 *                                 (biased); lag 0 is the wavelet covariance.
 * NaN where M_j <= 0 and for |tau| >= M_j, never an error.  Outputs are double in both precisions (host or
 * device memory per WTB_DEVICE_PTRS); sums run in double in a fixed order that depends on n, L and j only, so
 * results are bit-identical across batch, chunking, pool size and host vs device pointers.  y == NULL is the
 * variance of x alone (var_y_out and xcov_out must then be NULL; var_x_out has the pair call's bits).
 * K = max_lag.  WTB_EINVAL: no output requested, J outside [1, 30], max_lag outside [0, 8192] or >= n; L outside
 * [2, 32]: WTB_EUNSUPPORTED.  Refusals come before any copy or launch; batch == 0 is a no-op.  Flags: WTB_F64,
 * WTB_DEVICE_PTRS, WTB_GENERIC_ONLY (the MODWT's generic kernels). */
int wtb_modwt_wavelet_stats(const void *x, const void *y, int64_t batch, int n, const double *g,
                            const double *h, int L, int J, int max_lag, int flags,
                            double *var_x_out, double *var_y_out, double *xcov_out, void *stream);

/* ---- DWT: replaces pywt.wavedec / pywt.waverec (src/dwt.py:104,71,120) ---- */
/* lens: [level+1] lengths of cA_L, cD_L, ..., cD_1 for symmetric mode. */
int wtb_dwt_coeff_lens(int n, int L, int level, int *lens);
int wtb_dwt_max_level(int n, int L);
/* coeffs: [batch, sum(lens)] packed in pywt order cA_L | cD_L | ... | cD_1. */
int wtb_wavedec(const void *x, int64_t batch, int n, const double *dec_lo,
                const double *dec_hi, int L, int level, int flags, void *coeffs,
                void *stream);
/* lens as produced by wtb_dwt_coeff_lens (or any consistent pywt-style list);
 * x_out: [batch, n_out] with n_out = wtb_waverec_len(lens, level, L). */
int wtb_waverec_len(const int *lens, int level, int L);
int wtb_waverec(const void *coeffs, int64_t batch, const int *lens, int level,
                const double *rec_lo, const double *rec_hi, int L, int flags,
                void *x_out, void *stream);

/* ---- per-component regressions: replaces sm.OLS(output_j, add_constant(input_j)).fit()
 * (src/regression.py:76-81,118-121, src/modwt.py:218-222) ------------------------------ */
/* One simple regression y = a + b x per row.  x: [x_rows, n], y: [y_rows, n]; the row counts
 * are equal, or one of them is 1 and that row is used for every regression (the reference's
 * wavelet_approximation regresses ONE series on each smooth).  add_constant = 0 fits y = b x.
 * stats_out: [rows, 8] doubles { nobs, intercept, slope, ssr, tss, sxx, mean_x, mean_y } with
 * tss / sxx centred when add_constant (statsmodels' centered_tss), raw sums otherwise.
 * Standard errors, t and p values follow on the host (api/regression.py). */
int wtb_rowwise_ols(const void *x, int64_t x_rows, const void *y, int64_t y_rows, int n,
                    int add_constant, int flags, double *stats_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* WTB_H */
