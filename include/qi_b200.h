/* qi_b200.h -- C ABI of libqi_b200.so: the B200 (sm_100a) kernels behind the quantum-inferno
 * time-frequency hot path.
 *
 * The reference (ISLA-UH/quantum-inferno v1.1.3) has no FFI layer: its boundary is the
 * module-level Python API.  Each entry point below names the reference function whose
 * arithmetic it replaces (file:line relative to the reference checkout); the Python modules
 * in quantum_inferno_b200/ keep the reference's names and signatures and call these through
 * ctypes.  All pointers except those marked HOST are device pointers (HBM); no entry point
 * allocates; all work is enqueued on `stream` (a cudaStream_t passed as void*); every call
 * returns 0 on success or a negative QI_ERR_* code and never throws.
 */
#ifndef QI_B200_H
#define QI_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QI_ABI_VERSION 5

/* dtype of the arithmetic and of every real/complex buffer in a call */
#define QI_F32 0
#define QI_F64 1

#define QI_OK 0
#define QI_ERR_ARG (-1)       /* bad size / pointer / dtype                     -> ValueError   */
#define QI_ERR_WORKSPACE (-2) /* workspace too small                            -> ValueError   */
#define QI_ERR_CUDA (-3)      /* a CUDA runtime error was raised                -> RuntimeError */
#define QI_ERR_UNSUPPORTED (-4)

int qi_abi_version(void);
const char* qi_error_string(int code);
/* text of the last CUDA error seen by this thread (empty string if none) */
const char* qi_last_cuda_error(void);

/* ---- launch accounting / live timing (used by bench.py) ---------------------------------------
 * qi_launch_count: kernels this library has launched in this process so far.
 * qi_profile_enable(1) makes every launch be bracketed by CUDA events on its own stream, grouped by
 * category; qi_profile_read synchronises those events and returns per-category totals, then clears them. */
#define QI_CAT_FFT_FWD 0      /* forward FFT passes (record / atom spectra)            */
#define QI_CAT_INV_FIRST 1    /* first inverse pass: spectrum x band response          */
#define QI_CAT_INV_MID 2      /* middle inverse pass                                   */
#define QI_CAT_INV_LAST 3     /* last inverse pass: slice + |.|^2 + band sums          */
#define QI_CAT_INFO 4         /* tfr_info planes / reductions                          */
#define QI_CAT_STFT 5
#define QI_CAT_OTHER 6
#define QI_N_CATEGORIES 7
int64_t qi_launch_count(void);
int qi_profile_enable(int on);
int qi_profile_read(double* total_ms /*[QI_N_CATEGORIES]*/, int64_t* launches /*[QI_N_CATEGORIES]*/);

/* ---- plain batched FFT (building block; also used by tfr_info.ShannonFFT, tfr_info.py:177) ----
 * in : complex [batch, 2^log2n] natural order
 * out: forward -> spectrum in BIT-REVERSED order (position p holds bin bitrev(p));
 *      inverse -> takes bit-reversed order, returns natural order scaled by 1/n.
 * in == out is allowed. */
int qi_fft_c2c(const void* in, void* out, int64_t batch, int log2n, int inverse, int dtype, void* stream);

/* ---- Gabor-atom CWT by FFT convolution -------------------------------------------------------
 * Replaces quantum_inferno/styx_cwt.py:147-198 (cwt_complex_any_scale_pow2: wavelet_centered_4cwt
 * :113-144 + scipy.signal.fftconvolve :195) and quantum_inferno/cwt_atoms.py:343-444
 * (cwt_chirp_complex, "fft" :406-421 and "conv" :423-435 branches).
 *
 * One band = one atom  a(x) = amp * exp(-(p_re + i p_im) x^2) * exp(i omega x),
 * x = fs*(m/fs - ((n_points-1)/fs)/2), m = 0..n_points-1 (the reference's own rounding of the
 * centred time axis, styx_cwt.py:65,132,135 / cwt_atoms.py:227-236).
 *   analytic = 1 : the atom's frequency response is synthesised on the fly inside the inverse-FFT
 *                  kernel (requires p_im == 0 and a Gaussian that has decayed at the record edge);
 *   analytic = 0 : the truncated time-domain atom is transformed once (shared by all channels)
 *                  and multiplied from HBM -- exact for any atom.
 */
typedef struct {
    double omega;
    double p_re;
    double p_im;
    double amp;
    int32_t analytic;
    int32_t reserved;
} QiAtomBand;

/* conv_mode */
#define QI_CONV_LINEAR_SAME 0   /* out = fftconvolve(sig, conj(atom)[::-1], 'same')  (styx_cwt.py:195, cwt_atoms.py:435) */
#define QI_CONV_CIRC_CORR 1     /* out = roll(ifft(fft(sig)*conj(fft(atom))), -n/2)  (cwt_atoms.py:406-421); n = 2^m */
/* OR-ed into conv_mode: every band takes the plain route (three full-length passes).  By default the Gaussian atoms
 * that have decayed inside the record take band-limited routes with the same result to the accuracy of the arithmetic
 * type (csrc/qi_cwt_fast.cuh): short atoms an overlap-save convolution in shared memory, long atoms a short inverse
 * transform of their baseband bins + Kaiser-windowed-sinc interpolation. */
#define QI_CONV_PLAIN_ONLY 0x100

size_t qi_cwt_workspace_bytes(int64_t n_channels, int64_t n_points, int n_bands, int n_table_bands,
                              int bands_per_group, int conv_mode, int dtype);

/* sig        : real [n_channels, n_points] rows `sig_stride` elements apart
 * bands      : HOST array of n_bands descriptors
 * out_cwt    : complex [n_channels, n_bands, n_points] or NULL
 * out_power  : real    [n_channels, n_bands, n_points] (|cwt|^2) or NULL
 * band_sum   : double  [n_channels, n_bands] (sum over time of |cwt|^2, fp64 accumulation) or NULL
 * workspace  : >= qi_cwt_workspace_bytes(...) bytes, 256-byte aligned */
int qi_cwt_fft(const void* sig, int64_t n_channels, int64_t n_points, int64_t sig_stride,
               const QiAtomBand* bands, int n_bands, double fs, int conv_mode, int dtype,
               void* out_cwt, void* out_power, double* band_sum,
               void* workspace, size_t workspace_bytes, int bands_per_group, void* stream);

/* Time-domain atoms themselves (styx_cwt.py:68-144 wavelet_complex / wavelet_centered_4cwt,
 * cwt_atoms.py:16-50 chirp_complex): out complex [n_bands, n_points].  xtime: optional device fp64
 * [n_points] array of non-dimensional times x; NULL = the centred axis defined above. */
int qi_atoms_time(const QiAtomBand* bands, int n_bands, int64_t n_points, double fs, int dtype,
                  const double* xtime, void* out_atoms, void* workspace, size_t workspace_bytes, void* stream);

/* ---- multirate fp32 Gabor CWT (fast path) ------------------------------------------------------
 * Same quantity as qi_cwt_fft(QI_CONV_LINEAR_SAME) for Gaussian (p_im = 0) atoms, float32 only, to the
 * north-star fp32 tolerance (power relative L2 <= 1e-4): half-band decimation pyramid of the record, each band
 * convolved (overlap-save FFT in shared memory) at the deepest level whose alias-free band holds its response,
 * then half-band interpolation back to the full rate fused with |.|^2 and the fp64 band sums.  The atoms the
 * reference truncates at the record (n_points / scale < 10) are reproduced with that truncation: its jump is carried by
 * exact running sums of the record, so every band meets the tolerance on its own (measured 1e-5 .. 3e-5).
 * Replaces quantum_inferno/styx_cwt.py:147-198 followed by np.abs(cwt)**2.
 * bands: HOST array sorted by ascending centre frequency; level = log2 of the decimation the host planner chose
 * (non-increasing along the array, 0 <= level <= log2(n_points) - 10).  n_points = 2^m, m >= 13. */
typedef struct {
    double omega;    /* centre, rad/sample at the full rate */
    double scale;    /* atom scale s in samples             */
    double amp;
    int32_t level;
    int32_t reserved;
} QiMrBand;

size_t qi_cwt_multirate_workspace_bytes(int64_t n_channels, int64_t n_points, const QiMrBand* bands, int n_bands);

/* sig float [C, sig_stride]: 16-byte aligned, sig_stride a multiple of 4 samples (the record is read with 128-bit
 * loads); a record that starts elsewhere, such as a slice x[k:] of a device buffer, is QI_ERR_ARG, so copy it first.
 * out_power float [C,B,N] or NULL; out_cwt complex64 [C,B,N] or NULL; band_sum double [C,B] (exact sums of the
 * stored power) or NULL; out_power, out_cwt and out_info 32-byte aligned.
 *
 * Fused information / entropy (replaces tfr_info.py:231-236 on top of the CWT, one pass over the planes):
 * pass out_info float [C,B,N]; then out_power, band_sum, band_sum_est [C,B] and total_power [C] are required and
 * entropy_sum double [C,B] (sum_t pdf*info per band) is optional.  info = -log2(P/S + eps) with S = total_power[c].
 * S must be known before the planes are written, so it is first estimated from the decimated band outputs
 * (relative error ~1e-6, see qi_mr_expand.cuh); `phase` lets a band-sharded caller all-reduce it in between:
 *   QI_MR_PHASE_ALL      everything; total_power is written, then used
 *   QI_MR_PHASE_ESTIMATE up to band_sum_est [C,B] (and total_power = its row sums); nothing expanded yet
 *   QI_MR_PHASE_EXPAND   expand with the total_power the caller provides (same workspace, untouched in between) */
#define QI_MR_PHASE_ALL 0
#define QI_MR_PHASE_ESTIMATE 1
#define QI_MR_PHASE_EXPAND 2
int qi_cwt_multirate(const void* sig, int64_t n_channels, int64_t n_points, int64_t sig_stride,
                     const QiMrBand* bands, int n_bands, void* out_power, void* out_cwt, double* band_sum,
                     void* out_info, double* entropy_sum, double* band_sum_est, double* total_power, double eps,
                     int phase, void* workspace, size_t workspace_bytes, void* stream);

/* ---- Stockwell transform ----------------------------------------------------------------------
 * Replaces quantum_inferno/styx_stx.py:195-236 (stx_complex_any_scale_pow2) and the band loop of
 * :52-192 (tfr_stx_fft :166-190):  tfr[b,:] = ifft( X[(k + shift_b) mod n] * exp(-0.5*sigma_b^2*w_k^2) ),
 * w_k = 2*pi*fftfreq(n)[k].  n_points must be a power of two.  shift_b (the argmin of :233) and sigma_b
 * are computed on the host in float64 exactly as the reference does. */
typedef struct {
    double sigma;
    int64_t shift;
} QiStxBand;

size_t qi_stx_workspace_bytes(int64_t n_channels, int64_t n_points, int n_bands, int bands_per_group, int dtype);

/* out_tfr complex [C,B,N] or NULL; out_power real [C,B,N] or NULL; band_sum double [C,B] or NULL.
 * Records of 2^13 samples or more: a voice whose Gaussian window fits K <= n / 4 bins is inverse-transformed at length K
 * and interpolated to the full rate (Kaiser-windowed sinc; float64 24 taps / -231 dB, float32 16 taps / -110 dB), the
 * others take full-length passes.  A NEGATIVE bands_per_group keeps every band on the full-length passes (|value| bands
 * per launch): the arbiter the band-limited route is tested against. */
int qi_stx_fft(const void* sig, int64_t n_channels, int64_t n_points, int64_t sig_stride,
               const QiStxBand* bands, int n_bands, int dtype,
               void* out_tfr, void* out_power, double* band_sum,
               void* workspace, size_t workspace_bytes, int bands_per_group, void* stream);

/* Multirate float32 Stockwell (same quantity as qi_stx_fft to the north-star float32 tolerance: relative L2 <= 1e-4;
 * measured 3e-6).  Every voice is a baseband signal of bandwidth ~ 5.5 / (sigma 2 pi / n) bins: it is computed at the
 * 2x-oversampled decimated rate by a short inverse transform and brought to the full rate by a 16-tap polyphase
 * interpolator (circular, like the reference's product); bands too wide to decimate keep the exact passes.
 * n_points = 2^m >= 4096.  out_tfr complex64 [C,B,N] or NULL; out_power float [C,B,N] or NULL. */
size_t qi_stx_multirate_workspace_bytes(int64_t n_channels, int64_t n_points, const QiStxBand* bands, int n_bands);
int qi_stx_multirate(const void* sig, int64_t n_channels, int64_t n_points, int64_t sig_stride, const QiStxBand* bands,
                     int n_bands, void* out_tfr, void* out_power, void* workspace, size_t workspace_bytes, void* stream);

/* windows_fft of tfr_stx_fft (styx_stx.py:179): out complex [n_bands, n_points], natural bin order */
size_t qi_stx_windows_workspace_bytes(int n_bands);
int qi_stx_windows(const QiStxBand* bands, int n_bands, int64_t n_points, int dtype, void* out,
                   void* workspace, size_t workspace_bytes, void* stream);

/* ---- STFT / Welch -----------------------------------------------------------------------------
 * Replaces scipy.signal.stft / welch as called by quantum_inferno/styx_fft.py:175-187 (stft_complex_pow2),
 * :215-227 (gtx_complex_pow2), :254-266 (welch_power_pow2).  Frame f covers extended-record samples
 * [f*hop - pad_left, f*hop - pad_left + nperseg) with zeros outside [0, n_points); each frame has its mean
 * removed (detrend != 0), is multiplied by window[nperseg] (device pointer), zero-padded to nfft = 2^m,
 * transformed, and the one-sided bins multiplied by `scale`.
 *   out     : complex [n_channels, nfft/2+1, n_frames] (time fastest, scipy's layout) or NULL
 *   psd_acc : double  [n_channels, nfft/2+1] receives sum over frames of |X_k|^2 (unscaled) or NULL
 *   roll    : the windowed, zero-padded segment is rotated left by `roll` samples before the transform, i.e. bin k is
 *             multiplied by exp(+2*pi*i*k*roll/nfft) (scipy.signal.ShortTimeFFT phase_shift, used through
 *             quantum_inferno/utilities/short_time_fft.py:54-58); 0 for scipy.signal.stft
 * A frame is transformed in one CTA's shared memory up to nfft = 8192 (float32) / 4096 (float64) and needs no
 * workspace (NULL, 0).  Longer frames take multi-pass FFTs of frame pairs through the workspace, in as many chunks as it
 * takes: any workspace of at least one frame pair per channel (qi_stft_workspace_bytes with n_frames = 2) works, a
 * smaller one is QI_ERR_WORKSPACE and NULL is QI_ERR_UNSUPPORTED.  The complex outputs do not depend on the chunk size,
 * psd_acc only up to the order of its fp64 additions.
 *   workspace: 256-byte aligned, or NULL */
int qi_stft(const void* sig, int64_t n_channels, int64_t n_points, int64_t sig_stride, const void* window,
            int nperseg, int hop, int nfft, int64_t n_frames, int pad_left, double scale, int detrend, int roll,
            int dtype, void* out, double* psd_acc, void* workspace, size_t workspace_bytes, void* stream);

/* Workspace of qi_stft that transforms all frames in one chunk: 0 for every nfft one CTA takes; otherwise
 * n_channels * ceil(n_frames / 2) * (nfft complex values + 2 reals). */
size_t qi_stft_workspace_bytes(int64_t n_channels, int64_t n_frames, int nfft, int dtype);

/* Inverse STFT by overlap-add (scipy.signal.ShortTimeFFT.istft as called by
 * quantum_inferno/utilities/short_time_fft.py:106-134).
 *   S        : complex [n_channels, nfft/2+1, n_frames] (time fastest), one-sided spectra made with the same `roll`
 *   dual_win : real [nperseg] device pointer (canonical dual window; any scaling folded in)
 *   frame p covers output samples [first_start + p*hop, ... + nperseg); frames [frame_lo, frame_hi) are summed
 *   out      : real [n_channels, n_out] = samples k0 .. k0 + n_out - 1
 *   workspace: >= qi_istft_workspace_bytes, 256-byte aligned */
int qi_istft(const void* S, int64_t n_channels, int64_t n_frames, const void* dual_win, int nperseg, int hop, int nfft,
             int roll, int64_t first_start, int64_t frame_lo, int64_t frame_hi, int64_t k0, int64_t n_out, int dtype,
             void* out, void* workspace, size_t workspace_bytes, void* stream);

/* Workspace of qi_istft: the windowed inverse transforms of all frames, n_channels * n_frames * nperseg reals, for the
 * frame lengths one CTA transforms (nfft <= 8192 float32 / 4096 float64); for longer frames those rounded up to 256
 * bytes plus the pair spectra of up to 65535 frame pairs (multi-pass inverse FFTs). */
size_t qi_istft_workspace_bytes(int64_t n_channels, int64_t n_frames, int nperseg, int nfft, int dtype);

/* ---- power / information / entropy (tfr_info) -------------------------------------------------
 * `power` is real [M, F, T] (M independent matrices: channels).  All reductions accumulate in fp64. */

/* Replaces np.sum(axis=1), np.sum(axis=0), np.sum(), np.max() of quantum_inferno/tfr_info.py:236,247,259,79.
 * row_sum [M,F], col_sum [M,T], total [M], max_value [M]; any of them may be NULL. */
int qi_power_reduce(const void* power, int64_t M, int64_t F, int64_t T, int dtype,
                    double* row_sum, double* col_sum, double* total, double* max_value, void* stream);

/* Replaces ShannonStft.__init__ (tfr_info.py:219-228) for the pdf of
 *   mode 0: P / norm[m]              shannon_stft_from_tfr_power   :231-236   (norm = total,   D = F*T)
 *   mode 1: (1/norm[m,t] + eps) * P  ShannonStftPerTime            :239-248   (norm = col_sum, D = F)
 *   mode 2: (1/norm[m,f] + eps) * P  ShannonStftPerFreq            :251-260   (norm = row_sum, D = T)
 *   mode 3: P                        Shannon (1-D marginal, EPS32) :97-135    (D = T, F = 1)
 * Outputs (each may be NULL): pdf, info = -log2(pdf+eps), bits = pdf*info, isnr = log2(D)-info,
 * esnr = bits/(log2(D)/D); entropy_sum [M,F] = row sums of bits (fp64). */
int qi_shannon(const void* power, int64_t M, int64_t F, int64_t T, int dtype, int mode, const double* norm,
               double eps, double deg_free, void* out_pdf, void* out_info, void* out_bits, void* out_isnr,
               void* out_esnr, double* entropy_sum, void* stream);

/* Replaces scale_power_bits (tfr_info.py:73-79): out = log2(P+eps) - log2(max_value[m]+eps); per_mat = F*T */
int qi_power_bits(const void* power, int64_t M, int64_t per_mat, int dtype, const double* max_value, double eps,
                  void* out, void* stream);

/* Replaces ShannonTDR.__init__ (tfr_info.py:147-151): sumsq[m] = sum x^2, out_sig = x/sqrt(sumsq) (or NULL),
 * out_marginal = out_sig^2 */
int qi_tdr_marginal(const void* sig, int64_t M, int64_t n, int64_t sig_stride, int dtype, double* sumsq,
                    void* out_sig, void* out_marginal, void* stream);

/* Elementwise on n values of a real (is_complex=0), complex (is_complex=1) or signed-real (is_complex=2: no
 * modulus, log2(x + eps) as in tfr_info.py:65-70) buffer:
 * square=0: out = log2(|x| + eps)  (quantum_inferno/utilities/rescaling.py:13-20 to_log2_with_epsilon, used at
 *           cwt_atoms.py:442 and styx_fft.py:55);  square=1: out = |x|^2 + eps (styx_stx.py:188-190);
 *           square=2: out = |x| + eps (np.abs of utilities/short_time_fft.py:95).  out is real. */
int qi_abs_log2(const void* in, int64_t n, int dtype, int is_complex, int square, double eps, void* out, void* stream);

/* Replaces scipy.fft.rfft in ShannonFFT.__init__ (tfr_info.py:177): real [M, n=2^m] -> complex [M, n/2+1]
 * in natural bin order.  workspace >= M*n complex elements. */
int qi_rfft(const void* sig, int64_t M, int64_t n, int64_t sig_stride, int dtype, void* out,
            void* workspace, size_t workspace_bytes, void* stream);

/* ---- after the path: display / picking summaries (SURVEY 8(f) rank 3) --------------------------
 * Replaces quantum_inferno/utilities/sampling.py:13-50 (subsample) and :87-120 (subsample_2d): every row of
 * in [M, n_in] (rows `stride` elements apart) is cut into groups of `factor` consecutive samples;
 *   NTH     : out[m, j] = in[m, j*factor],                 n_out = ceil(n_in / factor)
 *   others  : out[m, j] = mean / median / max / min of in[m, j*factor .. (j+1)*factor), n_out = floor(n_in / factor)
 * (the remainder is dropped, as the reference truncates it).  NaNs propagate like numpy's.  The mean accumulates in
 * fp64 (float32 records on the 128-bit path: the four samples of one load are first added in float32); median / max /
 * min return input values (or the dtype's mean of the two middle ones) bit-exactly. */
#define QI_SUB_NTH 0
#define QI_SUB_AVERAGE 1
#define QI_SUB_MEDIAN 2
#define QI_SUB_MAX 3
#define QI_SUB_MIN 4
int qi_subsample(const void* in, int64_t M, int64_t n_in, int64_t stride, int64_t factor, int method, int dtype,
                 void* out, int64_t n_out, void* stream);

/* Replaces np.nanmax / np.nanmin / np.nanmax(np.abs()) / np.max of quantum_inferno/utilities/picker.py:34-53,141-144:
 * out double [M, 4] = (max, min, max |x|, number of NaNs) of every row, NaNs ignored (all-NaN row -> NaN). */
int qi_extrema(const void* in, int64_t M, int64_t n, int64_t stride, int dtype, double* out, void* stream);

/* Replaces the scan of scipy.signal.find_peaks(x, height=h) called at quantum_inferno/utilities/picker.py:105,119,147:
 * plateau-aware strict local maxima (scipy _local_maxima_1d: midpoint of a flat top, edges excluded) that satisfy
 * x[peak] >= height when use_height != 0.  peaks int64 [capacity] receives the positions UNORDERED and values
 * double [capacity] (or NULL) x at those positions; *count (device) the number found, which may exceed capacity
 * (then only `capacity` were stored: call again with more room). */
int qi_local_maxima(const void* in, int64_t n, int dtype, double height, int use_height, int64_t* peaks,
                    double* values, int64_t capacity, int64_t* count, void* stream);

/* HOST function (no device work): the minimum-distance selection of scipy.signal.find_peaks(distance=)
 * (scipy/signal/_peak_finding_utils.pyx::_select_by_peak_distance) on the short candidate list that
 * qi_local_maxima returned.  peaks HOST int64 [n] ascending; order HOST int64 [n] = argsort of the priorities
 * (ascending; the highest priority is visited first); keep HOST uint8 [n] out: 1 = kept.  A kept peak removes every
 * neighbour nearer than `distance` samples. */
int qi_select_peaks_by_distance(const int64_t* peaks, const int64_t* order, int64_t n, int64_t distance, uint8_t* keep);

/* Replaces `in_signal / np.nanmax(in_signal)` etc. of quantum_inferno/utilities/picker.py:46-53: out = in / divisor,
 * the divisor rounded to the buffer's dtype first (numpy's array / same-dtype scalar). */
int qi_divide(const void* in, int64_t n, int dtype, double divisor, void* out, void* stream);

/* ---- before the path: zero-phase IIR filtering (SURVEY 8(f) rank 4) ----------------------------
 * Replaces scipy.signal.filtfilt(b, a, x) as called by quantum_inferno/styx_fft.py:60-149 (butter_bandpass /
 * butter_highpass / butter_lowpass) and quantum_inferno/synth/synthetic_signals.py:180-192 (antialias_half_nyquist),
 * and scipy.signal.sosfiltfilt(sos, x) as called by quantum_inferno/utilities/picker.py:56-76 (apply_bandpass):
 * odd extension by `padlen` samples, forward recursion from zi * ext[0], recursion over the reversed result from
 * zi * y[-1], middle n samples kept (scipy's method="pad", padtype="odd").  The recursions run as a blocked parallel
 * scan in fp64 whatever the record dtype.
 *   form QI_IIR_BA : n_coef = number of taps (b and a zero-padded to the same length, a[0] == 1), direct form II
 *                    transposed as scipy's lfilter; zi = scipy.signal.lfilter_zi(b, a)        [n_coef - 1 values]
 *   form QI_IIR_SOS: n_coef = number of second-order sections, sos[s] = (b0, b1, b2, 1, a1, a2) as scipy's sosfilt;
 *                    zi = scipy.signal.sosfilt_zi(sos) flattened                              [2 * n_coef values]
 *   tukey_alpha >= 0: the record is first multiplied by scipy.signal.windows.tukey(n, tukey_alpha) (styx_fft.py:88-89)
 *   sig / out: real [M, n] of `dtype` (out rows are n apart); n > padlen (else QI_ERR_ARG, scipy raises ValueError). */
#define QI_IIR_BA 0
#define QI_IIR_SOS 1
#define QI_IIR_MAX_STATE 16
typedef struct {
    int32_t form;
    int32_t n_coef;
    double b[QI_IIR_MAX_STATE + 1];
    double a[QI_IIR_MAX_STATE + 1];
    double sos[QI_IIR_MAX_STATE / 2][6];
    double zi[QI_IIR_MAX_STATE];
} QiIirFilter;
size_t qi_filtfilt_workspace_bytes(int64_t M, int64_t n, int padlen, int n_state);
int qi_filtfilt(const void* sig, int64_t M, int64_t n, int64_t stride, const QiIirFilter* filter /*HOST*/, int padlen,
                double tukey_alpha, int dtype, void* out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- device-side synthetic inputs (SURVEY 8(f) rank 2) -----------------------------------------
 * Replaces the array expressions of quantum_inferno/synth/benchmark_signals.py:92-101 (quantum_chirp) and :323-335
 * (well_tempered_tone).  For k = 0..n-1 (every one of the M rows gets the same waveform):
 *   time = (k + k0) - t_center;  u = time / chirp_scale;  phase = omega * time + half_gamma * u^2
 *   out_re = A cos(phase), out_im = A sin(phase) (or NULL), A = exp(-0.5 u^2) if gauss else 1
 * float64 arithmetic in the reference's order; outputs real [M, n] of `dtype`, rows `stride` apart. */
int qi_synth_chirp(int64_t M, int64_t n, int64_t stride, int64_t k0, double t_center, double omega, double half_gamma,
                   double chirp_scale, int gauss, int dtype, void* out_re, void* out_im, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* QI_B200_H */
