// qi_stx.cu -- Stockwell transform on the shared FFT core.
//
// One forward FFT per record (n = 2^m, no padding: the reference's product is circular), then per band
// the first inverse pass gathers the spectrum shifted by the band's bin index, multiplies by the Gaussian
// window exp(-0.5*sigma^2*w_k^2) synthesised on the fly, and the last inverse pass fuses |.|^2 / band sums.
// Reference: quantum_inferno/styx_stx.py:213-234 and :166-190.
#include "qi_fft.cuh"
#include "qi_host.h"
#include "qi_tfr.cuh"
#include "qi_interp.cuh"

#include <vector>

namespace qi {

// q = sigma*2*pi/n; |k| > kmax: the window underflows to 0; |k| > dec_kmax: below the cut of the band-limited route
struct DevStxBand { double q; long long shift; long long kmax; long long dec_kmax; };

template <typename T> struct SrcStxSpec {
    const cplx<T>* spec; const DevStxBand* bands; int band0; CwtGeom geo;
    QI_DEV cplx<T> load(i64 batch, i64 e) const {
        const i64 chan = batch % geo.n_channels;
        const DevStxBand b = bands[band0 + (int)(batch / geo.n_channels)];
        const i64 n = 1ll << geo.logL;
        const i64 k = (i64)brev_bits((unsigned)e, geo.logL);
        const i64 ks = (k < (n >> 1)) ? k : k - n;                 // signed bin (fftfreq ordering)
        // beyond kmax exp() returns exactly 0 in T: same product, without the gather and the exponential
        if (ks > b.kmax || -ks > b.kmax) return mk<T>((T)0, (T)0);
        const i64 ksrc = (k + b.shift) & (n - 1);
        const cplx<T> X = spec[(chan << geo.logL) + (i64)brev_bits((unsigned)ksrc, geo.logL)];
        const T u = (T)b.q * (T)ks;
        const T w = exp((T)-0.5 * u * u) * (T)(1.0 / (double)n);
        return X * w;
    }
};

// Band-limited route (both dtypes, and every decimated band of method="multirate").  A Stockwell voice is a BASEBAND signal: X[k + shift] exp(-0.5 (q k)^2) is below exp(-0.5 U^2) of its peak
// beyond |k| > kmax = U / q.  The K = 2^m >= RHO (2 kmax + 4) bins around zero, inverse-transformed at length K, are the
// voice at every D = n / K-th sample exactly; qi_interp.cuh brings it to the full rate (no carrier to put back).
template <typename T> struct SrcStxDecT {
    const cplx<T>* spec; const DevStxBand* bands; const int* ids; int n_channels, logN, logK;
    QI_DEV cplx<T> load(i64 batch, i64 e) const {
        const i64 chan = batch % n_channels;
        const DevStxBand b = bands[ids[batch / n_channels]];
        const i64 K = 1ll << logK, n = 1ll << logN;
        const i64 k = (i64)brev_bits((unsigned)e, logK);
        const i64 ks = (k < (K >> 1)) ? k : k - K;
        if (ks > b.dec_kmax || -ks > b.dec_kmax) return mk<T>((T)0, (T)0);
        const i64 ksrc = (ks + b.shift) & (n - 1);
        const cplx<T> X = spec[(chan << logN) + (i64)brev_bits((unsigned)ksrc, logN)];
        const T u = (T)b.q * (T)ks;
        return X * (exp((T)-0.5 * u * u) * (T)(1.0 / (double)n));
    }
};

template <typename T>
__global__ void stx_windows_kernel(const DevStxBand* bands, i64 n, cplx<T>* out) {
    const i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const DevStxBand b = bands[blockIdx.y];
    const i64 ks = (k < (n >> 1)) ? k : k - n;
    const T u = (T)b.q * (T)ks;
    out[(i64)blockIdx.y * n + k] = mk<T>(exp((T)-0.5 * u * u), (T)0);
}

// ---------------------------------------------------------------- overlap-save route of the widest voices
// A voice whose window is WIDE in frequency is SHORT in time: voice(t) = exp(-2 pi i shift t / n) * (x (*) h)(t) with
// h(t) = g_sigma(t) exp(+2 pi i shift t / n), g_sigma the (periodised) Gaussian of std sigma samples, (*) the circular
// convolution of the reference's spectral product (styx_stx.py:233-236).  For sigma <= ~60 samples that is an
// overlap-save convolution in 2048-sample blocks read circularly from the record: one forward transform per block, per
// band a real response exp(-0.5 (q u)^2) / F at u = j n / F - shift (an integer: the block grid is a subset of the
// record's) + one inverse transform in shared memory, the carrier taken out on the way to HBM.  Replaces two full-length
// HBM passes per voice (a third of a Stockwell call at 16 x 2^18).  Truncating h at U_CUT sigma costs exp(-U_CUT^2 / 2)
// (1.5e-7 float32, 1.3e-13 float64) of the peak, like the band-limited route.
template <typename T> struct OsStxRoute {
    const DevStxBand* bands;
    struct Band {
        DevStxBand b;
        QI_DEV cplx<T> weigh(cplx<T> x, int r, const CwtGeom& geo) const {
            const i64 N = geo.n_points;                                  // 2^logL
            const i64 j = (i64)brev_bits((unsigned)r, CWTF_OS_LOGF);    // block bin j <-> record bin j << (logL - logF)
            i64 u = ((j << (geo.logL - CWTF_OS_LOGF)) - b.shift) & (N - 1);
            if (u >= (N >> 1)) u -= N;                                  // signed distance from the voice's centre bin
            T w = (T)0;
            if (u <= b.kmax && -u <= b.kmax) {
                const T a = (T)b.q * (T)u;
                w = exp((T)-0.5 * a * a) * (T)(1.0 / (double)(1 << CWTF_OS_LOGF));
            }
            return x * w;
        }
        QI_DEV cplx<T> out(cplx<T> y, i64 n, const CwtGeom& geo) const {   // * exp(-2 pi i shift n / N), exact phase
            const unsigned long long m = ((unsigned long long)b.shift * (unsigned long long)n) & (unsigned long long)(geo.n_points - 1);
            return mul_conj(y, unit_root<T>(m, geo.logL));
        }
    };
    QI_DEV T sample(const T* xs, i64 k, i64 N) const { return xs[k & (N - 1)]; }   // circular, like the reference's product
    QI_DEV Band band(int, int band) const { return Band{bands[band]}; }
};

struct StxLayout { int logL; i64 L; size_t off_bands, off_spec, off_work, off_ids, off_coef, total; int group; };

template <typename T> static StxLayout stx_layout(i64 C, i64 N, int B, int group) {
    StxLayout lo;
    lo.logL = ceil_log2_i64(N);
    lo.L = 1ll << lo.logL;
    if (group < 1) group = 1;
    if (group > B) group = B;
    while ((i64)group * C > 65535 && group > 1) --group;
    lo.group = group;
    size_t o = 0;
    lo.off_bands = o; o = align_up(o + sizeof(DevStxBand) * (size_t)B, 256);
    lo.off_spec = o; o = align_up(o + sizeof(cplx<T>) * (size_t)C * lo.L, 256);
    lo.off_work = o; o = align_up(o + sizeof(cplx<T>) * (size_t)group * C * lo.L, 256);
    lo.off_ids = o; o = align_up(o + sizeof(int) * (size_t)B, 256);
    lo.off_coef = o; o = align_up(o + sizeof(T) * CwtFastCfg<T>::TAPS * (size_t)(CWTF_MAX_LOGD + 1) * (1u << CWTF_MAX_LOGD), 256);
    lo.total = o;
    return lo;
}

// u_zero: |u| from which exp(-0.5 u^2) is exactly 0 in the arithmetic type (below the smallest subnormal, with margin:
// float32 exp(-104) = 6.8e-46 < 2^-150; float64 exp(-746) < 2^-1075)
static void upload_stx_bands(const QiStxBand* hb, int B, i64 N, double u_zero, DevStxBand* d_bands, cudaStream_t st,
                             double u_cut = 0.0) {
    std::vector<DevStxBand> db(B);
    for (int b = 0; b < B; ++b) {
        db[b].q = hb[b].sigma * 2.0 * M_PI / (double)N;
        db[b].shift = ((hb[b].shift % N) + N) % N;
        const double aq = fabs(db[b].q);
        const double km = aq > 0.0 ? ceil(u_zero / aq) + 2.0 : (double)N;
        db[b].kmax = km < (double)N ? (long long)km : (long long)N;
        const double kd = (aq > 0.0 && u_cut > 0.0) ? ceil(u_cut / aq) + 1.0 : (double)N;
        db[b].dec_kmax = kd < (double)N ? (long long)kd : (long long)N;
    }
    stage_to_device(d_bands, db.data(), sizeof(DevStxBand) * (size_t)B, st);
}

static CwtGeom stx_geom(i64 C, i64 N, int B, int logL) {
    CwtGeom geo;
    geo.n_points = N; geo.n_channels = C; geo.n_bands = B; geo.logL = logL;
    geo.conv_mode = QI_CONV_LINEAR_SAME; geo.fs = 0; geo.centre_idx = 0; geo.half_shift = 0; geo.d_min = 0; geo.d_max = 0;
    return geo;
}

// full-length passes over maximal runs of at most `group` consecutive bands b with logK[b] == logL
template <typename T>
static void stx_full_length(const FftPlan& plan, const std::vector<int>& logK, int group, const cplx<T>* spec,
                            const DevStxBand* d_bands, cplx<T>* work, const CwtGeom& geo, void* out_c, void* out_p,
                            double* band_sum, cudaStream_t st) {
    const int B = (int)logK.size();
    for (int band0 = 0; band0 < B;) {
        if (logK[band0] != geo.logL) { ++band0; continue; }
        int g = 1;
        while (band0 + g < B && g < group && logK[band0 + g] == geo.logL) ++g;
        inverse_passes<T>(plan, (i64)g * geo.n_channels, SrcStxSpec<T>{spec, d_bands, band0, geo},
                          DstCwtOut<T>{static_cast<cplx<T>*>(out_c), static_cast<T*>(out_p), band_sum, band0, geo, 0.0}, 256,
                          true, work, geo.n_points, st);
        band0 += g;
    }
}

template <typename T>
static int stx_fft_impl(const void* sig, i64 C, i64 N, i64 stride, const QiStxBand* hb, int B, void* out_c,
                        void* out_p, double* band_sum, void* ws, size_t ws_bytes, int group, cudaStream_t st, bool fast) {
    typedef CwtFastCfg<T> Cfg;
    const StxLayout lo = stx_layout<T>(C, N, B, group);
    if (ws_bytes < lo.total) return QI_ERR_WORKSPACE;
    if (C > 65535) return QI_ERR_UNSUPPORTED;
    unsigned char* base = static_cast<unsigned char*>(ws);
    DevStxBand* d_bands = reinterpret_cast<DevStxBand*>(base + lo.off_bands);
    cplx<T>* spec = reinterpret_cast<cplx<T>*>(base + lo.off_spec);
    cplx<T>* work = reinterpret_cast<cplx<T>*>(base + lo.off_work);
    int* d_ids = reinterpret_cast<int*>(base + lo.off_ids);
    upload_stx_bands(hb, B, N, sizeof(T) == 4 ? 14.5 : 38.7, d_bands, st, Cfg::U_CUT);
    const CwtGeom geo = stx_geom(C, N, B, lo.logL);
    const FftPlan plan = make_plan(lo.logL, (int)sizeof(cplx<T>));
    prof_set_category(QI_CAT_FFT_FWD);
    forward_passes<T>(plan, C, SrcRealPad<T>{static_cast<const T*>(sig), stride, N}, spec, lo.L, st);
    if (band_sum) cudaMemsetAsync(band_sum, 0, sizeof(double) * (size_t)C * B, st);
    // ---- band-limited route: bands whose window fits K <= n / 4 bins, grouped by K
    std::vector<int> logK(B, lo.logL);
    int n_dec = 0;
    if (fast && lo.logL >= 13) {
        for (int b = 0; b < B; ++b) {
            const double aq = fabs(hb[b].sigma * 2.0 * M_PI / (double)N);
            if (!(aq > 0.0)) continue;
            logK[b] = dec_logk(ceil(Cfg::U_CUT / aq) + 1.0, Cfg::RHO, 4.0, lo.logL, false);
            if (logK[b] < lo.logL) ++n_dec;
        }
    }
    T* coef = reinterpret_cast<T*>(base + lo.off_coef);
    const auto dec_src = [&](const int* ids, int lk) { return SrcStxDecT<T>{spec, d_bands, ids, (int)C, lo.logL, lk}; };
    const int rc = decimated_route<T, false, true, 2>(logK, geo, dec_src, nullptr, 0, d_ids, coef, work, work,
                                                      (size_t)lo.group * C * lo.L, out_c, out_p, band_sum, st);
    if (rc != QI_OK) return rc;
    // ---- overlap-save route: voices that are too wide to decimate and short in time
    if (fast && lo.logL >= 13) {
        std::vector<int> os_ids;
        int os_half = 0;
        for (int b = 0; b < B; ++b) {
            if (logK[b] != lo.logL) continue;
            const double sg = fabs(hb[b].sigma);
            const int half = (int)ceil(Cfg::U_CUT * sg) + 2;
            // sigma >= 2.5: the window has decayed (exp(-30)) where the signed bin index wraps, so the response on the block
            // grid is the reference's window
            if (sg >= 2.5 && half <= CWTF_OS_MAX_HALF) { os_ids.push_back(b); if (half > os_half) os_half = half; }
        }
        if (!os_ids.empty()) {
            int* d_os = d_ids + n_dec;
            stage_to_device(d_os, os_ids.data(), sizeof(int) * os_ids.size(), st);
            for (int b : os_ids) logK[b] = -1;                          // taken: the full-length passes skip them
            overlap_save_route<T>(sig, stride, geo, d_os, (int)os_ids.size(), (os_half + 15) & ~15, OsStxRoute<T>{d_bands},
                                  out_c, out_p, band_sum, st);
        }
    }
    // ---- full-length passes: the bands that took no other route
    stx_full_length<T>(plan, logK, lo.group, spec, d_bands, work, geo, out_c, out_p, band_sum, st);
    prof_set_category(QI_CAT_OTHER);
    return check_cuda("qi_stx_fft");
}


// ---------------------------------------------------------------- multirate (float32) Stockwell
// The exact path's pieces under another plan: every band whose voice fits K <= n / 2 bins at a 5.5-sigma cut (2.7e-7 of
// its peak; K = 2^m >= 4 kmax + 4, i.e. the decimated samples 2x oversampled) takes the decimated route, the rest the
// full-length passes; no overlap-save route and no band sums.  numpy model and error budget:
// tools/stx_multirate_prototype.py; measured against the full-length transform: relative L2 3e-6, max 6e-6.
constexpr double STXMR_U = 5.5;

struct StxMrLayout { size_t off_bands, off_ids, off_spec, off_work, off_dec, off_coef, total, dec_elems; i64 gx; };

static StxMrLayout stxmr_layout(i64 C, i64 N, const QiStxBand* hb, int B, std::vector<int>& logK) {
    StxMrLayout lo;
    const int logN = ceil_log2_i64(N);
    size_t dec_elems = 0;
    int count[64] = {0};
    logK.resize(B);
    for (int b = 0; b < B; ++b) {
        logK[b] = dec_logk(ceil(STXMR_U / fabs(hb[b].sigma * 2.0 * M_PI / (double)N)) + 1.0, 2.0, 2.0, logN, true);
        ++count[logK[b]];
    }
    for (int lk = 0; lk < logN; ++lk) {
        const size_t e = (size_t)count[lk] * (size_t)C << lk;
        dec_elems = e > dec_elems ? e : dec_elems;
    }
    i64 gx = (i64)((1ull << 30) / ((size_t)C * (size_t)N * sizeof(cplx<float>)));   // exact bands per launch: <= 1 GiB of scratch
    if (gx < 1) gx = 1;
    if (gx > count[logN]) gx = count[logN] > 0 ? count[logN] : 1;
    while (gx * C > 65535 && gx > 1) --gx;
    lo.gx = gx;
    lo.dec_elems = dec_elems;
    const size_t work_elems = dec_elems > (size_t)gx * C * N ? dec_elems : (size_t)gx * C * N;
    size_t o = 0;
    lo.off_bands = o; o = align_up(o + sizeof(DevStxBand) * (size_t)B, 256);
    lo.off_ids = o; o = align_up(o + sizeof(int) * (size_t)B, 256);
    lo.off_spec = o; o = align_up(o + sizeof(cplx<float>) * (size_t)C * N, 256);
    lo.off_work = o; o = align_up(o + sizeof(cplx<float>) * work_elems, 256);
    lo.off_dec = o; o = align_up(o + sizeof(cplx<float>) * (dec_elems ? dec_elems : 1), 256);
    lo.off_coef = o; o = align_up(o + sizeof(float) * CwtFastCfg<float>::TAPS * (size_t)(CWTF_MAX_LOGD + 1) * (1u << CWTF_MAX_LOGD), 256);
    lo.total = o;
    return lo;
}

static int stx_multirate_impl(const void* sig, i64 C, i64 N, i64 stride, const QiStxBand* hb, int B, void* out_c, void* out_p,
                              void* ws, size_t ws_bytes, cudaStream_t st) {
    typedef float T;
    const int logN = ceil_log2_i64(N);
    std::vector<int> logK;
    const StxMrLayout lo = stxmr_layout(C, N, hb, B, logK);
    if (ws_bytes < lo.total) return QI_ERR_WORKSPACE;
    unsigned char* base = static_cast<unsigned char*>(ws);
    DevStxBand* d_bands = reinterpret_cast<DevStxBand*>(base + lo.off_bands);
    cplx<T>* spec = reinterpret_cast<cplx<T>*>(base + lo.off_spec);
    cplx<T>* work = reinterpret_cast<cplx<T>*>(base + lo.off_work);
    cplx<T>* dec = reinterpret_cast<cplx<T>*>(base + lo.off_dec);
    int* d_ids = reinterpret_cast<int*>(base + lo.off_ids);
    T* coef = reinterpret_cast<T*>(base + lo.off_coef);
    // decimated bands are cut at 5.5 sigma (dec_kmax), the full-length ones at the float32 underflow point (kmax)
    upload_stx_bands(hb, B, N, 14.5, d_bands, st, STXMR_U);
    const CwtGeom geo = stx_geom(C, N, B, logN);
    const FftPlan plan = make_plan(logN, (int)sizeof(cplx<T>));
    prof_set_category(QI_CAT_FFT_FWD);
    forward_passes<T>(plan, C, SrcRealPad<T>{static_cast<const T*>(sig), stride, N}, spec, N, st);
    const auto dec_src = [&](const int* ids, int lk) { return SrcStxDecT<T>{spec, d_bands, ids, (int)C, logN, lk}; };
    const int rc = decimated_route<T, false, false, 1>(logK, geo, dec_src, nullptr, 0, d_ids, coef, work, dec, lo.dec_elems,
                                                       out_c, out_p, nullptr, st);
    if (rc != QI_OK) return rc;
    // bands too wide to decimate: runs of consecutive band indices, at most gx per launch
    stx_full_length<T>(plan, logK, (int)lo.gx, spec, d_bands, work, geo, out_c, out_p, nullptr, st);
    prof_set_category(QI_CAT_OTHER);
    return check_cuda("qi_stx_multirate");
}

template <typename T>
static int stx_windows_impl(const QiStxBand* hb, int B, i64 N, void* out, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (ws_bytes < sizeof(DevStxBand) * (size_t)B) return QI_ERR_WORKSPACE;
    DevStxBand* d_bands = static_cast<DevStxBand*>(ws);
    upload_stx_bands(hb, B, N, 1e300, d_bands, st);
    dim3 grid((unsigned)((N + 255) / 256), (unsigned)B);
    QI_LAUNCH((stx_windows_kernel<T>), grid, dim3(256), 0, st, d_bands, N, static_cast<cplx<T>*>(out));
    return check_cuda("qi_stx_windows");
}

}  // namespace qi

extern "C" {

size_t qi_stx_workspace_bytes(int64_t C, int64_t N, int B, int group, int dtype) {
    if (C <= 0 || N <= 0 || B <= 0) return 0;
    if (group < 0) group = -group;
    return dtype == QI_F32 ? qi::stx_layout<float>(C, N, B, group).total : qi::stx_layout<double>(C, N, B, group).total;
}

int qi_stx_fft(const void* sig, int64_t C, int64_t N, int64_t stride, const QiStxBand* bands, int B, int dtype,
               void* out_tfr, void* out_power, double* band_sum, void* ws, size_t ws_bytes, int group, void* stream) {
    if (!sig || !bands || !ws || C <= 0 || N <= 0 || B <= 0 || stride < N) return QI_ERR_ARG;
    if (N & (N - 1)) return QI_ERR_ARG;
    if (N > (1ll << 30)) return QI_ERR_UNSUPPORTED;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool fast = group >= 0;                  // a negative bands_per_group keeps every band on the full-length passes
    if (group < 0) group = -group;
    if (dtype == QI_F32) return qi::stx_fft_impl<float>(sig, C, N, stride, bands, B, out_tfr, out_power, band_sum, ws, ws_bytes, group, st, fast);
    if (dtype == QI_F64) return qi::stx_fft_impl<double>(sig, C, N, stride, bands, B, out_tfr, out_power, band_sum, ws, ws_bytes, group, st, fast);
    return QI_ERR_ARG;
}

size_t qi_stx_multirate_workspace_bytes(int64_t C, int64_t N, const QiStxBand* bands, int B) {
    if (C <= 0 || N < 2 * qi::CWTF_TILE || (N & (N - 1)) || B <= 0 || !bands) return 0;
    std::vector<int> logK;
    return qi::stxmr_layout(C, N, bands, B, logK).total;
}

int qi_stx_multirate(const void* sig, int64_t C, int64_t N, int64_t stride, const QiStxBand* bands, int B, void* out_tfr,
                     void* out_power, void* ws, size_t ws_bytes, void* stream) {
    if (!sig || !bands || !ws || C <= 0 || C > 65535 || N <= 0 || B <= 0 || stride < N || (!out_tfr && !out_power)) return QI_ERR_ARG;
    if ((N & (N - 1)) || N < 2 * qi::CWTF_TILE) return QI_ERR_ARG;
    if (N > (1ll << 30)) return QI_ERR_UNSUPPORTED;
    return qi::stx_multirate_impl(sig, C, N, stride, bands, B, out_tfr, out_power, ws, ws_bytes, static_cast<cudaStream_t>(stream));
}

size_t qi_stx_windows_workspace_bytes(int B) { return B > 0 ? sizeof(qi::DevStxBand) * (size_t)B : 0; }

int qi_stx_windows(const QiStxBand* bands, int B, int64_t N, int dtype, void* out, void* ws, size_t ws_bytes, void* stream) {
    if (!bands || !out || !ws || B <= 0 || N <= 0) return QI_ERR_ARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (dtype == QI_F32) return qi::stx_windows_impl<float>(bands, B, N, out, ws, ws_bytes, st);
    if (dtype == QI_F64) return qi::stx_windows_impl<double>(bands, B, N, out, ws, ws_bytes, st);
    return QI_ERR_ARG;
}

}  // extern "C"
