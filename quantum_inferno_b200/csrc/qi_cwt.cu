// qi_cwt.cu -- Gabor / chirp atom CWT by FFT convolution (exact path).
//
//   forward : one batched FFT per record (real signal zero-extended to L >= 2N-1), spectrum kept in
//             bit-reversed order in HBM.
//   per band: first inverse pass reads the record spectrum, multiplies by the band response --
//             synthesised ON THE FLY from (omega, scale) for Gaussian atoms that have decayed at the
//             record edge, or read from a table made by transforming the truncated time-domain atom
//             once for all channels -- and the last inverse pass fuses the 'same' slice, |.|^2 and the
//             fp64 per-band power sum into its store.
//
// Reference arithmetic replaced: quantum_inferno/styx_cwt.py:101-107 (atoms), :195-196 (fftconvolve),
// quantum_inferno/cwt_atoms.py:406-435.
#include "qi_fft.cuh"
#include "qi_host.h"
#include "qi_reduce.cuh"
#include "qi_tfr.cuh"

#include <vector>
#include <math.h>

namespace qi {

struct DevBand {
    double gain;        // analytic: amp*sqrt(pi/p_re)/L ; table: 1/L
    double g;           // analytic: u = g*(k - kappa + j*L), g = (2*pi/L)/sqrt(2*p_re)
    double kappa_frac;
    long long kappa_int;
    long long table_off;   // element offset into the table buffer, -1 = analytic
    // time-domain atom (table bands)
    double omega, p_re, p_im, amp;
    // decimated route (qi_cwt_fast.cuh): nearest bin of the band centre, bins kept either side of it
    long long kc, dec_kmax;
};

// ---------------------------------------------------------------- on-the-fly Gabor response
template <typename T>
QI_DEV bool gabor_response_negligible(const DevBand& b, i64 k, int logL) {
    // distance (in bins) to the nearest alias of the band centre; beyond ~9.5 sigma (fp32: 6.3) the response is
    // below 3e-20 (2e-9) of its peak and the whole product is skipped -- spectrum load, exps and twiddle included
    const T Lf = (T)(1ll << logL);
    T dk = (T)(k - b.kappa_int) - (T)b.kappa_frac;
    dk -= Lf * rint(dk / Lf);
    const T u = (T)b.g * dk;
    return (T)0.5 * u * u > (sizeof(T) == 8 ? (T)45.0 : (T)20.0);
}

template <typename T>
QI_DEV cplx<T> gabor_response(const DevBand& b, i64 k, int logL, int half_shift) {
    const T g = (T)b.g;
    const T dk = (T)(k - b.kappa_int) - (T)b.kappa_frac;
    const T Lf = (T)(1ll << logL);
    T acc = (T)0;
#pragma unroll
    for (int j = -2; j <= 2; ++j) {
        const T u = g * (dk + (T)j * Lf);
        const T e = exp((T)-0.5 * u * u);
        acc += (half_shift && (j & 1)) ? -e : e;
    }
    acc *= (T)b.gain;
    if (!half_shift) return mk<T>(acc, (T)0);
    // exp(-i*theta_k/2) = exp(-i*pi*k/L)
    const cplx<T> ph = conj(unit_root<T>((unsigned long long)k, logL + 1));
    return ph * acc;
}

// ---------------------------------------------------------------- time-domain atom sample (double)
// x replicates the reference's rounding: fs*(m/fs - ((N-1)/fs)/2)
QI_DEV double atom_xtime(i64 m, i64 n_points, double fs) {
    const double t = (double)m / fs;
    const double off = ((double)(n_points - 1) / fs) / 2.0;
    return fs * (t - off);
}
QI_DEV void atom_value(const DevBand& b, double x, double* re, double* im) {
    const double env = b.amp * exp(-b.p_re * x * x);
    const double ph = b.omega * x - b.p_im * x * x;
    double s, c;
    sincos(ph, &s, &c);
    *re = env * c;
    *im = env * s;
}
QI_DEV void atom_sample(const DevBand& b, i64 m, i64 n_points, double fs, double* re, double* im) {
    atom_value(b, atom_xtime(m, n_points, fs), re, im);
}

// Source for the atom-table forward FFT.  batch = table band index.
template <typename T> struct SrcAtomKernel {
    const DevBand* bands; const int* table_band; CwtGeom geo;
    QI_DEV cplx<T> load(i64 batch, i64 e) const {
        const DevBand& b = bands[table_band[batch]];
        double re, im;
        if (geo.conv_mode == QI_CONV_LINEAR_SAME) {
            const i64 L = 1ll << geo.logL;
            i64 d;
            if (e <= geo.d_max) d = e;
            else if (e - L >= geo.d_min) d = e - L;
            else return mk<T>((T)0, (T)0);
            const i64 m = d + geo.centre_idx;          // index into h = conj(flip(atom))
            atom_sample(b, geo.n_points - 1 - m, geo.n_points, geo.fs, &re, &im);
            return mk<T>((T)re, (T)-im);
        }
        if (e >= geo.n_points) return mk<T>((T)0, (T)0);
        atom_sample(b, e, geo.n_points, geo.fs, &re, &im);
        return mk<T>((T)re, (T)im);
    }
};

// Source for the first inverse pass: record spectrum x band response.  batch = band_in_group*C + chan
template <typename T> struct SrcCwtSpec {
    const cplx<T>* spec; const cplx<T>* tables; const DevBand* bands; int band0; CwtGeom geo;
    QI_DEV cplx<T> load(i64 batch, i64 e) const {
        const i64 chan = batch % geo.n_channels;
        const DevBand& b = bands[band0 + (int)(batch / geo.n_channels)];
        if (b.table_off < 0 && gabor_response_negligible<T>(b, (i64)brev_bits((unsigned)e, geo.logL), geo.logL))
            return mk<T>((T)0, (T)0);
        const cplx<T> X = spec[(chan << geo.logL) + e];
        if (b.table_off >= 0) {
            cplx<T> H = tables[b.table_off + e];
            const T gn = (T)b.gain;
            if (geo.conv_mode == QI_CONV_CIRC_CORR) return mul_conj(X, H) * gn;
            return (X * H) * gn;
        }
        const i64 k = (i64)brev_bits((unsigned)e, geo.logL);
        return X * gabor_response<T>(b, k, geo.logL, geo.half_shift);
    }
};

// plain kernel writing time-domain atoms (public API wavelet_centered_4cwt)
template <typename T>
__global__ void atoms_time_kernel(const DevBand* bands, int n_bands, i64 n_points, double fs, const double* xtime,
                                  cplx<T>* out) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    if (i >= n_points) return;
    double re, im;
    atom_value(bands[b], xtime ? xtime[i] : atom_xtime(i, n_points, fs), &re, &im);
    out[(i64)b * n_points + i] = mk<T>((T)re, (T)im);
}

}  // namespace qi
#include "qi_cwt_fast.cuh"
namespace qi {

struct CwtLayout {
    int logL; i64 L;
    size_t off_bands, off_tabidx, off_spec, off_tables, off_work, off_bandsF, off_ids, off_coef, off_tabF, total;
    int group;
};

template <typename T>
static CwtLayout cwt_layout(i64 C, i64 N, int B, int n_tab, int group, int conv_mode) {
    CwtLayout lo;
    lo.logL = conv_mode == QI_CONV_CIRC_CORR ? ceil_log2_i64(N) : ceil_log2_i64(N > 1 ? 2 * N - 1 : 1);
    lo.L = 1ll << lo.logL;
    if (group < 1) group = 1;
    if (group > B) group = B;
    while ((i64)group * C > 65535 && group > 1) --group;
    lo.group = group;
    size_t o = 0;
    lo.off_bands = o; o = align_up(o + sizeof(DevBand) * (size_t)B, 256);
    lo.off_tabidx = o; o = align_up(o + sizeof(int) * (size_t)(n_tab > 0 ? n_tab : 1), 256);
    lo.off_spec = o; o = align_up(o + sizeof(cplx<T>) * (size_t)C * lo.L, 256);
    lo.off_tables = o; o = align_up(o + sizeof(cplx<T>) * (size_t)n_tab * lo.L, 256);
    lo.off_work = o; o = align_up(o + sizeof(cplx<T>) * (size_t)group * C * lo.L, 256);
    // band-limited routes (qi_cwt_fast.cuh): F-grid descriptors, id lists, interpolator and response tables
    lo.off_bandsF = o; o = align_up(o + sizeof(DevBand) * (size_t)B, 256);
    lo.off_ids = o; o = align_up(o + sizeof(int) * 2 * (size_t)B, 256);
    lo.off_coef = o; o = align_up(o + sizeof(T) * CwtFastCfg<T>::TAPS * (size_t)(CWTF_MAX_LOGD + 1) * (1u << CWTF_MAX_LOGD), 256);
    lo.off_tabF = o; o = align_up(o + sizeof(cplx<T>) * ((size_t)B << CWTF_OS_LOGF), 256);
    lo.total = o;
    return lo;
}

static void fill_dev_bands(const QiAtomBand* hb, int B, int logL, int half_shift, std::vector<DevBand>& db,
                           std::vector<int>& tab) {
    const double L = (double)(1ll << logL);
    db.resize(B);
    tab.clear();
    for (int b = 0; b < B; ++b) {
        DevBand d;
        d.omega = hb[b].omega; d.p_re = hb[b].p_re; d.p_im = hb[b].p_im; d.amp = hb[b].amp;
        d.kc = 0; d.dec_kmax = 0;
        if (hb[b].analytic) {
            // centre frequency folded into [0, 2*pi): a centre beyond the sampling rate (orders below the 0.75
            // floor produce such bands upstream) aliases onto omega - 2*pi*m, with a sign (-1)^m from the
            // half-sample offset of the 'same' slice
            const double wraps = floor(hb[b].omega / (2.0 * M_PI));
            const double omega_r = hb[b].omega - 2.0 * M_PI * wraps;
            const double sign = (half_shift && (((long long)wraps) & 1)) ? -1.0 : 1.0;
            d.gain = sign * hb[b].amp * sqrt(M_PI / hb[b].p_re) / L;
            d.g = (2.0 * M_PI / L) / sqrt(2.0 * hb[b].p_re);
            const double kappa = omega_r * L / (2.0 * M_PI);
            const double ki = floor(kappa);
            d.kappa_int = (long long)ki;
            d.kappa_frac = kappa - ki;
            d.table_off = -1;
            d.kc = (long long)llround(kappa) & ((1ll << logL) - 1);
        } else {
            d.gain = 1.0 / L; d.g = 0; d.kappa_frac = 0; d.kappa_int = 0;
            d.table_off = (long long)tab.size() << logL;
            tab.push_back(b);
        }
        db[b] = d;
    }
}

template <typename T>
static int cwt_fft_impl(const void* sig, i64 C, i64 N, i64 stride, const QiAtomBand* hb, int B, double fs,
                        int conv_mode, void* out_c, void* out_p, double* band_sum, void* ws, size_t ws_bytes,
                        int group, cudaStream_t st, bool fast) {
    int n_tab = 0;
    for (int b = 0; b < B; ++b) {
        if (!hb[b].analytic) ++n_tab;
        else if (hb[b].p_im != 0.0 || !(hb[b].p_re > 0.0) || conv_mode != QI_CONV_LINEAR_SAME) return QI_ERR_ARG;
    }
    const CwtLayout lo = cwt_layout<T>(C, N, B, n_tab, group, conv_mode);
    if (ws_bytes < lo.total) return QI_ERR_WORKSPACE;
    if (conv_mode == QI_CONV_CIRC_CORR && (N & (N - 1))) return QI_ERR_ARG;
    if (C > 65535) return QI_ERR_UNSUPPORTED;
    unsigned char* base = static_cast<unsigned char*>(ws);
    DevBand* d_bands = reinterpret_cast<DevBand*>(base + lo.off_bands);
    int* d_tab = reinterpret_cast<int*>(base + lo.off_tabidx);
    cplx<T>* spec = reinterpret_cast<cplx<T>*>(base + lo.off_spec);
    cplx<T>* tables = reinterpret_cast<cplx<T>*>(base + lo.off_tables);
    cplx<T>* work = reinterpret_cast<cplx<T>*>(base + lo.off_work);

    std::vector<DevBand> db; std::vector<int> tab;
    const int half_shift = (conv_mode == QI_CONV_LINEAR_SAME && (N % 2 == 0)) ? 1 : 0;
    fill_dev_bands(hb, B, lo.logL, half_shift, db, tab);
    CwtFastPlan fp;
    cwt_fast_plan<T>(hb, B, N, lo.logL, conv_mode, fast, fp);
    for (int b = 0; b < B; ++b)
        if (fp.route[b] == CWT_ROUTE_DEC)
            db[b].dec_kmax = (long long)ceil(CwtFastCfg<T>::U_CUT / db[b].g) + 1;
    stage_to_device(d_bands, db.data(), sizeof(DevBand) * (size_t)B, st);
    if (n_tab) stage_to_device(d_tab, tab.data(), sizeof(int) * (size_t)n_tab, st);

    CwtGeom geo;
    geo.n_points = N; geo.n_channels = C; geo.n_bands = B; geo.logL = lo.logL;
    geo.conv_mode = conv_mode; geo.fs = fs;
    geo.centre_idx = (N - 1) / 2;
    geo.half_shift = half_shift;
    geo.d_min = -geo.centre_idx;
    geo.d_max = N - 1 - geo.centre_idx;

    const FftPlan plan = make_plan(lo.logL, (int)sizeof(cplx<T>));
    if (band_sum) cudaMemsetAsync(band_sum, 0, sizeof(double) * (size_t)C * B, st);

    // ---- (S) short atoms: overlap-save in shared memory, straight from the record
    if (!fp.os_ids.empty()) {
        const int n_os = (int)fp.os_ids.size(), logF = CWTF_OS_LOGF;
        DevBand* d_bandsF = reinterpret_cast<DevBand*>(base + lo.off_bandsF);
        int* d_os = reinterpret_cast<int*>(base + lo.off_ids);
        cplx<T>* tabF = reinterpret_cast<cplx<T>*>(base + lo.off_tabF);
        std::vector<QiAtomBand> sel(n_os);
        for (int i = 0; i < n_os; ++i) sel[i] = hb[fp.os_ids[i]];
        std::vector<DevBand> dbF; std::vector<int> tabF_unused;
        fill_dev_bands(sel.data(), n_os, logF, half_shift, dbF, tabF_unused);
        stage_to_device(d_bandsF, dbF.data(), sizeof(DevBand) * (size_t)n_os, st);
        stage_to_device(d_os, fp.os_ids.data(), sizeof(int) * (size_t)n_os, st);
        prof_set_category(QI_CAT_FFT_FWD);
        QI_LAUNCH((cwtf_os_table_kernel<T>), dim3((unsigned)((1 << logF) / 256), (unsigned)n_os), dim3(256), 0, st,
                  (const DevBand*)d_bandsF, logF, half_shift, tabF);
        overlap_save_route<T>(sig, stride, geo, d_os, n_os, fp.os_half, OsTableRoute<T>{tabF}, out_c, out_p, band_sum, st);
    }

    // record spectra (the overlap-save route does not need them)
    prof_set_category(QI_CAT_FFT_FWD);
    if ((int)fp.os_ids.size() < B)
        forward_passes<T>(plan, C, SrcRealPad<T>{static_cast<const T*>(sig), stride, N}, spec, lo.L, st);
    // atom tables (one forward FFT per table band, shared by all channels)
    if (n_tab) forward_passes<T>(plan, n_tab, SrcAtomKernel<T>{d_bands, d_tab, geo}, tables, lo.L, st);

    // ---- (D) long decayed atoms: baseband bins -> short inverse transform -> Kaiser-sinc interpolation
    int* d_dec = reinterpret_cast<int*>(base + lo.off_ids) + B;
    T* coef = reinterpret_cast<T*>(base + lo.off_coef);
    const auto dec_src = [&](const int* ids, int lk) { return SrcCwtDec<T>{spec, d_bands, ids, (int)C, lo.logL, lk, half_shift}; };
    const int rc = decimated_route<T, true, true, 2>(fp.logK, geo, dec_src, &d_bands[0].kc, (int)(sizeof(DevBand) / sizeof(long long)),
                                                     d_dec, coef, work, work, (size_t)lo.group * C * lo.L, out_c, out_p, band_sum, st);
    if (rc != QI_OK) return rc;

    // ---- plain route: maximal runs of consecutive bands that took no other route
    for (int band0 = 0; band0 < B;) {
        if (fp.route[band0] != CWT_ROUTE_PLAIN) { ++band0; continue; }
        int g = 1;
        while (band0 + g < B && g < lo.group && fp.route[band0 + g] == CWT_ROUTE_PLAIN) ++g;
        inverse_passes<T>(plan, (i64)g * C, SrcCwtSpec<T>{spec, tables, d_bands, band0, geo},
                          DstCwtOut<T>{static_cast<cplx<T>*>(out_c), static_cast<T*>(out_p), band_sum, band0, geo, 0.0}, 256,
                          true, work, lo.L, st);
        band0 += g;
    }
    prof_set_category(QI_CAT_OTHER);
    return check_cuda("qi_cwt_fft");
}

template <typename T>
static int atoms_time_impl(const QiAtomBand* hb, int B, i64 N, double fs, const double* xtime, void* out, void* ws,
                           size_t ws_bytes, cudaStream_t st) {
    if (ws_bytes < sizeof(DevBand) * (size_t)B) return QI_ERR_WORKSPACE;
    std::vector<DevBand> db; std::vector<int> tab;
    std::vector<QiAtomBand> tmp(hb, hb + B);
    for (auto& t : tmp) t.analytic = 0;
    fill_dev_bands(tmp.data(), B, 0, 0, db, tab);
    DevBand* d_bands = static_cast<DevBand*>(ws);
    stage_to_device(d_bands, db.data(), sizeof(DevBand) * (size_t)B, st);
    dim3 grid((unsigned)((N + 255) / 256), (unsigned)B);
    QI_LAUNCH((atoms_time_kernel<T>), grid, dim3(256), 0, st, (const DevBand*)d_bands, B, N, fs, xtime, static_cast<cplx<T>*>(out));
    return check_cuda("qi_atoms_time");
}

}  // namespace qi

extern "C" {

size_t qi_cwt_workspace_bytes(int64_t C, int64_t N, int B, int n_tab, int group, int conv_mode, int dtype) {
    if (C <= 0 || N <= 0 || B <= 0) return 0;
    conv_mode &= ~QI_CONV_PLAIN_ONLY;
    if (dtype == QI_F32) return qi::cwt_layout<float>(C, N, B, n_tab, group, conv_mode).total;
    return qi::cwt_layout<double>(C, N, B, n_tab, group, conv_mode).total;
}

int qi_cwt_fft(const void* sig, int64_t C, int64_t N, int64_t stride, const QiAtomBand* bands, int B, double fs,
               int conv_mode, int dtype, void* out_cwt, void* out_power, double* band_sum, void* ws, size_t ws_bytes,
               int group, void* stream) {
    if (!sig || !bands || !ws || C <= 0 || N <= 0 || B <= 0 || stride < N) return QI_ERR_ARG;
    if (N > (1ll << 29)) return QI_ERR_UNSUPPORTED;
    const bool fast = !(conv_mode & QI_CONV_PLAIN_ONLY);
    conv_mode &= ~QI_CONV_PLAIN_ONLY;
    if (conv_mode != QI_CONV_LINEAR_SAME && conv_mode != QI_CONV_CIRC_CORR) return QI_ERR_ARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (dtype == QI_F32)
        return qi::cwt_fft_impl<float>(sig, C, N, stride, bands, B, fs, conv_mode, out_cwt, out_power, band_sum, ws,
                                       ws_bytes, group, st, fast);
    if (dtype == QI_F64)
        return qi::cwt_fft_impl<double>(sig, C, N, stride, bands, B, fs, conv_mode, out_cwt, out_power, band_sum, ws,
                                        ws_bytes, group, st, fast);
    return QI_ERR_ARG;
}

int qi_atoms_time(const QiAtomBand* bands, int B, int64_t N, double fs, int dtype, const double* xtime, void* out,
                  void* ws, size_t ws_bytes, void* stream) {
    if (!bands || !out || !ws || B <= 0 || N <= 0 || B > 65535) return QI_ERR_ARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (dtype == QI_F32) return qi::atoms_time_impl<float>(bands, B, N, fs, xtime, out, ws, ws_bytes, st);
    if (dtype == QI_F64) return qi::atoms_time_impl<double>(bands, B, N, fs, xtime, out, ws, ws_bytes, st);
    return QI_ERR_ARG;
}

}  // extern "C"
