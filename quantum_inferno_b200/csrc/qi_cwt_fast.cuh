// qi_cwt_fast.cuh -- band-limited routes of the exact (FFT) Gabor CWT, float32 and float64.
//
// The plain route of qi_cwt.cu spends three full-length HBM passes (length L = 2N) on every band.  A Gaussian atom
// whose support has decayed inside the record does not need them:
//
//  (D) DECIMATED route, long atoms (s large).  The band response exp(-0.5 s^2 (theta - omega)^2) is below CUT of its
//      peak beyond |k - k_c| > kmax = U / (s 2 pi / L) bins.  The K = 2^m >= RHO (2 kmax + 4) bins around k_c, moved to
//      baseband, are inverse-transformed at length K (same pass kernels, K << L): that is the band output at every
//      D = L / K-th sample, demodulated by exp(-2 pi i k_c n / L), EXACTLY (the product is band-limited on the circular
//      L-grid).  A TAPS-per-phase Kaiser-windowed-sinc interpolator brings it to the full rate, the carrier is put back
//      (exact integer phase, stepped inside a thread), and the store fuses the 'same' slice, |.|^2 and the fp64 band sum.
//          float32: RHO = 2, 16 taps, beta 11.2  (stop band -110 dB);   float64: RHO = 4, 24 taps, beta 24.5 (-231 dB)
//      HBM traffic per cell: the output + 2 RHO-ish / D reads instead of ~6 x 2 x sizeof(complex).
//
//  (S) OVERLAP-SAVE route, short atoms (the top bands, which are too wide to decimate).  Their kernels are a few
//      hundred samples long (|t| <= U s): the record is cut into blocks of F = 2048 samples held in shared memory, one
//      forward transform per block, and per band one product with the band's response on the F-grid (the same closed
//      form, periodised at F -- exact because the kernel has died out well inside the block) and one inverse transform;
//      the V = F - 2 half valid samples go straight to the planes.  Nothing but the record and the output touches HBM.
//
// Record-long truncated atoms (table bands) and the circular-correlation mode keep the plain route.
// Replaces quantum_inferno/styx_cwt.py:195-196 (scipy fftconvolve on the tiled record) for those bands.
#pragma once
#include "qi_interp.cuh"

namespace qi {

// First inverse pass of the K-point transform of a band's baseband bins.  batch = band_in_group * C + chan
template <typename T> struct SrcCwtDec {
    const cplx<T>* spec; const DevBand* bands; const int* ids; int n_channels, logL, logK, half_shift;
    QI_DEV cplx<T> load(i64 batch, i64 e) const {
        const i64 chan = batch % n_channels;
        const DevBand& b = bands[ids[batch / n_channels]];
        const i64 K = 1ll << logK, L = 1ll << logL;
        const i64 q = (i64)brev_bits((unsigned)e, logK);
        const i64 ks = (q < (K >> 1)) ? q : q - K;
        if (ks > b.dec_kmax || -ks > b.dec_kmax) return mk<T>((T)0, (T)0);
        const i64 k = (b.kc + ks) & (L - 1);
        const cplx<T> X = spec[(chan << logL) + (i64)brev_bits((unsigned)k, logL)];
        return X * gabor_response<T>(b, k, logL, half_shift);
    }
};

// ---------------------------------------------------------------- (S) overlap-save route
// response tables of the overlap-save bands on the F-grid, bit-reversed order: tabF[i][e]
template <typename T>
__global__ void cwtf_os_table_kernel(const DevBand* __restrict__ bandsF, int logF, int half_shift, cplx<T>* __restrict__ tabF) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (1 << logF)) return;
    const i64 k = (i64)brev_bits((unsigned)e, logF);
    tabF[((size_t)blockIdx.y << logF) + e] = gabor_response<T>(bandsF[blockIdx.y], k, logF, half_shift);
}

// Gabor bands on the overlap-save route: the record zero-extended, the response from the bands' F-grid tables, the output
// as the inverse transform leaves it
template <typename T> struct OsTableRoute {
    const cplx<T>* tabF;
    struct Band {
        const cplx<T>* H;
        QI_DEV cplx<T> weigh(cplx<T> x, int r, const CwtGeom&) const { return x * H[r]; }
        QI_DEV cplx<T> out(cplx<T> y, i64, const CwtGeom&) const { return y; }
    };
    QI_DEV T sample(const T* xs, i64 k, i64 N) const { return (k >= 0 && k < N) ? xs[k] : (T)0; }
    QI_DEV Band band(int i, int) const { return Band{tabF + ((size_t)i << CWTF_OS_LOGF)}; }
};

// ---------------------------------------------------------------- host side: which band takes which route
enum { CWT_ROUTE_PLAIN = 0, CWT_ROUTE_DEC = 1, CWT_ROUTE_OS = 2 };

struct CwtFastPlan {
    std::vector<int> route, logK;          // per band; logK < logL on the decimated route
    std::vector<int> os_ids;
    int os_half;
};

template <typename T>
static void cwt_fast_plan(const QiAtomBand* hb, int B, i64 N, int logL, int conv_mode, bool enable, CwtFastPlan& fp) {
    typedef CwtFastCfg<T> Cfg;
    fp.route.assign(B, CWT_ROUTE_PLAIN);
    fp.logK.assign(B, logL);
    fp.os_ids.clear();
    fp.os_half = 0;
    if (!enable || conv_mode != QI_CONV_LINEAR_SAME || logL < 14 || N < 4 * CWTF_TILE) return;
    const double L = (double)(1ll << logL);
    for (int b = 0; b < B; ++b) {
        if (!hb[b].analytic || hb[b].p_im != 0.0 || !(hb[b].p_re > 0.0)) continue;
        const double s = 1.0 / sqrt(2.0 * hb[b].p_re);
        if (s < 1.0) continue;                                   // sub-sample atoms: more aliases than the closed form keeps
        const int half = (int)ceil(Cfg::U_CUT * s) + 2;
        if (half <= CWTF_OS_MAX_HALF) {
            fp.route[b] = CWT_ROUTE_OS;
            fp.os_ids.push_back(b);
            if (half > fp.os_half) fp.os_half = half;
            continue;
        }
        fp.logK[b] = dec_logk(ceil(Cfg::U_CUT * L / (2.0 * M_PI * s)) + 1.0, Cfg::RHO, 4.0, logL, false);
        if (fp.logK[b] < logL) fp.route[b] = CWT_ROUTE_DEC;
    }
    fp.os_half = (fp.os_half + 15) & ~15;
}

}  // namespace qi
