// qi_interp.cuh -- the band-limited routes shared by the exact Gabor CWT (qi_cwt.cu, qi_cwt_fast.cuh) and the Stockwell
// transform (qi_stx.cu, methods "exact" and "multirate"), float32 and float64.
//
// DECIMATED route.  A band whose spectrum is negligible outside K = 2^m bins around its centre is known exactly from the
// K-point inverse transform of those bins: every D = L / K-th sample of its L-point (circular) output, demodulated by the
// centre bin.  A TAPS-per-phase Kaiser-windowed-sinc interpolator brings it to the full rate, puts the carrier back
// (exact integer phase, stepped inside a thread; a Stockwell voice is baseband and has none) and fuses the output slice,
// |.|^2 and the fp64 band sums.
//     float32: RHO = 2 (oversampling of the decimated samples), 16 taps, beta 11.2 (stop band -110 dB)
//     float64: RHO = 4, 24 taps, beta 24.5 (-231 dB)
// OVERLAP-SAVE route.  A band too wide in frequency to decimate is short in time: the record is cut into blocks of
// F = 2048 samples held in shared memory, one forward transform per block, and per band one product with the band's
// response on the F-grid and one inverse transform; the valid samples go straight to the planes.
#pragma once
#include "qi_host.h"
#include "qi_tfr.cuh"

#include <vector>

namespace qi {

constexpr int CWTF_MAX_LOGD = 8;
constexpr int CWTF_TILE = 2048;
constexpr int CWTF_SPAN = 4;                 // tiles per CTA of the interpolator
constexpr int CWTF_OS_LOGF = 11;             // overlap-save block length 2048
constexpr int CWTF_OS_MAX_HALF = 384;        // longest kernel half-support taken by the overlap-save route

template <typename T> struct CwtFastCfg;
template <> struct CwtFastCfg<float> {
    static constexpr int TAPS = 16, RHO = 2, PER = 8;
    static constexpr double U_CUT = 5.6, BETA = 11.2;
};
template <> struct CwtFastCfg<double> {
    static constexpr int TAPS = 24, RHO = 4, PER = 4;
    static constexpr double U_CUT = 7.7, BETA = 24.5;
};

template <typename T> struct CwtFastAcc { typedef double type; };
template <> struct CwtFastAcc<float> { typedef float type; };

// modified Bessel function I0 by its power series (converged to 1e-19 of the sum for x <= 23 after 64 terms)
QI_HD double cwtf_bessel_i0(double x) {
    double s = 1.0, term = 1.0;
    const double hh = 0.25 * x * x;
    for (int k = 1; k <= 64; ++k) { term *= hh / (double)(k * k); s += term; }
    return s;
}

// coef[logD][j * D + p] = h(p - (j - (TAPS/2 - 1)) D),  h(t) = sinc(t / D) kaiser(t / (TAPS/2 D); beta)
template <typename T>
__global__ void cwtf_coef_kernel(T* __restrict__ coef_all, unsigned need_mask, double inv_i0_beta) {
    constexpr int TAPS = CwtFastCfg<T>::TAPS;
    const int logD = blockIdx.y;
    if (!((need_mask >> logD) & 1u)) return;
    T* coef = coef_all + (size_t)logD * TAPS * (1u << CWTF_MAX_LOGD);
    const int D = 1 << logD;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= TAPS * D) return;
    const int j = idx >> logD, p = idx & (D - 1);
    const double t = (double)(p - (j - (TAPS / 2 - 1)) * D);
    const double x = t / (0.5 * TAPS * D);
    const double arg = 1.0 - x * x;
    const double w = cwtf_bessel_i0(CwtFastCfg<T>::BETA * sqrt(arg > 0.0 ? arg : 0.0)) * inv_i0_beta;
    const double y = t / (double)D;
    const double sinc = t == 0.0 ? 1.0 : sinpi(y) / (M_PI * y);
    coef[idx] = (T)(sinc * w);
}

// grid: (ceil(N / (SPAN * TILE)), bands of the group, channels);  dec: [band_in_group][chan][K]
// CARRIER: the output is the interpolated band times exp(2 pi i k_c n / L), k_c = kc_of_band[band * kc_stride].  SUMS: the
// fp64 band sums are accumulated (into band_sum, when it is not null).  MIN_LOGD: the smallest decimation launched; it
// sizes the shared segment (at D = 2 twice that of D >= 4, which would cost the CWT and exact Stockwell routes occupancy).
// float64 keeps the real and the imaginary parts of the decimated samples in separate shared arrays and runs the taps over
// one part at a time: 27 + 24 doubles live instead of 54 + 24, i.e. ~120 instead of 198 registers and two CTAs per SM
// instead of one (ncu before: occupancy 12 %, issue-active 45 %, no memory stall -- the FP64 pipe waiting for issue slots).
// float32 without the band sums fits 64 registers: four CTAs per SM, on which the speed of method="multirate" rests.
template <typename T, bool CARRIER, bool SUMS, int MIN_LOGD>
__global__ void __launch_bounds__(256, sizeof(T) == 8 ? 2 : (SUMS ? 1 : 4))
cwtf_interp_kernel(const cplx<T>* __restrict__ dec, const int* __restrict__ ids, const long long* __restrict__ kc_of_band,
                   int kc_stride, CwtGeom geo, int logD, const T* __restrict__ coef, cplx<T>* __restrict__ out_c, T* __restrict__ out_p,
                   double* __restrict__ band_sum) {
    constexpr int TAPS = CwtFastCfg<T>::TAPS, PER = CwtFastCfg<T>::PER, NSUB = 8 / PER, J0 = TAPS / 2 - 1;
    constexpr bool SPLIT = sizeof(T) == 8;
    // one pad slot per 8 decimated samples: at small D the lanes of a warp start their windows PER samples apart
    constexpr int SEGN = ((CWTF_SPAN * CWTF_TILE >> MIN_LOGD) + TAPS) * 9 / 8 + 2;
    __shared__ cplx<T> seg[SEGN];
    T* seg_re = reinterpret_cast<T*>(seg);                  // SPLIT: [SEGN] real parts, then [SEGN] imaginary parts
    T* seg_im = seg_re + SEGN;
    __shared__ double scratch[32];
    const int D = 1 << logD, logK = geo.logL - logD;
    const i64 K = 1ll << logK, N = geo.n_points;
    const i64 span0 = (i64)blockIdx.x * (CWTF_SPAN * CWTF_TILE);
    const i64 left = (N - span0 + CWTF_TILE - 1) / CWTF_TILE;
    const int ntile = left < CWTF_SPAN ? (int)left : CWTF_SPAN;
    const int bi = blockIdx.y, chan = blockIdx.z, band = ids[bi];
    const cplx<T>* src = dec + (((i64)bi * geo.n_channels + chan) << logK);
    const i64 m_base = (span0 >> logD) - J0;
    const int nseg = ((ntile * CWTF_TILE) >> logD) + TAPS;
    for (int i = threadIdx.x; i < nseg; i += blockDim.x) {
        const cplx<T> v = src[(m_base + i) & (K - 1)];
        if (SPLIT) { seg_re[i + (i >> 3)] = v.re; seg_im[i + (i >> 3)] = v.im; }
        else seg[i + (i >> 3)] = v;
    }
    __syncthreads();
    const i64 row = ((i64)chan * geo.n_bands + band) * N;
    const int p = threadIdx.x & (D - 1);
    const int MT = CWTF_TILE >> logD;                       // decimated samples per tile
    T cf[TAPS];
#pragma unroll
    for (int j = 0; j < TAPS; ++j) cf[j] = coef[(j << logD) + p];
    // carrier exp(2 pi i k_c n / L) at n = m D + p: exact at the first sample of a run, stepped by exp(2 pi i k_c D / L)
    const unsigned long long Lmask = (1ull << geo.logL) - 1ull;
    const unsigned long long kc = CARRIER ? (unsigned long long)kc_of_band[(size_t)band * kc_stride] : 0ull;
    const cplx<T> step = unit_root<T>((kc << logD) & Lmask, geo.logL);
    // float32: partial sums of a thread's <= 64 non-negative outputs in the arithmetic type, fp64 across the CTA
    typename CwtFastAcc<T>::type acc = 0;
    for (int tl = 0; tl < ntile; ++tl) {
#pragma unroll
        for (int sub = 0; sub < NSUB; ++sub) {
            const int m0 = tl * MT + sub * (MT / NSUB) + (threadIdx.x >> logD) * PER;
            T re[PER], im[PER];
            if (SPLIT) {
                // m0 is a multiple of PER = 4: the window starts at slot m0 + (m0 >> 3) and crosses a padding slot where
                // (m0 & 7) + j reaches a multiple of 8
                const int s0 = m0 + (m0 >> 3), r0 = m0 & 7;
#pragma unroll
                for (int part = 0; part < 2; ++part) {
                    const T* sp = (part ? seg_im : seg_re) + s0;
                    T win[PER + TAPS - 1];
#pragma unroll
                    for (int j = 0; j < PER + TAPS - 1; ++j) win[j] = sp[j + ((r0 + j) >> 3)];
#pragma unroll
                    for (int i = 0; i < PER; ++i) {
                        T a = (T)0;
#pragma unroll
                        for (int j = 0; j < TAPS; ++j) a += cf[j] * win[i + j];
                        if (part) im[i] = a; else re[i] = a;
                    }
                }
            } else {
                // float32: one packed fma.rn.f32x2 per tap on the (re, im) pair (the kernel is issue-bound: ncu 76 %
                // issue-active, 87 thread instructions per output cell with scalar taps)
                const f32x2* seg2 = reinterpret_cast<const f32x2*>(seg);
                f32x2 win[PER + TAPS - 1];
#pragma unroll
                for (int j = 0; j < PER + TAPS - 1; ++j) win[j] = seg2[m0 + j + ((m0 + j) >> 3)];
#pragma unroll
                for (int i = 0; i < PER; ++i) {
                    f32x2 a = f2_make(0.0f, 0.0f);
#pragma unroll
                    for (int j = 0; j < TAPS; ++j) a = f2_fma(f2_make((float)cf[j], (float)cf[j]), win[i + j], a);
                    re[i] = (T)f2_lo(a); im[i] = (T)f2_hi(a);
                }
            }
            const i64 n0 = span0 + ((i64)m0 << logD) + p;
            cplx<T> car = mk<T>((T)1, (T)0);
            if (CARRIER && out_c) car = unit_root<T>((kc * (unsigned long long)n0) & Lmask, geo.logL);
#pragma unroll
            for (int i = 0; i < PER; ++i) {
                const i64 n = n0 + ((i64)i << logD);
                if (n < N) {
                    const T pw = re[i] * re[i] + im[i] * im[i];
                    if (out_c) out_c[row + n] = CARRIER ? mk<T>(re[i], im[i]) * car : mk<T>(re[i], im[i]);
                    if (out_p) out_p[row + n] = pw;
                    if (SUMS) acc += pw;
                }
                if (CARRIER && out_c) car = car * step;
            }
        }
    }
    if (SUMS && band_sum) {
        const double tot = block_sum((double)acc, scratch);
        if (threadIdx.x == 0) atomicAdd(&band_sum[(i64)chan * geo.n_bands + band], tot);
    }
}

// log2 K of the decimated route for a band whose bins farther than kmax from its centre are negligible: the smallest
// K = 2^m >= rho (2 kmax + guard), at most 2^CWTF_MAX_LOGD-fold decimation and at least 64 bins.  logL (no decimation) when
// that K is above L / 4 (above L / 2 with allow_d2).
inline int dec_logk(double kmax, double rho, double guard, int logL, bool allow_d2) {
    const double need = rho * (2.0 * kmax + guard);
    int lk = logL - CWTF_MAX_LOGD;
    if (lk < 6) lk = 6;
    while (lk < logL && (double)(1ll << lk) < need) ++lk;
    return lk <= logL - (allow_d2 ? 1 : 2) ? lk : logL;
}

// Decimated route of every band b with logK[b] < geo.logL: the interpolator tables of the decimations in use, then, by
// increasing K, groups of bands with the same K (capped by grid.y and by `work_elems` elements of `work` and `dec`): the
// K-point inverse transform -- first pass `src_of(device ids of the group, logK)`, the passes between in `work`, the last
// into `dec` (which may be `work`) -- and the interpolator.
template <typename T, bool CARRIER, bool SUMS, int MIN_LOGD, class SrcOf>
static int decimated_route(const std::vector<int>& logK, const CwtGeom& geo, SrcOf src_of, const long long* kc_of_band,
                           int kc_stride, int* d_ids, T* coef, cplx<T>* work, cplx<T>* dec, size_t work_elems,
                           void* out_c, void* out_p, double* band_sum, cudaStream_t st) {
    typedef CwtFastCfg<T> Cfg;
    const int logL = geo.logL;
    const i64 C = geo.n_channels;
    std::vector<int> ids;
    unsigned need_mask = 0;
    for (int lk = 0; lk < logL; ++lk)
        for (int b = 0; b < (int)logK.size(); ++b)
            if (logK[b] == lk) { ids.push_back(b); need_mask |= 1u << (logL - lk); }
    if (ids.empty()) return QI_OK;
    stage_to_device(d_ids, ids.data(), sizeof(int) * ids.size(), st);
    prof_set_category(QI_CAT_OTHER);
    QI_LAUNCH((cwtf_coef_kernel<T>), dim3((unsigned)((Cfg::TAPS << CWTF_MAX_LOGD) / 256 + 1), (unsigned)(CWTF_MAX_LOGD + 1)),
              dim3(256), 0, st, coef, need_mask, 1.0 / cwtf_bessel_i0(Cfg::BETA));
    for (size_t pos = 0; pos < ids.size();) {
        const int lk = logK[ids[pos]], logD = logL - lk;
        size_t end = pos;
        while (end < ids.size() && logK[ids[end]] == lk) ++end;
        const T* cf = coef + (size_t)logD * Cfg::TAPS * (1u << CWTF_MAX_LOGD);
        const FftPlan pk = make_plan(lk, (int)sizeof(cplx<T>));
        const i64 K = 1ll << lk;
        while (pos < end) {
            i64 gs = (i64)(end - pos);
            while (gs > 1 && (gs * C > 65535 || (size_t)gs * C * K > work_elems)) --gs;
            if (gs * C > 65535 || (size_t)gs * C * K > work_elems) return QI_ERR_WORKSPACE;
            inverse_passes<T>(pk, gs * C, src_of(d_ids + pos, lk), DstComplex<T>{dec, K, (T)1}, 0, false, work, K, st);
            prof_set_category(QI_CAT_INV_LAST);
            dim3 grid((unsigned)((geo.n_points + CWTF_SPAN * CWTF_TILE - 1) / (CWTF_SPAN * CWTF_TILE)), (unsigned)gs, (unsigned)C);
            QI_LAUNCH((cwtf_interp_kernel<T, CARRIER, SUMS, MIN_LOGD>), grid, dim3(256), 0, st, (const cplx<T>*)dec,
                      (const int*)(d_ids + pos), kc_of_band, kc_stride, geo, logD, cf, static_cast<cplx<T>*>(out_c),
                      static_cast<T*>(out_p), band_sum);
            pos += (size_t)gs;
        }
    }
    return QI_OK;
}

// Overlap-save route.  grid: (ceil(N / V), channels); one block of F samples, all n_os bands.
// dyn smem: (2 pad8(F) + F) complex + 256 B.  logF (= CWTF_OS_LOGF) is a run-time argument: with a compile-time block
// length the unrolled tile transforms need more registers (float64: 84) than two 512-thread CTAs per SM leave.
// `Route` supplies what differs between the transforms:
//   T sample(xs, k, N)        sample k of the record xs (k may lie outside [0, N): zero-extended or circular)
//   Route::Band band(i, b)    the i-th band (band index b), with
//     cplx<T> weigh(x, r, geo)   block bin x (bit-reversed slot r) times the band's response on the F-grid
//     cplx<T> out(y, n, geo)     the complex output stored for the band's filtered sample y at n
template <typename T, class Route>
__global__ void __launch_bounds__(512)
cwtf_os_kernel(const T* __restrict__ sig, i64 stride, CwtGeom geo, const int* __restrict__ ids, int n_os, int logF,
               int half, Route route, cplx<T>* __restrict__ out_c, T* __restrict__ out_p, double* __restrict__ band_sum) {
    QI_DYN_SMEM(smem_raw);
    const int F = 1 << logF, V = F - 2 * half;
    const int FP = pad8(F);                                   // tiles in the padded single-column layout of tile_fft<.., true>
    cplx<T>* tile_x = reinterpret_cast<cplx<T>*>(smem_raw);
    cplx<T>* tile_y = tile_x + FP;
    cplx<T>* tw = tile_y + FP;
    double* scratch = reinterpret_cast<double*>(tw + F);
    const i64 chan = blockIdx.y, N = geo.n_points;
    const i64 n0 = (i64)blockIdx.x * V;
    const T* xs = sig + chan * stride;
    fill_stage_twiddles<T>(tw, logF);
    for (int p = threadIdx.x; p < F; p += blockDim.x) tile_x[padt<T>(p)] = mk<T>(route.sample(xs, n0 - half + p, N), (T)0);
    __syncthreads();
    tile_fft<T, FFT_FWD, true>(tile_x, tw, logF, 1, 1);
    for (int i = 0; i < n_os; ++i) {
        const int band = ids[i];
        const typename Route::Band h = route.band(i, band);
        for (int r = threadIdx.x; r < F; r += blockDim.x) tile_y[padt<T>(r)] = h.weigh(tile_x[padt<T>(r)], r, geo);
        __syncthreads();
        tile_fft<T, FFT_INV, true>(tile_y, tw, logF, 1, 1);
        const i64 row = (chan * geo.n_bands + band) * N;
        double acc = 0.0;
        for (int v = threadIdx.x; v < V; v += blockDim.x) {
            const i64 n = n0 + v;
            if (n < N) {
                const cplx<T> y = tile_y[padt<T>(half + v)];
                const T pw = norm2(y);
                if (out_c) out_c[row + n] = h.out(y, n, geo);
                if (out_p) out_p[row + n] = pw;
                acc += (double)pw;
            }
        }
        if (band_sum) {
            acc = block_sum(acc, scratch);
            if (threadIdx.x == 0) atomicAdd(&band_sum[chan * geo.n_bands + band], acc);
        }
        __syncthreads();
    }
}

// the n_os bands d_ids[0 .. n_os) by the overlap-save route, kernel half-support `half` samples (a multiple of 16)
template <typename T, class Route>
static void overlap_save_route(const void* sig, i64 stride, const CwtGeom& geo, const int* d_ids, int n_os, int half,
                               Route route, void* out_c, void* out_p, double* band_sum, cudaStream_t st) {
    const int F = 1 << CWTF_OS_LOGF, V = F - 2 * half;
    const size_t smem = sizeof(cplx<T>) * (2 * (size_t)pad8(F) + (size_t)F) + 256;
#ifndef QI_EMUL
    cudaFuncSetAttribute(cwtf_os_kernel<T, Route>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
#endif
    prof_set_category(QI_CAT_INV_LAST);
    QI_LAUNCH((cwtf_os_kernel<T, Route>), dim3((unsigned)((geo.n_points + V - 1) / V), (unsigned)geo.n_channels), dim3(512),
              smem, st, static_cast<const T*>(sig), stride, geo, d_ids, n_os, CWTF_OS_LOGF, half, route, static_cast<cplx<T>*>(out_c),
              static_cast<T*>(out_p), band_sum);
}

}  // namespace qi
