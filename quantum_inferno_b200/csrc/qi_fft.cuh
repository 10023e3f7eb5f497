// qi_fft.cuh -- shared-memory radix-8/4/2 FFT tile core and the multi-pass ("four-step")
// large-FFT pass kernel built on it.
//
// Conventions
//   * Forward = decimation-in-frequency, natural order in -> bit-reversed order out.
//     Inverse = decimation-in-time, bit-reversed order in -> natural order out.
//     A spectrum therefore lives in HBM at position p = bitrev_m(k); products are taken in
//     that order and no transpose / permutation kernel ever runs.  (Replaces the three
//     scipy.fft c2c calls inside scipy.signal.fftconvolve that
//     reference quantum_inferno/styx_cwt.py:195 bottoms out in.)
//   * A length-2^m transform is split into passes of 2^m_i points (m = sum m_i).  Pass i is a
//     set of independent 2^m_i-point FFTs over "rows" r at element stride sR = 2^(bits below),
//     followed (forward) / preceded (inverse) by the Cooley-Tukey twiddle w_(R*sR)^(inner*k).
//   * A CTA holds a tile of R rows x TC columns in shared memory as tile[r*TP + c]
//     (TP = TC+1 -> conflict-free both for column-wise butterflies and row-wise staging).
//     Butterfly lanes run along the columns, so twiddles are warp-uniform broadcasts.
#pragma once
#include "qi_platform.cuh"

// Loads requested per thread before the first is consumed in the load phase of a pass, and the shared-memory budget that
// sets the tile width.  Measured on B200 once the per-element sincospi of the inter-pass twiddles was gone (before that
// the passes were instruction-bound and neither knob mattered), forward / inverse ms of tools/fft_probe.py:
//   (loads, KB)      8 x 2^25 f32     8 x 2^25 f64     672 x 2^18 f32   336 x 2^18 f64
//   (1, 96)          9.19 / 9.08      11.94 / 11.79    4.08 / 3.99      2.60 / 2.58
//   (8, 96)          5.24 / 5.06      11.93 / 11.80    2.27 / 2.15      2.60 / 2.58
//   (4, 48)          5.57 / 5.23       9.59 /  9.42    2.53 / 2.28      2.38 / 2.32
//   (8, 48)          4.23 / 3.97       7.57 /  7.43    2.52 / 2.28      2.04 / 1.98      <- default
//   (8, 32)          6.54 / 6.18      10.24 / 10.62    2.10 / 2.11      3.01 / 3.02
// (gpurun_out r2j, summarised in profiles/r02_fft_pass_tuning.md): the passes are latency-bound -- two ~80 KB CTAs per SM
// with one load in flight per thread kept 8 KB per SM in flight where HBM needs ~20 KB.
#ifndef QI_FFT_LOADS_IN_FLIGHT
#define QI_FFT_LOADS_IN_FLIGHT 8
#endif
#ifndef QI_FFT_TILE_BUDGET_KB
#define QI_FFT_TILE_BUDGET_KB 48
#endif

namespace qi {

enum { FFT_FWD = 0, FFT_INV = 1 };

// ---------------------------------------------------------------- small DFTs in registers
// Outputs are left in BIT-REVERSED slot order (slot brev(f) holds frequency f), which makes a
// radix-8 step identical to three in-place radix-2 DIF steps.
template <typename T, int DIR> QI_DEV cplx<T> rot90(cplx<T> a) {   // * (-i) forward, * (+i) inverse
    return DIR == FFT_FWD ? mul_mi(a) : mul_pi(a);
}
template <typename T, int DIR> QI_DEV cplx<T> rot45(cplx<T> a) {   // * w8^1
    const T h = (T)0.70710678118654752440;
    return DIR == FFT_FWD ? mk<T>((a.re + a.im) * h, (a.im - a.re) * h)
                          : mk<T>((a.re - a.im) * h, (a.im + a.re) * h);
}
template <typename T, int DIR> QI_DEV cplx<T> rot135(cplx<T> a) {  // * w8^3
    const T h = (T)0.70710678118654752440;
    return DIR == FFT_FWD ? mk<T>((a.im - a.re) * h, -(a.re + a.im) * h)
                          : mk<T>(-(a.re + a.im) * h, (a.re - a.im) * h);
}

// DIF butterflies: natural slots in, bit-reversed slots out (sign by DIR).
template <typename T, int DIR> QI_DEV void dif2(cplx<T>* a) {
    cplx<T> t = a[0] - a[1]; a[0] = a[0] + a[1]; a[1] = t;
}
template <typename T, int DIR> QI_DEV void dif4(cplx<T>* a) {
    cplx<T> b0 = a[0] + a[2], b2 = a[0] - a[2];
    cplx<T> b1 = a[1] + a[3], b3 = rot90<T, DIR>(a[1] - a[3]);
    a[0] = b0 + b1; a[1] = b0 - b1; a[2] = b2 + b3; a[3] = b2 - b3;
}
template <typename T, int DIR> QI_DEV void dif8(cplx<T>* a) {
    cplx<T> b0 = a[0] + a[4], b4 = a[0] - a[4];
    cplx<T> b1 = a[1] + a[5], b5 = rot45<T, DIR>(a[1] - a[5]);
    cplx<T> b2 = a[2] + a[6], b6 = rot90<T, DIR>(a[2] - a[6]);
    cplx<T> b3 = a[3] + a[7], b7 = rot135<T, DIR>(a[3] - a[7]);
    cplx<T> c0 = b0 + b2, c2 = b0 - b2, c1 = b1 + b3, c3 = rot90<T, DIR>(b1 - b3);
    cplx<T> c4 = b4 + b6, c6 = b4 - b6, c5 = b5 + b7, c7 = rot90<T, DIR>(b5 - b7);
    a[0] = c0 + c1; a[1] = c0 - c1; a[2] = c2 + c3; a[3] = c2 - c3;
    a[4] = c4 + c5; a[5] = c4 - c5; a[6] = c6 + c7; a[7] = c6 - c7;
}
// DIT butterflies: bit-reversed slots in, natural slots out (exact mirror of the above).
template <typename T, int DIR> QI_DEV void dit2(cplx<T>* a) {
    cplx<T> t = a[0] - a[1]; a[0] = a[0] + a[1]; a[1] = t;
}
template <typename T, int DIR> QI_DEV void dit4(cplx<T>* a) {
    cplx<T> b0 = a[0] + a[1], b1 = a[0] - a[1];
    cplx<T> b2 = a[2] + a[3], b3 = rot90<T, DIR>(a[2] - a[3]);
    a[0] = b0 + b2; a[2] = b0 - b2; a[1] = b1 + b3; a[3] = b1 - b3;
}
template <typename T, int DIR> QI_DEV void dit8(cplx<T>* a) {
    // slots: a[brev3(f)] holds frequency-ordered input f
    cplx<T> c0 = a[0] + a[1], c1 = a[0] - a[1];
    cplx<T> c2 = a[2] + a[3], c3 = rot90<T, DIR>(a[2] - a[3]);
    cplx<T> c4 = a[4] + a[5], c5 = a[4] - a[5];
    cplx<T> c6 = a[6] + a[7], c7 = rot90<T, DIR>(a[6] - a[7]);
    cplx<T> b0 = c0 + c2, b2 = c0 - c2, b1 = c1 + c3, b3 = c1 - c3;
    cplx<T> b4 = c4 + c6, b6 = rot90<T, DIR>(c4 - c6);
    cplx<T> b5 = rot45<T, DIR>(c5 + c7), b7 = rot135<T, DIR>(c5 - c7);
    a[0] = b0 + b4; a[4] = b0 - b4; a[1] = b1 + b5; a[5] = b1 - b5;
    a[2] = b2 + b6; a[6] = b2 - b6; a[3] = b3 + b7; a[7] = b3 - b7;
}

// radix 16 = one radix-2 step around two radix-8 halves.  * w16^n for the odd n (n = 1, 3, 5, 7, sign by DIR):
template <typename T, int DIR, int N> QI_DEV cplx<T> rot16(cplx<T> a) {
    const T c = (T)0.92387953251128675613, s = (T)0.38268343236508977173;     // cos, sin (pi / 8)
    const T wr = N == 1 ? c : (N == 3 ? s : (N == 5 ? -s : -c));
    const T wi = N == 1 ? s : (N == 3 ? c : (N == 5 ? c : s));
    return DIR == FFT_FWD ? mk<T>(a.re * wr + a.im * wi, a.im * wr - a.re * wi)
                          : mk<T>(a.re * wr - a.im * wi, a.im * wr + a.re * wi);
}
// natural slots in, bit-reversed slots out: a[brev4(f)] = frequency f.  Slots 0..7 hold the even frequencies in brev3
// order (brev4(2m) = brev3(m)), slots 8..15 the odd ones (brev4(2m + 1) = 8 + brev3(m)).
template <typename T, int DIR> QI_DEV void dif16(cplx<T>* a) {
    cplx<T> d[8];
#pragma unroll
    for (int n = 0; n < 8; ++n) { d[n] = a[n] - a[n + 8]; a[n] = a[n] + a[n + 8]; }
    d[1] = rot16<T, DIR, 1>(d[1]); d[2] = rot45<T, DIR>(d[2]); d[3] = rot16<T, DIR, 3>(d[3]);
    d[4] = rot90<T, DIR>(d[4]);
    d[5] = rot16<T, DIR, 5>(d[5]); d[6] = rot135<T, DIR>(d[6]); d[7] = rot16<T, DIR, 7>(d[7]);
    dif8<T, DIR>(a);
    dif8<T, DIR>(d);
#pragma unroll
    for (int n = 0; n < 8; ++n) a[n + 8] = d[n];
}
// bit-reversed slots in, natural slots out (exact mirror of dif16)
template <typename T, int DIR> QI_DEV void dit16(cplx<T>* a) {
    dit8<T, DIR>(a);
    dit8<T, DIR>(a + 8);
    a[9] = rot16<T, DIR, 1>(a[9]); a[10] = rot45<T, DIR>(a[10]); a[11] = rot16<T, DIR, 3>(a[11]);
    a[12] = rot90<T, DIR>(a[12]);
    a[13] = rot16<T, DIR, 5>(a[13]); a[14] = rot135<T, DIR>(a[14]); a[15] = rot16<T, DIR, 7>(a[15]);
#pragma unroll
    for (int n = 0; n < 8; ++n) { const cplx<T> d = a[n] - a[n + 8]; a[n] = a[n] + a[n + 8]; a[n + 8] = d; }
}

QI_HD int brev3(int f) { return ((f & 1) << 2) | (f & 2) | ((f >> 2) & 1); }
QI_HD int brev2(int f) { return ((f & 1) << 1) | ((f >> 1) & 1); }
QI_HD int brev4(int f) { return (brev3(f & 7) << 1) | (f >> 3); }

// ---------------------------------------------------------------- one radix-2^STEP stage on a tile
// tile[r*TP + c], R = 2^logR rows, TC columns; tw[m] = exp(-2*pi*i*m/R), m in [0,R).
// Block size 2^logB, sub-stride h = 2^(logB-STEP).
// STW = true: TC independent single-column tiles, TP elements apart; `tw` is the per-stage table of fill_stage_twiddles
// (lanes run along j: the strided tw[(j * f) << twshift] of the plain table is an 8-way bank conflict per quarter warp).
QI_HD int stage_tw_off(int logR, int logB) {     // radix-8 stages sit at logB = logR - 3k
    int off = 0;
    for (int lb = logR; lb > logB; lb -= 3) off += 7 << (lb - 3);
    return off;
}
// STW also selects the single-column tile layout phys(r) = r + (r >> 3) (pad8): with lanes along the block offset j the
// plain layout puts the 32 / h blocks a warp touches in stages with h < 32 a multiple of 512 B apart -- an 8-way conflict
// on 16-byte elements; with one padding slot per 8 rows every stage of a 2^m-point transform is conflict free.
QI_HD int pad8(int r) { return r + (r >> 3); }
// The slot of row r for elements of cplx<T>.  16-byte elements (double): one padding slot per 8 rows -- a quarter warp is
// the unit of a 128-bit access.  8-byte elements (float): the unit is the half warp, and one slot per 8 rows makes 16
// consecutive rows wrap onto their own first bank pair (ncu: 2x the wavefronts in every stage with h >= 16 and in every
// row-contiguous pass); TWO slots per 16 rows keep 16 consecutive rows, the 8 x 2 rows of the h = 2 stage, the 4 x 4 of
// h = 4 and the 2 x 8 of h = 8 on distinct bank pairs.  Same footprint: pad8(R) slots for R a multiple of 16.
template <typename T> QI_HD int padt(int r) { return sizeof(T) == 4 ? r + 2 * (r >> 4) : r + (r >> 3); }
template <typename T, int DIR, int STEP, bool STW = false>
QI_DEV void tile_stage(cplx<T>* tile, const cplx<T>* tw, int logR, int logB, int TC, int TP) {
    constexpr int Q = 1 << STEP;
    const int logH = logB - STEP;
    const int h = 1 << logH;
    const int ntask = (1 << (logR - STEP)) * TC;
    const int logTC = 31 - __clz(TC);
    const int twshift = logR - logB;
    const cplx<T>* tws = STW ? tw + stage_tw_off(logR, logB) - h : tw;      // slot s of block offset j: tws[s * h + j]
    for (int task = threadIdx.x; task < ntask; task += blockDim.x) {
        const int c = task & (TC - 1);              // TC is a power of two
        const int u = task >> logTC;
        const int j = u & (h - 1);
        const int g = u >> logH;
        if (STW) {
            // TC independent single-column tiles TP elements apart, padded rows, per-stage twiddle tables; the lanes of a
            // warp run along the butterflies of ONE tile (task = tile * butterflies + butterfly)
            const int logPer = logR - STEP;
            const int uu = task & ((1 << logPer) - 1);
            cplx<T>* tl = tile + (size_t)(task >> logPer) * TP;
            const int jj = uu & (h - 1);
            const int r0 = ((uu >> logH) << logB) + jj;
            if (STEP == 1 && (sizeof(T) == 8 || (TP & 1) == 0)) {
                // the radix-2 remainder stage (h = 1): rows 2 uu and 2 uu + 1 are neighbours in the padded layout, one
                // vector access each way instead of two (which a half warp could only serve in twice the wavefronts)
                struct __align__(16) Pair { cplx<T> x, y; };        // float: needs an even tile pitch
                Pair* pp = reinterpret_cast<Pair*>(tl + padt<T>(r0));
                Pair v = *pp;
                const cplx<T> d = v.x - v.y;
                v.x = v.x + v.y; v.y = d;
                *pp = v;
                continue;
            }
            cplx<T> a[Q];
            if (DIR == FFT_FWD) {
#pragma unroll
                for (int i = 0; i < Q; ++i) a[i] = tl[padt<T>(r0 + i * h)];
                if (STEP == 3) dif8<T, DIR>(a); else if (STEP == 2) dif4<T, DIR>(a); else dif2<T, DIR>(a);
#pragma unroll
                for (int s = 0; s < Q; ++s) {
                    cplx<T> v = a[s];
                    if (s != 0 && STEP == 3 && logH > 0) v = v * tws[s * h + jj];
                    tl[padt<T>(r0 + s * h)] = v;
                }
            } else {
#pragma unroll
                for (int s = 0; s < Q; ++s) {
                    cplx<T> v = tl[padt<T>(r0 + s * h)];
                    if (s != 0 && STEP == 3 && logH > 0) v = mul_conj(v, tws[s * h + jj]);
                    a[s] = v;
                }
                if (STEP == 3) dit8<T, DIR>(a); else if (STEP == 2) dit4<T, DIR>(a); else dit2<T, DIR>(a);
#pragma unroll
                for (int i = 0; i < Q; ++i) tl[padt<T>(r0 + i * h)] = a[i];
            }
            continue;
        }
        cplx<T>* p = tile + (size_t)(((g << logB) + j) * TP + c);
        const int stride = h * TP;
        cplx<T> a[Q];
        if (DIR == FFT_FWD) {
#pragma unroll
            for (int i = 0; i < Q; ++i) a[i] = p[i * stride];
            if (STEP == 3) dif8<T, DIR>(a); else if (STEP == 2) dif4<T, DIR>(a); else dif2<T, DIR>(a);
#pragma unroll
            for (int s = 0; s < Q; ++s) {
                const int f = STEP == 3 ? brev3(s) : (STEP == 2 ? brev2(s) : s);
                cplx<T> v = a[s];
                if (f != 0) v = v * tw[(j * f) << twshift];
                p[s * stride] = v;
            }
        } else {
#pragma unroll
            for (int s = 0; s < Q; ++s) {
                const int f = STEP == 3 ? brev3(s) : (STEP == 2 ? brev2(s) : s);
                cplx<T> v = p[s * stride];
                if (f != 0) v = mul_conj(v, tw[(j * f) << twshift]);
                a[s] = v;
            }
            if (STEP == 3) dit8<T, DIR>(a); else if (STEP == 2) dit4<T, DIR>(a); else dit2<T, DIR>(a);
#pragma unroll
            for (int i = 0; i < Q; ++i) p[i * stride] = a[i];
        }
    }
}

// Full tile FFT.  All threads of the CTA must call it; it ends with a __syncthreads().
template <typename T, int DIR, bool STW = false>
QI_DEV void tile_fft(cplx<T>* tile, const cplx<T>* tw, int logR, int TC, int TP) {
    if (logR == 0) { __syncthreads(); return; }
    const int rem = logR % 3;            // the odd-sized stage sits at the small-block end
    if (DIR == FFT_FWD) {
        int logB = logR;
        while (logB >= 3 && logB - 3 >= rem) {
            tile_stage<T, DIR, 3, STW>(tile, tw, logR, logB, TC, TP);
            __syncthreads();
            logB -= 3;
        }
        if (logB == 2) { tile_stage<T, DIR, 2, STW>(tile, tw, logR, 2, TC, TP); __syncthreads(); }
        else if (logB == 1) { tile_stage<T, DIR, 1, STW>(tile, tw, logR, 1, TC, TP); __syncthreads(); }
    } else {
        int logB = rem;
        if (rem == 2) { tile_stage<T, DIR, 2, STW>(tile, tw, logR, 2, TC, TP); __syncthreads(); }
        else if (rem == 1) { tile_stage<T, DIR, 1, STW>(tile, tw, logR, 1, TC, TP); __syncthreads(); }
        while (logB < logR) {
            logB += 3;
            tile_stage<T, DIR, 3, STW>(tile, tw, logR, logB, TC, TP);
            __syncthreads();
        }
    }
}

// per-stage twiddles of the radix-8 stages, contiguous in the block offset j: entry stage_tw_off(logR, logB) + (s - 1) h + j
// = exp(-2 pi i j brev3(s) / 2^logB), h = 2^(logB - 3).  Fewer than 2^logR entries in total.  (The radix-4 / radix-2
// stage of lengths that are not a power of 8 sits at the small-block end, where every twiddle is 1.)
template <typename T> QI_DEV void fill_stage_twiddles(cplx<T>* tw, int logR) {
    for (int logB = logR; logB >= 3 && logB - 3 >= logR % 3; logB -= 3) {
        const int logH = logB - 3, h = 1 << logH;
        cplx<T>* dst = tw + stage_tw_off(logR, logB);
        for (int e = threadIdx.x; e < 7 * h; e += blockDim.x) {
            const int s = (e >> logH) + 1, j = e & (h - 1);
            dst[e] = conj(unit_root<T>((unsigned long long)(j * brev3(s)), logB));
        }
    }
}

// fill tw[m] = exp(-2*pi*i*m/R)
template <typename T> QI_DEV void fill_twiddles(cplx<T>* tw, int logR) {
    const int R = 1 << logR;
    for (int m = threadIdx.x; m < R; m += blockDim.x) tw[m] = conj(unit_root<T>((unsigned long long)m, logR));
}
// The same table from 2 sqrt(R) exact roots and one complex product per entry (a sincospi per entry was a tenth of a
// pass's instructions in float64).  `scratch` holds 2^lo + 2^(logR-lo) entries and must not overlap tw; two barriers inside.
template <typename T> QI_DEV void fill_twiddles_fast(cplx<T>* tw, int logR, cplx<T>* scratch) {
    if (logR < 6) { fill_twiddles<T>(tw, logR); return; }
    const int lo = logR >> 1, nlo = 1 << lo, nhi = 1 << (logR - lo);
    for (int j = threadIdx.x; j < nlo + nhi; j += blockDim.x)
        scratch[j] = conj(unit_root<T>(j < nlo ? (unsigned long long)j : ((unsigned long long)(j - nlo) << lo), logR));
    __syncthreads();
    for (int m = threadIdx.x; m < (1 << logR); m += blockDim.x) tw[m] = scratch[m & (nlo - 1)] * scratch[nlo + (m >> lo)];
    __syncthreads();
}

// ---------------------------------------------------------------- pass geometry
struct PassGeom {
    int logR;        // rows per FFT = 2^logR
    int logS;        // row stride in elements = 2^logS (bits below this pass)
    int logL;        // total transform length 2^logL
    int TC;          // tile columns
    // column id c in [0, L/R): outer = c >> logS, inner = c & (S-1); element = outer*R*S + r*S + inner
};

QI_HD i64 pass_elem(const PassGeom& g, int r, i64 col) {
    const i64 inner = col & ((1ll << g.logS) - 1);
    const i64 outer = col >> g.logS;
    return (outer << (g.logR + g.logS)) + ((i64)r << g.logS) + inner;
}

// Generic pass kernel.
//   Src:  cplx<T> load(i64 batch, i64 elem) const
//   Dst:  void store(i64 batch, i64 elem, cplx<T> v);  void finish(i64 batch, unsigned char* scratch)
// grid = (tiles_per_batch, batches); block = 256; dyn smem = (R*TP + R) * sizeof(cplx<T>) (+ Dst scratch)
template <typename T, int DIR, class Src, class Dst>
__global__ void __launch_bounds__(256)
fft_pass_kernel(PassGeom g, Src src, Dst dst) {
    QI_DYN_SMEM(smem_raw);
    const int R = 1 << g.logR;
    const int TC = g.TC, TP = g.TC + 1;
    cplx<T>* tile = reinterpret_cast<cplx<T>*>(smem_raw);
    cplx<T>* tw = tile + (size_t)R * TP;
    const i64 batch = blockIdx.y;
    const i64 col0 = (i64)blockIdx.x * TC;
    const int nelem = R * TC;
    const int logTC = 31 - __clz(TC);
    const int twlog = g.logR + g.logS;           // modulus of the inter-pass twiddle

    fill_twiddles_fast<T>(tw, g.logR, tile);

    const bool row_major = (g.logS == 0);        // rows contiguous in memory -> lanes along r
    // Cooley-Tukey twiddle between the passes, W^(inner * k) with W = exp(2 pi i / 2^twlog), k = brev(r).  A thread keeps
    // its column (256 is a multiple of TC) and visits the rows r0 + i * RPI, so k = k_hi(r0) + k_lo(i) and the twiddle
    // factors into a per-thread constant W^(inner k_hi) and a CTA-wide table xtw[i][c] = W^(inner_c k_lo(i)): one shared
    // load and one complex product per element instead of a sincospi (a third of a float32 pass, half of a float64 one).
    cplx<T>* xtw = tw + R;
    const int lr0 = 8 - logTC;                                   // log2 of the rows per 256-thread sweep
    const bool fact = !row_major && (int)blockDim.x == 256 && g.logR >= lr0;
    const int logNI = g.logR - lr0, NI = fact ? 1 << logNI : 0;
    cplx<T> tw_thread = mk<T>((T)1, (T)0);
    if (fact) {
        for (int e = threadIdx.x; e < TC * NI; e += blockDim.x) {
            const int c = e & (TC - 1), i = e >> logTC;           // [i][c]: the lanes of a warp read consecutive entries
            const unsigned long long inner = (unsigned long long)((col0 + c) & ((1ll << g.logS) - 1));
            xtw[e] = unit_root<T>(inner * brev_bits((unsigned)i, logNI), twlog);
        }
        const int c = threadIdx.x & (TC - 1), r0 = threadIdx.x >> logTC;
        const unsigned long long inner = (unsigned long long)((col0 + c) & ((1ll << g.logS) - 1));
        const unsigned long long k_hi = (unsigned long long)brev_bits((unsigned)r0, lr0) << logNI;
        tw_thread = unit_root<T>((inner * k_hi) & ((1ull << twlog) - 1ull), twlog);
        __syncthreads();
    }
    constexpr int LU = QI_FFT_LOADS_IN_FLIGHT;
    for (int base = threadIdx.x; base < nelem; base += blockDim.x * LU) {
        cplx<T> v[LU];
#pragma unroll
        for (int u = 0; u < LU; ++u) {
            const int idx = base + u * (int)blockDim.x;
            if (idx < nelem) {
                int r, c;
                if (row_major) { r = idx & (R - 1); c = idx >> g.logR; }
                else { c = idx & (TC - 1); r = idx >> logTC; }
                v[u] = src.load(batch, pass_elem(g, r, col0 + c));
            }
        }
#pragma unroll
        for (int u = 0; u < LU; ++u) {
            const int idx = base + u * (int)blockDim.x;
            if (idx < nelem) {
                int r, c;
                if (row_major) { r = idx & (R - 1); c = idx >> g.logR; }
                else { c = idx & (TC - 1); r = idx >> logTC; }
                const i64 col = col0 + c;
                cplx<T> w = v[u];
                if (DIR == FFT_INV && g.logS > 0) {
                    if (fact) {
                        w = w * (xtw[((idx >> 8) << logTC) + c] * tw_thread);
                    } else {
                        const unsigned long long inner = (unsigned long long)(col & ((1ll << g.logS) - 1));
                        const unsigned k = brev_bits((unsigned)r, g.logR);
                        if (inner * k) w = mul_conj(w, conj(unit_root<T>(inner * k, twlog)));
                    }
                }
                tile[r * TP + c] = w;
            }
        }
    }
    __syncthreads();
    tile_fft<T, DIR>(tile, tw, g.logR, TC, TP);
    for (int idx = threadIdx.x; idx < nelem; idx += blockDim.x) {
        int r, c;
        if (row_major) { r = idx & (R - 1); c = idx >> g.logR; }
        else { c = idx & (TC - 1); r = idx >> logTC; }
        const i64 col = col0 + c;
        const i64 e = pass_elem(g, r, col);
        cplx<T> v = tile[r * TP + c];
        if (DIR == FFT_FWD && g.logS > 0) {
            if (fact) {
                v = mul_conj(v, xtw[((idx >> 8) << logTC) + c] * tw_thread);
            } else {
                const unsigned long long inner = (unsigned long long)(col & ((1ll << g.logS) - 1));
                const unsigned k = brev_bits((unsigned)r, g.logR);
                if (inner * k) v = mul_conj(v, unit_root<T>(inner * k, twlog));
            }
        }
        dst.store(batch, e, v);
    }
    dst.finish(batch, reinterpret_cast<unsigned char*>(xtw + TC * NI));
}

// ---------------------------------------------------------------- host-side plan
struct FftPlan {
    int logL;
    int npass;
    int logR[4];     // forward order: pass 0 handles the TOP bits of the index
    int logS[4];
    int TC[4];
};

// max rows per pass chosen so that R*(TC+1)*sizeof(cplx) stays <= ~100 KB with TC >= 8
inline FftPlan make_plan(int logL, int elem_bytes /* sizeof(cplx<T>) */) {
    FftPlan p;
    p.logL = logL;
    const int maxlog = 10;  // 1024 rows per pass
    int np = (logL + maxlog - 1) / maxlog;
    if (np < 1) np = 1;
    p.npass = np;
    int rem = logL;
    int below = logL;
    for (int i = 0; i < np; ++i) {
        int lr = (rem + (np - i) - 1) / (np - i);   // balanced split, larger first
        p.logR[i] = lr;
        below -= lr;
        p.logS[i] = below;
        rem -= lr;
        // tile columns: target ~96 KB tile, power of two, between 1 and 32
        long budget = QI_FFT_TILE_BUDGET_KB * 1024 / elem_bytes;
        int tc = 1;
        while (tc < 32 && (long)(1 << lr) * (2 * tc + 1) <= budget) tc *= 2;
        long ncols = 1l << (logL - lr);
        while (tc > ncols) tc /= 2;
        if (tc < 1) tc = 1;
        p.TC[i] = tc;
    }
    return p;
}

template <typename T> inline size_t pass_smem_bytes(int logR, int TC, size_t dst_scratch) {
    // tile + stage twiddles + the inter-pass twiddle table xtw[TC][R * TC / 256] of fft_pass_kernel
    const size_t xtw = ((size_t)(1 << logR) * TC * TC + 255) / 256;
    return ((size_t)(1 << logR) * (TC + 1) + (size_t)(1 << logR) + xtw) * sizeof(cplx<T>) + dst_scratch;
}

// Launch one pass.  `pass` indexes the FORWARD order; an inverse transform runs passes npass-1 .. 0.
template <typename T, int DIR, class Src, class Dst>
inline void launch_pass(const FftPlan& plan, int pass, i64 nbatch, Src src, Dst dst, size_t dst_scratch,
                        cudaStream_t stream) {
    PassGeom g;
    g.logR = plan.logR[pass];
    g.logS = plan.logS[pass];
    g.logL = plan.logL;
    g.TC = plan.TC[pass];
    const i64 ncols = 1ll << (plan.logL - g.logR);
    dim3 grid((unsigned)(ncols / g.TC), (unsigned)nbatch, 1);
    const size_t smem = pass_smem_bytes<T>(g.logR, g.TC, dst_scratch);
#ifndef QI_EMUL
    cudaFuncSetAttribute(fft_pass_kernel<T, DIR, Src, Dst>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
#endif
    QI_LAUNCH((fft_pass_kernel<T, DIR, Src, Dst>), grid, dim3(256), smem, stream, g, src, dst);
}

// ---------------------------------------------------------------- plain sources / sinks
template <typename T> struct SrcComplex {
    const cplx<T>* buf; i64 batch_stride;
    QI_DEV cplx<T> load(i64 b, i64 e) const { return buf[b * batch_stride + e]; }
};
template <typename T> struct DstComplex {
    cplx<T>* buf; i64 batch_stride; T scale;
    QI_DEV void store(i64 b, i64 e, cplx<T> v) const { buf[b * batch_stride + e] = v * scale; }
    QI_DEV void finish(i64, unsigned char*) const {}
};
// real input of n_points per batch row, zero-extended to 2^logL
template <typename T> struct SrcRealPad {
    const T* sig; i64 batch_stride; i64 n_points;
    QI_DEV cplx<T> load(i64 b, i64 e) const {
        return mk<T>(e < n_points ? sig[b * batch_stride + e] : (T)0, (T)0);
    }
};

// ---------------------------------------------------------------- whole transforms
// Forward transform of `nbatch` rows into `buf` (row stride `stride`, bit-reversed order): pass 0 reads `src`, the later
// passes run on `buf` in place.
template <typename T, class Src>
inline void forward_passes(const FftPlan& plan, i64 nbatch, Src src, cplx<T>* buf, i64 stride, cudaStream_t st) {
    const DstComplex<T> d{buf, stride, (T)1};
    launch_pass<T, FFT_FWD>(plan, 0, nbatch, src, d, 0, st);
    for (int p = 1; p < plan.npass; ++p) launch_pass<T, FFT_FWD>(plan, p, nbatch, SrcComplex<T>{buf, stride}, d, 0, st);
}

// Inverse transform of `nbatch` rows: the first pass (npass - 1) reads `src`, the last (0) writes `dst` with
// `dst_scratch` bytes of sink scratch, and the passes between run on `buf` (row stride `stride`) in place.  The last pass
// is timed as QI_CAT_INV_LAST when its sink writes the output planes (`dst_is_output`).
template <typename T, class Src, class Dst>
inline void inverse_passes(const FftPlan& plan, i64 nbatch, Src src, Dst dst, size_t dst_scratch, bool dst_is_output,
                           cplx<T>* buf, i64 stride, cudaStream_t st) {
    const SrcComplex<T> s_mid{buf, stride};
    const DstComplex<T> d_mid{buf, stride, (T)1};
    for (int p = plan.npass - 1; p >= 0; --p) {
        const bool first = (p == plan.npass - 1), last = (p == 0);
        prof_set_category(last && dst_is_output ? QI_CAT_INV_LAST : (first ? QI_CAT_INV_FIRST : QI_CAT_INV_MID));
        if (first && last) launch_pass<T, FFT_INV>(plan, p, nbatch, src, dst, dst_scratch, st);
        else if (first) launch_pass<T, FFT_INV>(plan, p, nbatch, src, d_mid, 0, st);
        else if (last) launch_pass<T, FFT_INV>(plan, p, nbatch, s_mid, dst, dst_scratch, st);
        else launch_pass<T, FFT_INV>(plan, p, nbatch, s_mid, d_mid, 0, st);
    }
}

}  // namespace qi
