// qi_stft.cu -- short-time Fourier transform / Welch on the shared FFT tile core.
//
// One CTA transforms 2*TC consecutive frames of one channel: frames are gathered from the (virtually
// zero-extended) record straight into shared memory, two real frames packed into one complex column,
// the per-frame mean removed, the periodic window applied, one radix-8 tile FFT run, the two spectra
// separated with the Hermitian split and the one-sided bins stored with time as the fastest axis (the
// layout scipy returns).  Frames too long for one CTA take multi-pass FFTs of frame pairs instead (the long-frame route
// below).  Replaces scipy.signal.stft / welch as called by
// quantum_inferno/styx_fft.py:175-187, :215-227, :254-266, and scipy.signal.ShortTimeFFT.stft_detrend / spectrogram /
// istft as called by quantum_inferno/utilities/short_time_fft.py:64-175.
#include "qi_fft.cuh"
#include "qi_host.h"
#include "qi_reduce.cuh"

namespace qi {

// log2(n) of a power of two n, else -1
static int log2_pow2(int n) {
    if (n <= 0 || (n & (n - 1))) return -1;
    int l = 0;
    while ((1 << l) < n) ++l;
    return l;
}

struct StftGeom {
    i64 n_points, sig_stride, n_frames;
    int nperseg, hop, logF, pad_left, TC, detrend, roll;
    double scale;
};

// float32: two 512-thread CTAs per SM (8 tile columns at nfft = 1024); float64: one 1024-thread CTA with twice the tile
// columns -- measured 1.12 -> 1.03 ms on 64 x 2^20 (the 16-byte elements suffer most from the 2x shared-memory
// wavefronts of narrow tiles), while float32 measured the same either way (0.534 / 0.530 ms).
template <typename T> struct StftLaunch {
    static constexpr int threads = sizeof(T) == 8 ? 1024 : 512;
    static constexpr int min_ctas = sizeof(T) == 8 ? 1 : 2;
    static constexpr size_t budget = sizeof(T) == 8 ? 200 * 1024 : 100 * 1024;
};
// pitch (elements) between the single-column tiles of the STFT kernels: the padded tile plus an offset that puts the lanes
// of the Hermitian split (which run along the tiles) on different banks -- one 16-byte element for double; two 8-byte
// elements for float, which also keeps every tile 16-byte aligned for the vector accesses of the radix-2 stage
template <typename T> QI_HD int stft_tile_pitch(int R) { return sizeof(T) == 8 ? (pad8(R) | 1) : pad8(R) + 2; }

// Hermitian split of the spectrum Z = Xa + i Xb of two real frames a, b (z1 = Z[k], z2 = Z[nfft - k]) into bin k of both
// frames, times exp(+2 pi i k roll / nfft): the segment rotated left by roll samples (roll in [0, nfft))
template <typename T>
QI_DEV void pair_split(cplx<T> z1, cplx<T> z2, int k, int roll, int logF, cplx<T>& xa, cplx<T>& xb) {
    const int R = 1 << logF;
    xa = mk<T>((T)0.5 * (z1.re + z2.re), (T)0.5 * (z1.im - z2.im));
    xb = mk<T>((T)0.5 * (z1.im + z2.im), (T)-0.5 * (z1.re - z2.re));
    if (roll) {
        const cplx<T> ph = unit_root<T>((unsigned long long)(((i64)k * roll) & (R - 1)), logF);
        xa = xa * ph; xb = xb * ph;
    }
}

// Hermitian completion, the inverse of pair_split: bin k <= nfft / 2 of frames a and b, the roll undone, gives
// zk = Z[k] and zp = Z[nfft - k].  Bins 0 and nfft / 2 are their own partners and lose their imaginary parts, as in
// irfft: for them the result is false and zp is not to be stored.
template <typename T>
QI_DEV bool pair_complete(cplx<T> xa, cplx<T> xb, int k, int roll, int logF, cplx<T>& zk, cplx<T>& zp) {
    const int R = 1 << logF;
    if (roll) {
        const cplx<T> ph = conj(unit_root<T>((unsigned long long)(((i64)k * roll) & (R - 1)), logF));
        xa = xa * ph; xb = xb * ph;
    }
    const bool partner = k != 0 && k != R / 2;
    zk = partner ? mk<T>(xa.re - xb.im, xa.im + xb.re) : mk<T>(xa.re, xb.re);
    zp = mk<T>(xa.re + xb.im, xb.re - xa.im);
    return partner;
}

// LOGF / LOGTC > 0: FFT length and tiles per CTA known at compile time (the common sizes: every index computation of the
// gather, the stage loops and the Hermitian split folds to shifts and immediates; ncu of the generic kernel had a third of
// its instructions in integer index arithmetic); 0: taken from the geometry at run time.
template <typename T, int LOGF, int LOGTC>
__global__ void __launch_bounds__(StftLaunch<T>::threads, StftLaunch<T>::min_ctas)
stft_kernel(const T* __restrict__ sig, const T* __restrict__ window, StftGeom g0, cplx<T>* __restrict__ out,
            double* __restrict__ psd_acc) {
    QI_DYN_SMEM(smem_raw);
    StftGeom g = g0;
    if (LOGF > 0) { g.logF = LOGF; g.TC = 1 << LOGTC; }
    const int R = 1 << g.logF;
    // TC single-column tiles (two real frames each) in the padded layout of tile_fft<.., true>, PT elements apart
    const int TC = g.TC, PT = stft_tile_pitch<T>(R);
    const int logTC = 31 - __clz(TC);
    cplx<T>* tile = reinterpret_cast<cplx<T>*>(smem_raw);
    cplx<T>* tw = tile + (size_t)TC * PT;
    T* means = reinterpret_cast<T*>(tw + R);              // 2*TC means
    double* bsum = reinterpret_cast<double*>(means + 2 * TC);   // 2*TC + 16 hop-block sums (fused path)
    const i64 chan = blockIdx.y;
    const i64 frame0 = (i64)blockIdx.x * (2 * TC);
    const T* x = sig + chan * g.sig_stride;

    fill_stage_twiddles<T>(tw, g.logF);
    // gather (lanes along the sample axis -> coalesced global reads)
    // interior CTAs (every frame exists and lies inside the record) take the path without bounds checks
    const i64 first = frame0 * g.hop - g.pad_left;
    const bool interior = frame0 + 2 * TC <= g.n_frames && first >= 0 &&
                          first + (i64)(2 * TC - 1) * g.hop + g.nperseg <= g.n_points &&
                          (i64)(2 * TC - 1) * g.hop + R < (1ll << 30);
    // Interior CTAs whose frames are whole numbers of hops apart make the frame means first (sums of hop-sized blocks
    // of the span, one warp per block, every sample read once more from L1 / L2) and then gather (x - mean) * window
    // straight into the tile: no separate mean and window passes over shared memory.
    const int hops_per_frame = g.nperseg / g.hop;
    // Compile-time sizes with at least one tile row per thread: a thread owns the rows r = tid + NT k of EVERY tile, so its
    // window values sit in registers, its 2 TC R / NT samples (32 floats / 16 doubles) are requested in one go with
    // lanes along the samples, the frame sums come from those registers (warp shuffles in the arithmetic type, fp64
    // across the warps), and (x - mean) * window goes straight into the tiles.  Any hop, any nperseg <= R.
    constexpr int NT = StftLaunch<T>::threads;
    constexpr bool REG_GATHER = LOGF > 0 && (1 << (LOGF > 0 ? LOGF : 0)) >= NT;
    bool gathered = false;
    if (REG_GATHER && interior) {
        constexpr int RPT = REG_GATHER ? (1 << LOGF) / NT : 1, TCC = REG_GATHER ? 1 << LOGTC : 1;
        const T* xb0 = x + first;
        const int t = threadIdx.x, warp = t >> 5, lane = t & 31;
        T va[TCC][RPT], vb[TCC][RPT], wv[RPT];
#pragma unroll
        for (int k = 0; k < RPT; ++k) {
            const int r = t + NT * k;
            const bool in = r < g.nperseg;
            wv[k] = in ? window[r] : (T)0;
#pragma unroll
            for (int c = 0; c < TCC; ++c) {
                const T* pa = xb0 + (i64)(2 * c) * g.hop + r;
                va[c][k] = in ? pa[0] : (T)0;
                vb[c][k] = in ? pa[g.hop] : (T)0;
            }
        }
        double* wsums = reinterpret_cast<double*>(tile);          // [warps][2 TCC]; the tiles are written after the means
        if (g.detrend) {
#pragma unroll
            for (int c = 0; c < TCC; ++c) {
                T sa = (T)0, sb = (T)0;
#pragma unroll
                for (int k = 0; k < RPT; ++k) { sa += va[c][k]; sb += vb[c][k]; }
                sa = warp_sum(sa); sb = warp_sum(sb);
                if (lane == 0) { wsums[warp * 2 * TCC + 2 * c] = (double)sa; wsums[warp * 2 * TCC + 2 * c + 1] = (double)sb; }
            }
        }
        __syncthreads();
        if (t < 2 * TCC) {
            double sm = 0.0;
            if (g.detrend) for (int w = 0; w < NT / 32; ++w) sm += wsums[w * 2 * TCC + t];
            means[t] = (T)(sm / (double)g.nperseg);
        }
        __syncthreads();
#pragma unroll
        for (int c = 0; c < TCC; ++c) {
            const T m0 = means[2 * c], m1 = means[2 * c + 1];
#pragma unroll
            for (int k = 0; k < RPT; ++k)
                tile[c * PT + padt<T>(t + NT * k)] = mk<T>((va[c][k] - m0) * wv[k], (vb[c][k] - m1) * wv[k]);
        }
        gathered = true;
    }
    const bool fused = !gathered && interior && hops_per_frame * g.hop == g.nperseg && hops_per_frame <= 16;
    if (fused) {
        const T* xb0 = x + first;
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
        const int nblk = 2 * TC - 1 + hops_per_frame;
        if (g.detrend) {
            for (int blk = warp; blk < nblk; blk += nw) {
                const T* pb = xb0 + (i64)blk * g.hop;
                double s0 = 0.0, s1 = 0.0;
                int i = lane;
                for (; i + 32 < g.hop; i += 64) { s0 += (double)pb[i]; s1 += (double)pb[i + 32]; }
                if (i < g.hop) s0 += (double)pb[i];
                const double s = warp_sum(s0 + s1);
                if (lane == 0) bsum[blk] = s;
            }
        }
        __syncthreads();
        if (threadIdx.x < 2 * TC) {
            double s = 0.0;
            if (g.detrend) for (int j = 0; j < hops_per_frame; ++j) s += bsum[threadIdx.x + j];
            means[threadIdx.x] = (T)(s / (double)g.nperseg);
        }
        __syncthreads();
    }
    if (gathered) {
        // tiles are complete (registers path above)
    } else if (interior) {
        // eight (frame a, frame b) sample pairs per thread are requested before the first is stored: the gather is the
        // only HBM-latency-bound phase of the kernel and needs the loads in flight, not one dependent pair per trip
        const T* xb0 = x + first;
        constexpr int GU = 8;
        const int total_g = R * TC;
        for (int base = threadIdx.x; base < total_g; base += blockDim.x * GU) {
            T va[GU], vb[GU];
#pragma unroll
            for (int u = 0; u < GU; ++u) {
                const int idx = base + u * (int)blockDim.x;
                const int r = idx & (R - 1);
                const int c = idx >> g.logF;
                va[u] = (T)0; vb[u] = (T)0;
                if (idx < total_g && r < g.nperseg) {
                    const int o = 2 * c * g.hop + r;
                    va[u] = xb0[o];
                    vb[u] = xb0[o + g.hop];
                }
            }
#pragma unroll
            for (int u = 0; u < GU; ++u) {
                const int idx = base + u * (int)blockDim.x;
                if (idx < total_g) {
                    const int r = idx & (R - 1), c = idx >> g.logF;
                    cplx<T> v = mk<T>(va[u], vb[u]);
                    if (fused && r < g.nperseg) {
                        const T w = window[r];
                        v.re = (v.re - means[2 * c]) * w;
                        v.im = (v.im - means[2 * c + 1]) * w;
                    }
                    tile[c * PT + padt<T>(r)] = v;
                }
            }
        }
    } else {
        for (int idx = threadIdx.x; idx < R * TC; idx += blockDim.x) {
            const int r = idx & (R - 1);
            const int c = idx >> g.logF;
            T va = (T)0, vb = (T)0;
            if (r < g.nperseg) {
                const i64 fa = frame0 + 2 * c, fb = fa + 1;
                const i64 pa = fa * g.hop + r - g.pad_left, pb = fb * g.hop + r - g.pad_left;
                if (fa < g.n_frames && pa >= 0 && pa < g.n_points) va = x[pa];
                if (fb < g.n_frames && pb >= 0 && pb < g.n_points) vb = x[pb];
            }
            tile[c * PT + padt<T>(r)] = mk<T>(va, vb);
        }
    }
    __syncthreads();
    // per-frame mean over the nperseg samples (scipy detrend='constant', after the zero extension)
    if (!fused && !gathered) {
        const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
        for (int col = warp; col < 2 * TC; col += nw) {
            double s = 0.0;
            if (g.detrend) {
                const int c = col >> 1;
                for (int r = lane; r < g.nperseg; r += 32) {
                    const cplx<T> v = tile[c * PT + padt<T>(r)];
                    s += (double)((col & 1) ? v.im : v.re);
                }
            }
            s = warp_sum(s);
            if (lane == 0) means[col] = (T)(s / (double)g.nperseg);
        }
        __syncthreads();
        for (int c = 0; c < TC; ++c) {                      // lanes along the samples of one tile
            const T m0 = means[2 * c], m1 = means[2 * c + 1];
            for (int r = threadIdx.x; r < g.nperseg; r += blockDim.x) {
                const T w = window[r];
                cplx<T> v = tile[c * PT + padt<T>(r)];
                v.re = (v.re - m0) * w;
                v.im = (v.im - m1) * w;
                tile[c * PT + padt<T>(r)] = v;
            }
        }
        __syncthreads();
    }
    tile_fft<T, FFT_FWD, true>(tile, tw, g.logF, TC, PT);
    // Hermitian split + store, lanes along frames (time is the fastest output axis)
    const int K = (R >> 1) + 1;
    const T sc = (T)g.scale;
    const int total = K * TC;
    const int padded = (total + (int)blockDim.x - 1) / (int)blockDim.x * (int)blockDim.x;   // whole warps stay converged
    for (int idx = threadIdx.x; idx < padded; idx += blockDim.x) {
        const bool active = idx < total;
        const int c = idx & (TC - 1);
        const int k = active ? idx >> logTC : 0;
        const cplx<T> z1 = tile[c * PT + padt<T>((int)brev_bits((unsigned)k, g.logF))];
        const cplx<T> z2 = tile[c * PT + padt<T>((int)brev_bits((unsigned)((R - k) & (R - 1)), g.logF))];
        cplx<T> xa, xb;
        pair_split<T>(z1, z2, k, g.roll, g.logF, xa, xb);
        const i64 fa = frame0 + 2 * c;
        if (out && active) {
            cplx<T>* o = out + (chan * K + k) * g.n_frames + fa;
            if (interior) { o[0] = xa * sc; o[1] = xb * sc; }
            else {
                if (fa < g.n_frames) o[0] = xa * sc;
                if (fa + 1 < g.n_frames) o[1] = xb * sc;
            }
        }
        if (psd_acc) {
            double p = 0.0;
            if (active && fa < g.n_frames) p += (double)norm2(xa);
            if (active && fa + 1 < g.n_frames) p += (double)norm2(xb);
            // reduce over the TC lanes that share k before touching HBM
            for (int o2 = TC >> 1; o2 > 0; o2 >>= 1) p += __shfl_down_sync(0xffffffffu, p, o2);
            if (active && c == 0) atomicAdd(&psd_acc[chan * K + k], p);
        }
    }
}

// dynamic shared memory of stft_kernel with tc tiles of nfft points
template <typename T> static size_t stft_tile_smem(int nfft, int tc) {
    return ((size_t)stft_tile_pitch<T>(nfft) * tc + nfft) * sizeof(cplx<T>) + 2 * tc * sizeof(T) +
           (2 * tc + 16) * sizeof(double) + 64;
}
// QI_STFT_TILE_MAX_NFFT > 0 sends every longer frame to the long-frame route below (tools/stft_long_probe.py builds such a
// variant to time both routes at the same size); 0: the shared-memory budget alone decides
#ifndef QI_STFT_TILE_MAX_NFFT
#define QI_STFT_TILE_MAX_NFFT 0
#endif
// tiles per CTA of a tile kernel whose dynamic shared memory is smem(nfft, tiles), or 0 when one frame does not fit a CTA
// (the long-frame route): down to 2 tiles within `budget` (~100 KB lets two 512-thread CTAs share an SM), then down to
// one tile in one big CTA of up to 200 KB
static int tile_columns(int nfft, size_t budget, size_t (*smem)(int nfft, int tc)) {
    if (QI_STFT_TILE_MAX_NFFT > 0 && nfft > QI_STFT_TILE_MAX_NFFT) return 0;
    int TC = 16;
    while (TC > 2 && smem(nfft, TC) > budget) TC >>= 1;
    if (smem(nfft, TC) > budget) {
        budget = 200 * 1024;
        while (TC > 1 && smem(nfft, TC) > budget) TC >>= 1;
    }
    return smem(nfft, TC) > budget ? 0 : TC;
}
template <typename T> static int stft_tile_columns(int nfft) {
    return tile_columns(nfft, StftLaunch<T>::budget, stft_tile_smem<T>);
}

// ---------------------------------------------------------------- frames longer than one CTA's shared memory
// The frame lengths stft_kernel / istft_frames_kernel refuse (float32 nfft >= 2^14, float64 >= 2^13) take the multi-pass
// FFT of qi_fft.cuh with the same two-real-frames-per-complex-row packing.  Frame pairs are processed in chunks of npc
// pairs per channel: batch row b = chan * npc + (p - p0) holds pair p (frames 2p, 2p + 1), its spectrum in bit-reversed
// order, nfft elements per row.
//   forward: stft_long_means_kernel (fp64 frame sums) -> forward passes whose first pass gathers (x - mean) * window
//            (SrcStftPair) -> stft_split_kernel (Hermitian split, roll phase, scale, scipy's layout, Welch sums)
//   inverse: istft_gather_kernel (undo the roll, Hermitian-completed Z = Xa + i Xb) -> inverse passes whose last pass
//            applies the dual window (DstIstftPair) -> istft_ola_kernel as for the tile route
// The split and the gather work on aligned blocks of P = STFT_LONG_P storage positions: block brev(c) holds the bins
// c + j nfft / P (j < P), and the Hermitian partners nfft - k of those bins fill the block of residue nfft / P - c.  A CTA
// takes one such block pair for P consecutive frame pairs: contiguous reads along the positions, runs of 2 P consecutive
// frames in the [C, nfft/2+1, n_frames] store.
constexpr int STFT_LONG_LOGP = 5, STFT_LONG_P = 1 << STFT_LONG_LOGP;   // positions per block = frame pairs per CTA

// bytes of workspace per frame pair and channel: the pair spectrum and the two frame means
template <typename T> static size_t stft_long_pair_bytes(int nfft) { return (size_t)nfft * sizeof(cplx<T>) + 2 * sizeof(T); }
// workspace of the forward: 0 on the tile route, else all frame pairs in one chunk
template <typename T> static size_t stft_workspace_bytes(i64 C, i64 n_frames, int nfft) {
    if (stft_tile_columns<T>(nfft)) return 0;
    return (size_t)C * (size_t)((n_frames + 1) / 2) * stft_long_pair_bytes<T>(nfft);
}

// frame pairs per channel in one chunk: all of them, but at most 65535 / C (the C npc batch rows of a launch are grid.y)
static i64 long_pairs_per_chunk(i64 C, i64 n_frames) {
    const i64 npairs = (n_frames + 1) / 2, cap = 65535 / C;
    return npairs < cap ? npairs : cap;
}

// batch row b of a chunk (npc pairs per channel from pair p0 on): its channel and its first frame
struct PairRow { i64 chan, fa; };
QI_DEV PairRow pair_row(i64 b, int npc, i64 p0) {
    const unsigned bu = (unsigned)b;                      // b < 65536 (grid.y)
    return {(i64)(bu / (unsigned)npc), 2 * (p0 + bu % (unsigned)npc)};
}

// mean of frame f0 + blockIdx.x over its nperseg samples of the zero-extended record, summed in fp64 and rounded to T as
// stft_kernel does; frames >= n_frames get 0.  means[chan][gridDim.x]
template <typename T>
__global__ void __launch_bounds__(256)
stft_long_means_kernel(const T* __restrict__ sig, i64 sig_stride, i64 n_points, i64 n_frames, i64 f0, int nperseg,
                       int hop, int pad_left, T* __restrict__ means) {
    __shared__ double scratch[32];
    const i64 chan = blockIdx.y, f = f0 + blockIdx.x;
    const T* x = sig + chan * sig_stride;
    double s0 = 0.0, s1 = 0.0;
    if (f < n_frames) {
        const i64 start = f * hop - pad_left;
        const i64 lo = start > 0 ? start : 0, hi = start + nperseg < n_points ? start + nperseg : n_points;
        i64 i = lo + threadIdx.x;
        for (; i + (i64)blockDim.x < hi; i += 2 * (i64)blockDim.x) { s0 += (double)x[i]; s1 += (double)x[i + blockDim.x]; }
        if (i < hi) s0 += (double)x[i];
    }
    const double s = block_sum(s0 + s1, scratch);
    if (threadIdx.x == 0) means[chan * gridDim.x + blockIdx.x] = (T)(s / (double)nperseg);
}

// first forward pass: element e of row b = ((x[fa hop + e - pad_left] - mean_a) w[e], (x[fb hop + ...] - mean_b) w[e]),
// the record zero-extended, the frame zero-padded from nperseg to nfft, a frame >= n_frames all zero
template <typename T> struct SrcStftPair {
    const T* sig; const T* window; const T* means;       // means [rows][2], or NULL without detrend
    i64 sig_stride, n_points, n_frames, p0;
    int npc, nperseg, hop, pad_left;
    QI_DEV cplx<T> load(i64 b, i64 e) const {
        if (e >= nperseg) return mk<T>((T)0, (T)0);
        const PairRow r = pair_row(b, npc, p0);
        const T* x = sig + r.chan * sig_stride;
        const i64 pa = r.fa * hop + e - pad_left, pb = pa + hop;
        T va = r.fa < n_frames && pa >= 0 && pa < n_points ? x[pa] : (T)0;
        T vb = r.fa + 1 < n_frames && pb >= 0 && pb < n_points ? x[pb] : (T)0;
        if (means) { va -= means[2 * b]; vb -= means[2 * b + 1]; }
        const T w = window[e];
        return mk<T>(va * w, vb * w);
    }
};

// shared-memory slot of storage offset i of block q (0: residue c, 1: its partner) for frame pair t
QI_HD int stft_long_slot(int q, int t, int i) { return (q * STFT_LONG_P + t) * (STFT_LONG_P + 1) + i; }

// The block pair of one CTA of stft_split_kernel / istft_gather_kernel, grid = (nblk / 2 + 1, ceil(npc / P), C) with
// nblk = nfft / P: blocks c = blockIdx.x and c2 = nblk - c (nb = 1 when they coincide), frame pairs t0 .. t0 + ntp - 1
// of the chunk.  Slot q P + j of the pair is bin k = (q ? c2 : c) + j nfft / P at position i of its block; its Hermitian
// partner k2 = nfft - k sits at position i2 of block q2.
struct LongBlockPair {
    int logL, nblk, c, c2, nb, t0, ntp;
    struct Slot { int q, k, i, k2, q2, i2; };
    QI_DEV LongBlockPair(int logL_, int npc)
        : logL(logL_), nblk((1 << logL_) >> STFT_LONG_LOGP), c(blockIdx.x), c2((nblk - c) & (nblk - 1)),
          nb(c2 == c ? 1 : 2), t0(blockIdx.y * STFT_LONG_P), ntp(npc - t0 < STFT_LONG_P ? npc - t0 : STFT_LONG_P) {}
    // storage position of element 0 of block q in a bit-reversed row
    QI_DEV unsigned row_pos(int q) const { return brev_bits((unsigned)(q ? c2 : c), logL); }
    QI_DEV Slot slot(int s) const {
        constexpr int logP = STFT_LONG_LOGP;
        const int q = s >> logP, j = s & (STFT_LONG_P - 1);
        const int k = (q ? c2 : c) + (j << (logL - logP));
        const int k2 = ((1 << logL) - k) & ((1 << logL) - 1);
        return {q, k, (int)brev_bits((unsigned)j, logP), k2, (k2 & (nblk - 1)) == c ? 0 : 1,
                (int)brev_bits((unsigned)(k2 >> (logL - logP)), logP)};
    }
};
// launch geometry of those kernels for a chunk of npc frame pairs per channel: 256 threads and this grid and shared memory
static dim3 long_pair_grid(int logL, int npc, i64 C) {
    return dim3((unsigned)(((1 << logL) >> STFT_LONG_LOGP) / 2 + 1), (unsigned)((npc + STFT_LONG_P - 1) / STFT_LONG_P),
                (unsigned)C);
}
template <typename T> static size_t long_pair_smem() {
    return (size_t)2 * STFT_LONG_P * (STFT_LONG_P + 1) * sizeof(cplx<T>);
}

// Hermitian split of the pair spectra of one chunk (buf [C * npc][nfft], bit-reversed) into the one-sided bins of both
// frames, times the roll phase and the scale: out [C, nfft/2+1, n_frames] and / or psd_acc [C, nfft/2+1] += |X_k|^2.
// 256 threads; one warp per bin, lanes along the frame pairs.
template <typename T>
__global__ void __launch_bounds__(256)
stft_split_kernel(const cplx<T>* __restrict__ buf, int logL, int npc, i64 p0, i64 n_frames, int roll, T sc,
                  cplx<T>* __restrict__ out, double* __restrict__ psd_acc) {
    QI_DYN_SMEM(smem_raw);
    constexpr int P = STFT_LONG_P, logP = STFT_LONG_LOGP;
    cplx<T>* s = reinterpret_cast<cplx<T>*>(smem_raw);
    const int L = 1 << logL, K = (L >> 1) + 1;
    const LongBlockPair bp(logL, npc);
    const i64 chan = blockIdx.z;
    const cplx<T>* rows = buf + (chan * npc + bp.t0) * (i64)L;
    for (int idx = threadIdx.x; idx < bp.nb * P * P; idx += blockDim.x) {  // lanes along the positions of one row
        const int i = idx & (P - 1), t = (idx >> logP) & (P - 1), q = idx >> (2 * logP);
        if (t < bp.ntp) s[stft_long_slot(q, t, i)] = rows[(i64)t * L + bp.row_pos(q) + i];
    }
    __syncthreads();
    const int t = threadIdx.x & 31;
    const i64 fa = 2 * (p0 + bp.t0 + t);
    for (int slot = threadIdx.x >> 5; slot < bp.nb * P; slot += blockDim.x >> 5) {
        const LongBlockPair::Slot sl = bp.slot(slot);
        const int k = sl.k;
        if (k > (L >> 1)) continue;                                       // the partner's warp has it
        cplx<T> z1 = mk<T>((T)0, (T)0), z2 = z1;
        if (t < bp.ntp) {
            z1 = s[stft_long_slot(sl.q, t, sl.i)];
            z2 = s[stft_long_slot(sl.q2, t, sl.i2)];
        }
        cplx<T> xa, xb;
        pair_split<T>(z1, z2, k, roll, logL, xa, xb);
        if (out && t < bp.ntp) {
            cplx<T>* o = out + (chan * K + k) * n_frames + fa;
            if (fa < n_frames) o[0] = xa * sc;
            if (fa + 1 < n_frames) o[1] = xb * sc;
        }
        if (psd_acc) {
            double pw = 0.0;
            if (t < bp.ntp && fa < n_frames) pw += (double)norm2(xa);
            if (t < bp.ntp && fa + 1 < n_frames) pw += (double)norm2(xb);
            pw = warp_sum(pw);
            if (t == 0) atomicAdd(&psd_acc[chan * K + k], pw);
        }
    }
}

template <typename T>
static int stft_long(const T* sig, i64 C, i64 n_points, i64 stride, const T* window, int nperseg, int hop, int logL,
                     i64 n_frames, int pad_left, double scale, int detrend, int roll, cplx<T>* out, double* psd_acc,
                     void* ws, size_t ws_bytes, cudaStream_t st) {
    const int L = 1 << logL;
    const size_t per_pair = stft_long_pair_bytes<T>(L) * (size_t)C;
    if (ws_bytes < per_pair) return QI_ERR_WORKSPACE;
    if (reinterpret_cast<uintptr_t>(ws) % sizeof(cplx<T>)) return QI_ERR_ARG;
    const i64 npairs = (n_frames + 1) / 2;
    i64 npc = long_pairs_per_chunk(C, n_frames);
    if (npc > (i64)(ws_bytes / per_pair)) npc = (i64)(ws_bytes / per_pair);
    cplx<T>* buf = static_cast<cplx<T>*>(ws);
    T* means = reinterpret_cast<T*>(buf + (size_t)C * npc * L);
    const FftPlan plan = make_plan(logL, (int)sizeof(cplx<T>));
    if (psd_acc) cudaMemsetAsync(psd_acc, 0, sizeof(double) * (size_t)C * (L / 2 + 1), st);
    for (i64 p0 = 0; p0 < npairs; p0 += npc) {
        const int n = (int)(npairs - p0 < npc ? npairs - p0 : npc);
        prof_set_category(QI_CAT_STFT);
        if (detrend)
            QI_LAUNCH((stft_long_means_kernel<T>), dim3((unsigned)(2 * n), (unsigned)C), dim3(256), 0, st, sig, stride,
                      n_points, n_frames, 2 * p0, nperseg, hop, pad_left, means);
        const SrcStftPair<T> src{sig, window, detrend ? means : nullptr, stride, n_points, n_frames, p0, n, nperseg, hop,
                                 pad_left};
        forward_passes<T>(plan, C * n, src, buf, L, st);
        QI_LAUNCH((stft_split_kernel<T>), long_pair_grid(logL, n, C), dim3(256), long_pair_smem<T>(), st, buf, logL, n, p0,
                  n_frames, roll, (T)scale, out, psd_acc);
    }
    return check_cuda("qi_stft");
}

// nfft = 2^logF; roll in [0, nfft)
template <typename T>
static int stft_impl(const void* sig, i64 C, i64 n_points, i64 stride, const void* window, int nperseg, int hop,
                     int logF, i64 n_frames, int pad_left, double scale, int detrend, int roll, void* out,
                     double* psd_acc, void* ws, size_t ws_bytes, cudaStream_t st) {
    const int nfft = 1 << logF;
    const int TC = stft_tile_columns<T>(nfft);
    if (TC == 0 && !ws) return QI_ERR_UNSUPPORTED;
    if (C > 65535) return QI_ERR_UNSUPPORTED;
    if (TC == 0)
        return stft_long<T>(static_cast<const T*>(sig), C, n_points, stride, static_cast<const T*>(window), nperseg, hop,
                            logF, n_frames, pad_left, scale, detrend, roll, static_cast<cplx<T>*>(out), psd_acc, ws,
                            ws_bytes, st);
    // the psd reduction uses shuffles across the TC lanes of one k: needs TC | 32 (true: power of two <= 16)
    StftGeom g;
    g.n_points = n_points; g.sig_stride = stride; g.n_frames = n_frames;
    g.nperseg = nperseg; g.hop = hop; g.logF = logF; g.pad_left = pad_left; g.TC = TC; g.detrend = detrend;
    g.roll = roll;
    g.scale = scale;
    dim3 grid((unsigned)((n_frames + 2 * TC - 1) / (2 * TC)), (unsigned)C);
    const size_t smem = stft_tile_smem<T>(nfft, TC);
    if (psd_acc) cudaMemsetAsync(psd_acc, 0, sizeof(double) * (size_t)C * (nfft / 2 + 1), st);
    prof_set_category(QI_CAT_STFT);
    int logTC = 0;
    while ((1 << logTC) < TC) ++logTC;
#ifndef QI_EMUL
#define QI_STFT_LAUNCH(LF, LT)                                                                                          \
    do {                                                                                                                \
        cudaFuncSetAttribute(stft_kernel<T, LF, LT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);          \
        QI_LAUNCH((stft_kernel<T, LF, LT>), grid, dim3(StftLaunch<T>::threads), smem, st, static_cast<const T*>(sig),   \
                  static_cast<const T*>(window), g, static_cast<cplx<T>*>(out), psd_acc);                               \
    } while (0)
#else
#define QI_STFT_LAUNCH(LF, LT)                                                                                          \
    QI_LAUNCH((stft_kernel<T, LF, LT>), grid, dim3(StftLaunch<T>::threads), smem, st, static_cast<const T*>(sig),       \
              static_cast<const T*>(window), g, static_cast<cplx<T>*>(out), psd_acc)
#endif
    // compile-time sizes for the frame lengths 512 / 1024 / 2048 at the tile counts the budget gives them (16 / 8 / 4)
    if (logF == 9 && logTC == 4) QI_STFT_LAUNCH(9, 4);
    else if (logF == 10 && logTC == 3) QI_STFT_LAUNCH(10, 3);
    else if (logF == 11 && logTC == 2) QI_STFT_LAUNCH(11, 2);
    else QI_STFT_LAUNCH(0, 0);
#undef QI_STFT_LAUNCH
    return check_cuda("qi_stft");
}

// ---------------------------------------------------------------- inverse STFT
// (1) per CTA 2*TC frames of one channel: the one-sided spectra of two frames are combined into one Hermitian-
//     completed complex spectrum Z = Xa + i Xb (rows in bit-reversed order), one inverse tile FFT gives frame a in the
//     real and frame b in the imaginary part; times the dual window -> slices[chan][frame][nperseg].
// (2) overlap-add as a gather: every output sample sums the <= ceil(nperseg/hop) slices that cover it, in ascending
//     frame order (the order of scipy's loop).
struct IstftGeom {
    i64 n_frames, first_start, frame_lo, frame_hi, k0, n_out;
    int nperseg, hop, logF, TC, roll;
};

template <typename T>
__global__ void __launch_bounds__(512, 2)
istft_frames_kernel(const cplx<T>* __restrict__ S, const T* __restrict__ dual_win, IstftGeom g, T* __restrict__ slices) {
    QI_DYN_SMEM(smem_raw);
    const int R = 1 << g.logF;
    const int TC = g.TC, TP = TC + 1;
    const int logTC = 31 - __clz(TC);
    cplx<T>* tile = reinterpret_cast<cplx<T>*>(smem_raw);
    cplx<T>* tw = tile + (size_t)R * TP;
    const i64 chan = blockIdx.y;
    const i64 frame0 = (i64)blockIdx.x * (2 * TC);
    const int K = (R >> 1) + 1;
    fill_twiddles<T>(tw, g.logF);
    // lanes along the frames (fastest axis of S); four spectrum pairs per thread are requested before the first is used
    constexpr int LU = 4;
    for (int base = threadIdx.x; base < K * TC; base += blockDim.x * LU) {
        cplx<T> xa_[LU], xb_[LU];
#pragma unroll
        for (int u = 0; u < LU; ++u) {
            const int idx = base + u * (int)blockDim.x;
            xa_[u] = mk<T>((T)0, (T)0);
            xb_[u] = xa_[u];
            if (idx < K * TC) {
                const int c = idx & (TC - 1);
                const int k = idx >> logTC;
                const i64 fa = frame0 + 2 * c, fb = fa + 1;
                if (fa < g.n_frames) xa_[u] = S[(chan * K + k) * g.n_frames + fa];
                if (fb < g.n_frames) xb_[u] = S[(chan * K + k) * g.n_frames + fb];
            }
        }
#pragma unroll
        for (int u = 0; u < LU; ++u) {
            const int idx = base + u * (int)blockDim.x;
            if (idx >= K * TC) continue;
            const int c = idx & (TC - 1);
            const int k = idx >> logTC;
            cplx<T> zk, zp;
            const bool partner = pair_complete<T>(xa_[u], xb_[u], k, g.roll, g.logF, zk, zp);
            tile[(int)brev_bits((unsigned)k, g.logF) * TP + c] = zk;
            if (partner) tile[(int)brev_bits((unsigned)(R - k), g.logF) * TP + c] = zp;
        }
    }
    __syncthreads();
    tile_fft<T, FFT_INV>(tile, tw, g.logF, TC, TP);
    const T inv = (T)(1.0 / (double)R);
    for (int c = 0; c < TC; ++c) {                                          // lanes along the samples of a slice
        const i64 fa = frame0 + 2 * c;
        if (fa >= g.n_frames) break;
        for (int n = threadIdx.x; n < g.nperseg; n += blockDim.x) {
            const cplx<T> v = tile[n * TP + c];
            const T w = dual_win[n] * inv;
            slices[(chan * g.n_frames + fa) * g.nperseg + n] = v.re * w;
            if (fa + 1 < g.n_frames) slices[(chan * g.n_frames + fa + 1) * g.nperseg + n] = v.im * w;
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(256)
istft_ola_kernel(const T* __restrict__ slices, IstftGeom g, T* __restrict__ out) {
    const i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= g.n_out) return;
    const i64 chan = blockIdx.y;
    const i64 k = g.k0 + i;
    // frames p with first_start + p*hop <= k < first_start + p*hop + nperseg
    const i64 d = k - g.first_start;
    const i64 e = d - (g.nperseg - 1);
    i64 p_hi, p_lo;
    if ((g.hop & (g.hop - 1)) == 0) {                                                   // hop = 2^s: arithmetic shifts
        const int sh = 31 - __clz(g.hop);
        p_hi = d >> sh;                                                                 // floor(d / hop)
        p_lo = -((-e) >> sh);                                                           // ceil(e / hop)
    } else {
        p_hi = d >= 0 ? d / g.hop : -((-d + g.hop - 1) / g.hop);
        p_lo = e > 0 ? (e + g.hop - 1) / g.hop : -((-e) / g.hop);
    }
    if (p_lo < g.frame_lo) p_lo = g.frame_lo;
    if (p_hi > g.frame_hi - 1) p_hi = g.frame_hi - 1;
    T acc = (T)0;
    for (i64 p = p_lo; p <= p_hi; ++p)
        acc += slices[(chan * g.n_frames + p) * g.nperseg + (d - p * g.hop)];
    out[chan * g.n_out + i] = acc;
}

// dynamic shared memory of istft_frames_kernel with tc columns, and its columns per CTA (0: the frame does not fit)
template <typename T> static size_t istft_tile_smem(int nfft, int tc) { return (size_t)nfft * (tc + 2) * sizeof(cplx<T>) + 64; }
template <typename T> static int istft_tile_columns(int nfft) { return tile_columns(nfft, 100 * 1024, istft_tile_smem<T>); }

// Long frames: Hermitian-completed pair spectra Z = Xa + i Xb of one chunk (S [C, nfft/2+1, P] -> buf [C * npc][nfft],
// bit-reversed rows).  The block pairs of stft_split_kernel, the other way round.
template <typename T>
__global__ void __launch_bounds__(256)
istft_gather_kernel(const cplx<T>* __restrict__ S, int logL, int npc, i64 p0, i64 n_frames, int roll,
                    cplx<T>* __restrict__ buf) {
    QI_DYN_SMEM(smem_raw);
    constexpr int P = STFT_LONG_P, logP = STFT_LONG_LOGP;
    cplx<T>* s = reinterpret_cast<cplx<T>*>(smem_raw);
    const int L = 1 << logL, K = (L >> 1) + 1;
    const LongBlockPair bp(logL, npc);
    const i64 chan = blockIdx.z;
    const int t = threadIdx.x & 31;
    const i64 fa = 2 * (p0 + bp.t0 + t);
    for (int slot = threadIdx.x >> 5; slot < bp.nb * P; slot += blockDim.x >> 5) {
        const LongBlockPair::Slot sl = bp.slot(slot);
        const int k = sl.k;
        if (k > (L >> 1) || t >= bp.ntp) continue;                       // bins above nfft/2: the partner's warp
        cplx<T> xa = mk<T>((T)0, (T)0), xb = xa;
        if (fa < n_frames) xa = S[(chan * K + k) * n_frames + fa];
        if (fa + 1 < n_frames) xb = S[(chan * K + k) * n_frames + fa + 1];
        cplx<T> zk, zp;
        const bool partner = pair_complete<T>(xa, xb, k, roll, logL, zk, zp);
        s[stft_long_slot(sl.q, t, sl.i)] = zk;
        if (partner) s[stft_long_slot(sl.q2, t, sl.i2)] = zp;
    }
    __syncthreads();
    cplx<T>* rows = buf + (chan * npc + bp.t0) * (i64)L;
    for (int idx = threadIdx.x; idx < bp.nb * P * P; idx += blockDim.x) {  // lanes along the positions of one row
        const int i = idx & (P - 1), tt = (idx >> logP) & (P - 1), q = idx >> (2 * logP);
        if (tt < bp.ntp) rows[(i64)tt * L + bp.row_pos(q) + i] = s[stft_long_slot(q, tt, i)];
    }
}

// last inverse pass of the long route: sample n < nperseg of row b's two frames, times dual_win[n] / nfft, into the
// slices [C][n_frames][nperseg] of istft_frames_kernel
template <typename T> struct DstIstftPair {
    T* slices; const T* dual_win;
    i64 n_frames, p0;
    int npc, nperseg;
    T inv;
    QI_DEV void store(i64 b, i64 n, cplx<T> v) const {
        if (n >= nperseg) return;
        const PairRow r = pair_row(b, npc, p0);
        const T w = dual_win[n] * inv;
        T* o = slices + (r.chan * n_frames + r.fa) * nperseg + n;
        o[0] = v.re * w;
        if (r.fa + 1 < n_frames) o[nperseg] = v.im * w;
    }
    QI_DEV void finish(i64, unsigned char*) const {}
};

// workspace of the inverse: the slices; on the long route those rounded up to 256 bytes, then the pair spectra of one chunk
template <typename T> static size_t istft_slices_bytes(i64 C, i64 n_frames, int nperseg) {
    return (size_t)C * (size_t)n_frames * (size_t)nperseg * sizeof(T);
}
template <typename T> static size_t istft_workspace_bytes(i64 C, i64 n_frames, int nperseg, int nfft) {
    const size_t slices = istft_slices_bytes<T>(C, n_frames, nperseg);
    if (C > 65535 || log2_pow2(nfft) < 0 || istft_tile_columns<T>(nfft)) return slices;
    return (slices + 255) / 256 * 256 + (size_t)C * (size_t)long_pairs_per_chunk(C, n_frames) * (size_t)nfft * sizeof(cplx<T>);
}

template <typename T>
static void istft_long_slices(const cplx<T>* S, i64 C, i64 P, const T* dual_win, int nperseg, int logL, int roll, T* slices,
                              cudaStream_t st) {
    const int L = 1 << logL;
    const i64 npairs = (P + 1) / 2, npc = long_pairs_per_chunk(C, P);
    cplx<T>* buf = reinterpret_cast<cplx<T>*>(reinterpret_cast<unsigned char*>(slices) +
                                              (istft_slices_bytes<T>(C, P, nperseg) + 255) / 256 * 256);
    const FftPlan plan = make_plan(logL, (int)sizeof(cplx<T>));
    const T inv = (T)(1.0 / (double)L);
    for (i64 p0 = 0; p0 < npairs; p0 += npc) {
        const int n = (int)(npairs - p0 < npc ? npairs - p0 : npc);
        prof_set_category(QI_CAT_STFT);
        QI_LAUNCH((istft_gather_kernel<T>), long_pair_grid(logL, n, C), dim3(256), long_pair_smem<T>(), st, S, logL, n, p0,
                  P, roll, buf);
        const DstIstftPair<T> dst{slices, dual_win, P, p0, n, nperseg, inv};
        inverse_passes<T>(plan, C * n, SrcComplex<T>{buf, L}, dst, 0, false, buf, L, st);
    }
    prof_set_category(QI_CAT_STFT);
}

// nfft = 2^logF; roll in [0, nfft)
template <typename T>
static int istft_impl(const void* S, i64 C, i64 P, const void* dual_win, int nperseg, int hop, int logF, int roll,
                      i64 first_start, i64 frame_lo, i64 frame_hi, i64 k0, i64 n_out, void* out, void* ws,
                      cudaStream_t st) {
    const int nfft = 1 << logF;
    const int TC = istft_tile_columns<T>(nfft);
    if (C > 65535) return QI_ERR_UNSUPPORTED;
    IstftGeom g;
    g.n_frames = P; g.first_start = first_start; g.frame_lo = frame_lo; g.frame_hi = frame_hi; g.k0 = k0; g.n_out = n_out;
    g.nperseg = nperseg; g.hop = hop; g.logF = logF; g.TC = TC; g.roll = roll;
    if (TC == 0) {
        if (reinterpret_cast<uintptr_t>(ws) % sizeof(cplx<T>)) return QI_ERR_ARG;
        istft_long_slices<T>(static_cast<const cplx<T>*>(S), C, P, static_cast<const T*>(dual_win), nperseg, logF, roll,
                             static_cast<T*>(ws), st);
    } else {
        const size_t smem = istft_tile_smem<T>(nfft, TC);
#ifndef QI_EMUL
        cudaFuncSetAttribute(istft_frames_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
#endif
        prof_set_category(QI_CAT_STFT);
        dim3 grid((unsigned)((P + 2 * TC - 1) / (2 * TC)), (unsigned)C);
        QI_LAUNCH((istft_frames_kernel<T>), grid, dim3(512), smem, st, static_cast<const cplx<T>*>(S),
                  static_cast<const T*>(dual_win), g, static_cast<T*>(ws));
    }
    dim3 grid2((unsigned)((n_out + 255) / 256), (unsigned)C);
    QI_LAUNCH((istft_ola_kernel<T>), grid2, dim3(256), 0, st, static_cast<const T*>(ws), g, static_cast<T*>(out));
    return check_cuda("qi_istft");
}

}  // namespace qi

extern "C" size_t qi_stft_workspace_bytes(int64_t C, int64_t n_frames, int nfft, int dtype) {
    if (C <= 0 || n_frames <= 0 || qi::log2_pow2(nfft) < 0) return 0;
    if (dtype == QI_F32) return qi::stft_workspace_bytes<float>(C, n_frames, nfft);
    if (dtype == QI_F64) return qi::stft_workspace_bytes<double>(C, n_frames, nfft);
    return 0;
}

extern "C" int qi_stft(const void* sig, int64_t C, int64_t n_points, int64_t stride, const void* window, int nperseg,
                       int hop, int nfft, int64_t n_frames, int pad_left, double scale, int detrend, int roll, int dtype,
                       void* out, double* psd_acc, void* workspace, size_t workspace_bytes, void* stream) {
    if (!sig || !window || C <= 0 || n_points <= 0 || nperseg <= 0 || hop <= 0 || nfft < nperseg || n_frames <= 0)
        return QI_ERR_ARG;
    if (!out && !psd_acc) return QI_ERR_ARG;
    const int logF = qi::log2_pow2(nfft);
    if (logF < 0) return QI_ERR_ARG;
    roll = ((roll % nfft) + nfft) % nfft;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (dtype == QI_F32)
        return qi::stft_impl<float>(sig, C, n_points, stride, window, nperseg, hop, logF, n_frames, pad_left, scale,
                                    detrend, roll, out, psd_acc, workspace, workspace_bytes, st);
    if (dtype == QI_F64)
        return qi::stft_impl<double>(sig, C, n_points, stride, window, nperseg, hop, logF, n_frames, pad_left, scale,
                                     detrend, roll, out, psd_acc, workspace, workspace_bytes, st);
    return QI_ERR_ARG;
}

extern "C" size_t qi_istft_workspace_bytes(int64_t C, int64_t n_frames, int nperseg, int nfft, int dtype) {
    if (C <= 0 || n_frames <= 0 || nperseg <= 0) return 0;
    if (dtype == QI_F64) return qi::istft_workspace_bytes<double>(C, n_frames, nperseg, nfft);
    // float32; for an unknown dtype, which qi_istft refuses, the float32 slices alone
    return qi::istft_workspace_bytes<float>(C, n_frames, nperseg, dtype == QI_F32 ? nfft : 0);
}

extern "C" int qi_istft(const void* S, int64_t C, int64_t n_frames, const void* dual_win, int nperseg, int hop, int nfft,
                        int roll, int64_t first_start, int64_t frame_lo, int64_t frame_hi, int64_t k0, int64_t n_out,
                        int dtype, void* out, void* ws, size_t ws_bytes, void* stream) {
    if (!S || !dual_win || !out || !ws || C <= 0 || n_frames <= 0 || nperseg <= 0 || hop <= 0 || nfft < nperseg ||
        n_out <= 0 || frame_lo < 0 || frame_hi > n_frames || frame_lo >= frame_hi)
        return QI_ERR_ARG;
    if (ws_bytes < qi_istft_workspace_bytes(C, n_frames, nperseg, nfft, dtype)) return QI_ERR_WORKSPACE;
    const int logF = qi::log2_pow2(nfft);
    if (logF < 0) return QI_ERR_ARG;
    roll = ((roll % nfft) + nfft) % nfft;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (dtype == QI_F32)
        return qi::istft_impl<float>(S, C, n_frames, dual_win, nperseg, hop, logF, roll, first_start, frame_lo, frame_hi,
                                     k0, n_out, out, ws, st);
    if (dtype == QI_F64)
        return qi::istft_impl<double>(S, C, n_frames, dual_win, nperseg, hop, logF, roll, first_start, frame_lo,
                                      frame_hi, k0, n_out, out, ws, st);
    return QI_ERR_ARG;
}
