// qi_mr_level2k.cuh -- "A" of the multirate CWT (see qi_mr.cu): overlap-save convolution of one level signal with all
// bands of that level, 2048-point blocks, written for the fewest passes over shared memory per output sample (the
// kernel is bound by the shared-memory / L1 data pipe, not by HBM).
//
//   * A CTA of 256 threads convolves PAIRS of consecutive blocks: the two blocks are the two complex columns of a
//     float4 tile row.  The radix-8 stages work on whole rows (one 128-bit access serves both transforms); the radix-16
//     stages give each thread ONE column, with the two threads holding the same rows of blocks a and b in adjacent lanes
//     (t = 2u + column): a lane pair touches one 16-byte row, so a half warp's 64-bit access is conflict free exactly
//     when its 8 rows are, and both lanes of a pair read the same band-table lines.
//   * 2048 = 8 * 16 * 16.  Forward = DIF (natural -> bit-reversed), inverse = DIT (bit-reversed -> natural), as
//     everywhere in this library (qi_fft.cuh); dif16 / dit16 keep the fully bit-reversed spectrum, so the band tables of
//     mr_table_kernel and the envelope fold see the same row order as a radix-2 transform (the tables are stored in the
//     warp order of l2k_tab_slot so that their loads stay coalesced).
//   * forward: radix-8 at B=2048 straight from HBM (real input) -> tile, radix-16 at B=256 through the tile, radix-16 at
//     B=16 read from the tile: thread (u, column) keeps rows 16u .. 16u+15 of its block's spectrum X in REGISTERS.
//   * per band (level 0, and every level of the complex-TFR mode): X * K and the radix-16 B=16 stage in registers ->
//     tile, radix-16 at B=256 through the tile, radix-8 at B=2048 read from the tile; its natural-order outputs go from
//     registers to HBM (level 0: |.|^2 -> power plane; deeper levels: the decimated complex output w_b).  Two tile
//     buffers alternate between bands: 4 tile accesses and 2 barriers per band.
//   * per band pair (envelope bands, levels >= 1): the 16 register rows fold into rows 8u .. 8u+7 of the 1024-point
//     spectrum, whose radix-8 B=8 stage runs in registers -> tile, radix-16 at B=128, radix-8 at B=1024 read -> the
//     demodulated envelope: also 4 accesses and 2 barriers.
//     band_sum (optional) receives sum |y|^2 over the record's own samples: the exact band power at level 0, the raw
//     sum that mr_total_kernel turns into the band-power estimate at deeper levels.
//   * twiddles come from per-stage tables laid out [slot pair][j] (built once per call by mr_twiddle2k_kernel with the
//     exact sincospi roots, copied to shared memory per CTA): conflict-free 128-bit loads, one per two slots.  The
//     B=2048 twiddles depend on the thread only and stay in registers for the whole kernel.
//   * tile rows: the 2048-row tile pads one row per 16 (l2k_phys), the 1024-row envelope tiles one row per 8
//     (l2k_physe).  Rows a half warp touches per access, l2k_phys: t + 256 i (8 consecutive t), 256G + j + 16 i (8
//     consecutive j), 16u + i (8 consecutive u -> 17u + i, distinct mod 8); l2k_physe: 8u + i (9u + i), 128G + j + 8 i
//     and j + 128 i (8 consecutive j): every stage is bank-conflict free and every address is "base register +
//     immediate".
#pragma once
#include "qi_fft.cuh"
#include "qi_mr_expand.cuh"
#include "qi_reduce.cuh"

namespace qi {

constexpr int L2K_LOGF = 11;
constexpr int L2K_F = 1 << L2K_LOGF;
QI_HD int l2k_phys(int r) { return r + (r >> 4); }   // padded row of a 2048-row tile
QI_HD int l2k_physe(int r) { return r + (r >> 3); }  // padded row of a 1024-row envelope tile
constexpr int L2K_TILE = L2K_F + L2K_F / 8;          // rows per tile buffer: two 1024-row envelope tiles (>= l2k_phys(F))
// Band tables of 2048-point levels (mr_table_kernel) are stored in warp order: bit-reversed row r = 16u + 2m + e (group u
// of a radix-16 thread, float4 m of its rows, half e) sits at complex slot 2 (128 (u >> 4) + 16 m + (u & 15)) + e.  The 16
// groups of a warp then read float4 m of their rows from 256 consecutive bytes: 2 cache lines per load instruction
// instead of 16 (the lane pair of a group reads the same float4).
QI_HD int l2k_tab_slot(int r) {
    const int u = r >> 4, m = (r >> 1) & 7;
    return ((((u >> 4) << 7) | (m << 4) | (u & 15)) << 1) | (r & 1);
}
QI_HD int l2k_tab_group(int u) { return ((u >> 4) << 7) | (u & 15); }   // float4 index of (group u, m = 0)
// twiddle tables, float4 entries [m][j]: (w_B^(j * brev(2m)), w_B^(j * brev(2m+1))), brev = brev3 for the radix-8 stages
// (m < 4), brev4 for the radix-16 stages (m < 8).  The first L2K_TW_SMEM entries are copied to shared memory:
//   B=1024 (radix 8, j < 128), then radix 16 with L2K_TW16J rows per m: B=256 (j < 16) and B=128 (rows 16 + j, j < 8),
//   then 32 float4 holding the 64 demodulation phases exp(-2 pi i m / 64);
// the B=2048 stage (radix 8, j < 256) follows and is read into registers from global memory.
constexpr int L2K_TWE0 = 0;
constexpr int L2K_TW16 = 4 * 128, L2K_TW16J = 24;
constexpr int L2K_DEMOD = L2K_TW16 + 8 * L2K_TW16J;
constexpr int L2K_TW_SMEM = L2K_DEMOD + 32;
constexpr int L2K_TWA = L2K_TW_SMEM;
constexpr int L2K_TW_TOTAL = L2K_TWA + 4 * 256;     // float4 elements in the whole table
constexpr int L2K_MAXB = 64;                         // bands per level handled by this kernel
constexpr int L2K_THREADS = 256;
constexpr size_t L2K_SMEM = (size_t)(2 * L2K_TILE + L2K_TW_SMEM) * 16 + (size_t)(L2K_THREADS / 32) * L2K_MAXB * 4;

__global__ void mr_twiddle2k_kernel(float4* __restrict__ tw) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= L2K_TW_TOTAL) return;
    if (idx >= L2K_DEMOD && idx < L2K_TW_SMEM) {               // two consecutive phases per float4
        const int m = 2 * (idx - L2K_DEMOD);
        const cplx<float> w0 = conj(unit_root<float>((unsigned long long)m, 6));
        const cplx<float> w1 = conj(unit_root<float>((unsigned long long)(m + 1), 6));
        tw[idx] = make_float4(w0.re, w0.im, w1.re, w1.im);
        return;
    }
    int m, j, logB, f0, f1;
    if (idx < L2K_TW16) {
        m = idx / 128; j = idx % 128; logB = 10;
    } else if (idx < L2K_DEMOD) {
        const int row = (idx - L2K_TW16) % L2K_TW16J;
        m = (idx - L2K_TW16) / L2K_TW16J;
        logB = row < 16 ? 8 : 7; j = row < 16 ? row : row - 16;
    } else {
        m = (idx - L2K_TWA) / 256; j = (idx - L2K_TWA) % 256; logB = 11;
    }
    if (idx >= L2K_TW16 && idx < L2K_DEMOD) { f0 = brev4(2 * m); f1 = brev4(2 * m + 1); }
    else { f0 = brev3(2 * m); f1 = brev3(2 * m + 1); }
    const cplx<float> w0 = conj(unit_root<float>((unsigned long long)(j * f0), logB));
    const cplx<float> w1 = conj(unit_root<float>((unsigned long long)(j * f1), logB));
    tw[idx] = make_float4(w0.re, w0.im, w1.re, w1.im);
}

struct MrLevelGeom {
    int level, logF, TC;
    int band_first, band_count, n_bands;
    int wk;                 // two-sided kernel support reserved per block (even); valid outputs per block V = F - wk
    i64 n_points;           // N
    i64 n_level;            // N >> level
    i64 q_first;            // first output index (level rate): -MR_HALO for level >= 1, 0 for level 0
    i64 n_out;              // outputs per channel at this level
    i64 n_blocks;
    i64 x_stride, x_len;    // level signal: per-channel stride, stored length
    int x_halo;             // halo of the stored level signal (0 for level 0)
    int env;                // every band of this level is stored as a demodulated envelope at level + 1
    int no_sums;            // edge source bands (indices >= n_bands): no row of their own in the sum arrays
};

// one column of the tile: element p of column c of a float4 tile is col[2 p] with col = (float2*)tile + c
QI_DEV cplx<float> l2k_ld(const float2* col, int p) { const float2 v = col[2 * p]; return mk<float>(v.x, v.y); }
QI_DEV void l2k_st(float2* col, int p, cplx<float> v) { col[2 * p] = make_float2(v.re, v.im); }

// radix-16 stage on one column; rows base + i*H live at col[2 (p0 + i*STRIDE)], twiddles tw[L2K_TW16 + m L2K_TW16J + twrow]
template <int DIR, int STRIDE>
QI_DEV void l2k_stage16(float2* __restrict__ col, int p0, const float4* __restrict__ tw, int twrow) {
    cplx<float> a[16];
    const float4* w = tw + L2K_TW16 + twrow;
    if (DIR == FFT_FWD) {
#pragma unroll
        for (int i = 0; i < 16; ++i) a[i] = l2k_ld(col, p0 + i * STRIDE);
        dif16<float, DIR>(a);
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            cplx<float> v0 = a[2 * m], v1 = a[2 * m + 1];
            const float4 ww = w[m * L2K_TW16J];
            if (m) v0 = v0 * mk<float>(ww.x, ww.y);
            v1 = v1 * mk<float>(ww.z, ww.w);
            l2k_st(col, p0 + 2 * m * STRIDE, v0);
            l2k_st(col, p0 + (2 * m + 1) * STRIDE, v1);
        }
    } else {
#pragma unroll
        for (int m = 0; m < 8; ++m) {
            const float4 ww = w[m * L2K_TW16J];
            a[2 * m] = l2k_ld(col, p0 + 2 * m * STRIDE);
            a[2 * m + 1] = mul_conj(l2k_ld(col, p0 + (2 * m + 1) * STRIDE), mk<float>(ww.z, ww.w));
            if (m) a[2 * m] = mul_conj(a[2 * m], mk<float>(ww.x, ww.y));
        }
        dit16<float, DIR>(a);
#pragma unroll
        for (int i = 0; i < 16; ++i) l2k_st(col, p0 + i * STRIDE, a[i]);
    }
}

// radix-8 DIT stage on both columns of a float4 tile, rows base + s*H at tile[p0 + s*STRIDE], per-thread twiddles w
QI_DEV void l2k_read_dit8(const float4* __restrict__ tile, int p0, int stride, const float4 (&w)[4], cplx<float> (&a)[8],
                          cplx<float> (&c)[8]) {
#pragma unroll
    for (int s = 0; s < 8; ++s) {
        const float4 v = tile[p0 + s * stride];
        cplx<float> va = mk<float>(v.x, v.y), vb = mk<float>(v.z, v.w);
        if (s) {
            const float4 ww = w[s >> 1];
            const cplx<float> tt = (s & 1) ? mk<float>(ww.z, ww.w) : mk<float>(ww.x, ww.y);
            va = mul_conj(va, tt); vb = mul_conj(vb, tt);
        }
        a[s] = va; c[s] = vb;
    }
    dit8<float, FFT_INV>(a); dit8<float, FFT_INV>(c);
}

// bx: index of this CTA among the CTAs of its level (blockIdx.x, or the offset inside a merged multi-level launch)
// ENV = false compiles the envelope path out (the level-0 launch: fewer registers)
template <bool ENV>
QI_DEV void l2k_body(const float* __restrict__ x, const MrLevelGeom& g, const MrDevBand* __restrict__ bands,
                     const cplx<float>* __restrict__ tables, const float4* __restrict__ tw_g,
                     cplx<float>* __restrict__ wbuf, float* __restrict__ out_power, cplx<float>* __restrict__ out_complex,
                     double* __restrict__ band_sum, int pairs_per_cta, int bx) {
    QI_DYN_SMEM(smem_raw);
    float4* tile0 = reinterpret_cast<float4*>(smem_raw);
    float4* tile1 = tile0 + L2K_TILE;
    float4* tw = tile1 + L2K_TILE;
    float* wsum = reinterpret_cast<float*>(tw + L2K_TW_SMEM);          // [warps][L2K_MAXB]
    const int t = threadIdx.x;
    const int warp = t >> 5, lane = t & 31;
    const i64 chan = blockIdx.y;
    const int V = L2K_F - g.wk;
    const int half = g.wk / 2;
    const float* xs = x + chan * g.x_stride;

    for (int i = t; i < L2K_TW_SMEM; i += L2K_THREADS) tw[i] = tw_g[i];
    for (int i = t; i < (L2K_THREADS / 32) * L2K_MAXB; i += L2K_THREADS) wsum[i] = 0.0f;

    // per-thread tile addresses (padded rows), fixed for the whole kernel
    const int pA = l2k_phys(t);                                            // B=2048: rows t + 256 i    -> + 272 i
    const int cl = t & 1, u = t >> 1;                                      // radix-16 stages: column, row group
    const int pB = 272 * (u >> 4) + (u & 15);                              // B=256 : rows 256G + j + 16 i -> + 17 i
    const int pC = 17 * u;                                                 // B=16  : rows 16u + i         -> + i

    // twiddles of the stage B=2048 depend on the thread only: kept in registers for the forward stage and every band
    float4 wA[4];
#pragma unroll
    for (int m = 0; m < 4; ++m) wA[m] = tw_g[L2K_TWA + m * 256 + t];

    for (int pp = 0; pp < pairs_per_cta; ++pp) {
        const i64 blk0 = 2 * ((i64)bx * pairs_per_cta + pp);
        if (blk0 >= g.n_blocks) break;                                     // uniform over the CTA
        __syncthreads();                                                   // previous pair's last stage has left the tiles
        // ---- forward, stage B=2048 straight from HBM (real input, two blocks)
        {
            cplx<float> a[8], b[8];
            const i64 k0 = g.q_first + blk0 * V - half + g.x_halo + t;
            const bool has_b = blk0 + 1 < g.n_blocks;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const i64 ka = k0 + 256 * i, kb = ka + V;
                a[i] = mk<float>((ka >= 0 && ka < g.x_len) ? xs[ka] : 0.0f, 0.0f);
                b[i] = mk<float>((has_b && kb >= 0 && kb < g.x_len) ? xs[kb] : 0.0f, 0.0f);
            }
            dif8<float, FFT_FWD>(a); dif8<float, FFT_FWD>(b);
#pragma unroll
            for (int s = 0; s < 8; ++s) {
                cplx<float> va = a[s], vb = b[s];
                if (s) {
                    const float4 ww = wA[s >> 1];
                    const cplx<float> tt = (s & 1) ? mk<float>(ww.z, ww.w) : mk<float>(ww.x, ww.y);
                    va = va * tt; vb = vb * tt;
                }
                tile0[pA + s * 272] = make_float4(va.re, va.im, vb.re, vb.im);
            }
        }
        __syncthreads();
        l2k_stage16<FFT_FWD, 17>(reinterpret_cast<float2*>(tile0) + cl, pB, tw, u & 15);
        __syncthreads();
        // ---- forward stage B=16: the spectrum of block cl stays in registers (bit-reversed rows 16u .. 16u+15)
        cplx<float> X[16];
        {
            const float2* col = reinterpret_cast<const float2*>(tile0) + cl;
#pragma unroll
            for (int i = 0; i < 16; ++i) X[i] = l2k_ld(col, pC + i);
            dif16<float, FFT_FWD>(X);
        }

        // ---- envelope bands: two bands per pass, half-size inverse transforms (see mr_plan)
        //   fold   Z[k'] = Y[k'] + Y[k' + 1024]  <->  rows (2q, 2q+1) of the bit-reversed 2048-row spectrum add up to
        //          row q of the bit-reversed 1024-row one: y(2m) = IFFT_1024(Z)(m)
        //   rows 16u .. 16u+15 of Y fold into rows 8u .. 8u+7 of Z, whose radix-8 B=8 stage runs in registers; then
        //   radix-16 at B=128 (64 butterflies per band and column) and radix-8 at B=1024 (128 per band, both columns)
        for (int pi = 0; ENV && g.env && pi < g.band_count; pi += 2) {
            const int nbp = g.band_count - pi < 2 ? g.band_count - pi : 2;
            float4* tile = ((pi >> 1) & 1) ? tile0 : tile1;
            for (int bb = 0; bb < nbp; ++bb) {
                const float4* K = reinterpret_cast<const float4*>(tables + bands[g.band_first + pi + bb].table_off) +
                                 l2k_tab_group(u);
                cplx<float> z[8];
#pragma unroll
                for (int m = 0; m < 8; ++m) {
                    const float4 k = K[16 * m];
                    z[m] = X[2 * m] * mk<float>(k.x, k.y) + X[2 * m + 1] * mk<float>(k.z, k.w);
                }
                dit8<float, FFT_INV>(z);
                float2* col = reinterpret_cast<float2*>(tile + bb * (L2K_TILE / 2)) + cl;
#pragma unroll
                for (int i = 0; i < 8; ++i) l2k_st(col, 9 * u + i, z[i]);         // l2k_physe(8u + i)
            }
            __syncthreads();
            {   // stage B=128: rows 128G + j + 8i -> 144G + j + 9i, band u >> 6 of the pass
                const int bb = u >> 6, G = (u >> 3) & 7, j = u & 7;
                if (bb < nbp)
                    l2k_stage16<FFT_INV, 9>(reinterpret_cast<float2*>(tile + bb * (L2K_TILE / 2)) + cl, 144 * G + j, tw,
                                            16 + j);
            }
            __syncthreads();
            const int bb = t >> 7, v = t & 127;                            // band of the pass / butterfly of that band
            if (bb < nbp) {   // stage B=1024: rows v + 128i -> v + (v >> 3) + 144i; outputs m = v + 128 i leave from registers
                cplx<float> a[8], c[8];
                float4 w[4];
#pragma unroll
                for (int m = 0; m < 4; ++m) w[m] = tw[L2K_TWE0 + m * 128 + v];
                l2k_read_dit8(tile + bb * (L2K_TILE / 2), l2k_physe(v), 144, w, a, c);
                const int b = g.band_first + pi + bb;
                const MrDevBand band = bands[b];
                const cplx<float>* dm = reinterpret_cast<const cplx<float>*>(tw + L2K_DEMOD);   // exp(-2 pi i m / 64)
                const int Vh = V >> 1, hh = half >> 1;
                const i64 n_w = (g.n_level >> 1) + 2 * MR_HALO;              // stored samples of w at level + 1
                float acc = 0.0f;
#pragma unroll
                for (int col = 0; col < 2; ++col) {
                    const i64 blk = blk0 + col;
                    if (blk >= g.n_blocks) break;
                    const cplx<float>* y = col ? c : a;
                    cplx<float>* wdst = wbuf + band.w_off + chan * band.w_stride;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int mm = v + 128 * i - hh;
                        const i64 wi = blk * Vh + mm;                       // index into w (halo included): q' = wi - HALO
                        if (mm >= 0 && mm < Vh && wi < n_w) {
                            const i64 q = wi - MR_HALO;
                            const cplx<float> e = y[i] * dm[(int)((band.demod * q) & 63)];
                            wdst[wi] = e;
                            if (q >= 0 && q < (g.n_level >> 1)) acc += norm2(e);
                        }
                    }
                }
                if (band_sum) {
                    acc = warp_sum(acc);
                    if (lane == 0) wsum[warp * L2K_MAXB + pi + bb] += acc;
                }
            }
        }

        // ---- bands
        for (int bi = 0; !(ENV && g.env) && bi < g.band_count; ++bi) {
            const int b = g.band_first + bi;
            const MrDevBand band = bands[b];
            float4* tile = (bi & 1) ? tile0 : tile1;
            {   // inverse stage B=16 on X * K, from registers
                const float4* K = reinterpret_cast<const float4*>(tables + band.table_off) + l2k_tab_group(u);
                cplx<float> a[16];
#pragma unroll
                for (int m = 0; m < 8; ++m) {
                    const float4 k = K[16 * m];
                    a[2 * m] = X[2 * m] * mk<float>(k.x, k.y);
                    a[2 * m + 1] = X[2 * m + 1] * mk<float>(k.z, k.w);
                }
                dit16<float, FFT_INV>(a);
                float2* col = reinterpret_cast<float2*>(tile) + cl;
#pragma unroll
                for (int i = 0; i < 16; ++i) l2k_st(col, pC + i, a[i]);
            }
            __syncthreads();
            l2k_stage16<FFT_INV, 17>(reinterpret_cast<float2*>(tile) + cl, pB, tw, u & 15);
            __syncthreads();
            // ---- last stage B=2048: outputs n = t + 256 i leave from registers
            cplx<float> a[8], c[8];
            l2k_read_dit8(tile, pA, 272, wA, a, c);
            float acc = 0.0f;
#pragma unroll
            for (int col = 0; col < 2; ++col) {
                const i64 blk = blk0 + col;
                if (blk >= g.n_blocks) break;
                const i64 o0 = blk * V;                  // output ordinal of this block's first valid sample
                const cplx<float>* y = col ? c : a;
                if (g.level == 0) {
                    const i64 cell0 = (chan * g.n_bands + b) * g.n_points + o0 - half;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int pv = t + 256 * i - half;
                        if (pv >= 0 && pv < V && o0 + pv < g.n_out) {
                            const float pw = norm2(y[i]);
                            if (out_power) out_power[cell0 + t + 256 * i] = pw;
                            if (out_complex) out_complex[cell0 + t + 256 * i] = y[i];
                            acc += pw;
                        }
                    }
                } else {
                    cplx<float>* wdst = wbuf + band.w_off + chan * band.w_stride + o0 - half;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int pv = t + 256 * i - half;
                        if (pv >= 0 && pv < V && o0 + pv < g.n_out) {
                            wdst[t + 256 * i] = y[i];
                            // sum over the record proper (q in [0, N >> level), not the halo) for the power estimate
                            const i64 q = g.q_first + o0 + pv;
                            if (q >= 0 && q < g.n_level) acc += norm2(y[i]);
                        }
                    }
                }
            }
            if (band_sum) {
                acc = warp_sum(acc);
                if (lane == 0) wsum[warp * L2K_MAXB + bi] += acc;
            }
        }
    }
    if (band_sum) {
        __syncthreads();
        if (t < g.band_count) {
            double s = 0.0;
            for (int w = 0; w < L2K_THREADS / 32; ++w) s += (double)wsum[w * L2K_MAXB + t];
            atomicAdd(&band_sum[chan * g.n_bands + g.band_first + t], s);
        }
    }
}

template <bool ENV>
__global__ void __launch_bounds__(L2K_THREADS, 2)
mr_level2k_kernel(const float* __restrict__ x, MrLevelGeom g, const MrDevBand* __restrict__ bands,
                  const cplx<float>* __restrict__ tables, const float4* __restrict__ tw_g,
                  cplx<float>* __restrict__ wbuf, float* __restrict__ out_power, cplx<float>* __restrict__ out_complex,
                  double* __restrict__ band_sum, int pairs_per_cta) {
    l2k_body<ENV>(x, g, bands, tables, tw_g, wbuf, out_power, out_complex, band_sum, pairs_per_cta, (int)blockIdx.x);
}

// The deep levels are a few CTAs each and independent of one another: one launch runs up to L2K_MULTI of them side by
// side instead of a chain of latency-bound launches.
constexpr int L2K_MULTI = 8;
struct MrMultiLevel {
    int n;
    int cta_end[L2K_MULTI];          // exclusive prefix sums of CTAs per level (grid.x = cta_end[n-1])
    int ppc[L2K_MULTI];
    MrLevelGeom g[L2K_MULTI];
    const float* x[L2K_MULTI];
    double* sum[L2K_MULTI];
};

__global__ void __launch_bounds__(L2K_THREADS, 2)
mr_level2k_multi_kernel(MrMultiLevel m, const MrDevBand* __restrict__ bands, const cplx<float>* __restrict__ tables,
                        const float4* __restrict__ tw_g, cplx<float>* __restrict__ wbuf) {
    int li = 0;
    while (li + 1 < m.n && (int)blockIdx.x >= m.cta_end[li]) ++li;
    const int bx = (int)blockIdx.x - (li ? m.cta_end[li - 1] : 0);
    const MrLevelGeom g = m.g[li];
    l2k_body<true>(m.x[li], g, bands, tables, tw_g, wbuf, nullptr, nullptr, m.sum[li], m.ppc[li], bx);
}

}  // namespace qi
