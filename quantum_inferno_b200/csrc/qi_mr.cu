// qi_mr.cu -- multirate fp32 Gabor CWT: the fast path behind cwt_entropy / styx_cwt(dtype=float32, method=multirate).
//
// The output plane [bands x N] is compulsory HBM traffic (4 B/cell); everything else is kept far below it:
//
//   P  pyramid      x_(l+1)[q] = halfband(x_l)[2q]  (zero-phase minimax half-band FIR, |error| <= 1e-6, exact
//                   zero extension of the record carried in a 16-sample halo).  Total work ~ N per channel.
//   T  tables       every band lives at the deepest level l whose alias-free band [0, pi/2] still holds its response out
//                   to |theta - omega| <= 2.4/s (the host's choice, _plan.MR_KAPPA: beyond that the last decimation
//                   stage is still within 4e-5 of unity where the band answers with less than 6 %).  Its kernel at that rate,
//                   2^l * psi(2^l d - 1/2) truncated like the reference's N-sample atom, is sampled in fp64,
//                   transformed once in shared memory and kept (bit-reversed order, L2 resident) for all channels.
//   A  level conv   overlap-save convolution of x_l with all bands of level l in 2048-point blocks
//                   (qi_mr_level2k.cuh): block spectra in registers, per band multiply + inverse FFT in shared
//                   memory.  Level-0 bands go straight to |.|^2 -> power rows (+ exact fp64 band sums); deeper bands
//                   leave their decimated complex output w_b (8 B per 2^l cells) in HBM, together with the raw sum
//                   of |w_b|^2 that the band-power estimate needs.
//                   With power / information outputs the bands of levels 1 .. cap-1 are stored as demodulated
//                   ENVELOPES one level deeper (half-size inverse transforms, see mr_plan).
//   S  total power  mr_total_kernel: S per record from those sums (Euler-Maclaurin corrected), BEFORE any plane of
//                   the deeper bands is written, so that the information plane can be fused into E.
//   E  expand       qi_mr_expand.cuh: per (channel, band, 16384-cell span) the band's decimated samples are read
//                   once, brought to level k = min(l, 3) by half-band stages in shared memory and to the full rate
//                   by one merged polyphase interpolator x2^k from registers, fused with |.|^2, -log2(P/S + eps),
//                   both plane stores (256-bit) and the band / entropy sums.  Every band is read at its own level (a
//                   deep band: a few samples per tile), so that almost no DRAM read disturbs the kernel's write stream.
//                   Bands deeper than level 5 are also brought to level 5 once (MID mode, 1/32 of the cells) for the
//                   raw sums and end samples that the band-power estimate is made from.
//   I  info rows    the level-0 rows' information plane (their power was written before S was known).
//   R  edge rows    the reference cuts its atoms off at the record; for the record-long atoms of the lowest bands that
//                   jump answers to every frequency of the record.  It is split off as a straight line over the atom's
//                   support, whose contribution is a running sum + first moment of the record (prefix_block in mr_pyramid3_kernel, mr_prefix_scan_kernel and
//                   a block scan inside E); the continuous remainder runs through T / A / E as an extra source band.
//                   See MrDevBand in qi_mr_expand.cuh.
//
// Replaces (fp32 tolerance of the north star: power rel. L2 <= 1e-4) quantum_inferno/styx_cwt.py:147-198 + np.abs()**2.
// tools/multirate_prototype.py is the numpy model the first version of this algorithm was validated with.
#include "qi_fft.cuh"
#include "qi_host.h"
#include "qi_reduce.cuh"
#include "qi_tfr.cuh"
#include "qi_halfband_coeffs.h"
#include "qi_mr_expand.cuh"
#include "qi_mr_level2k.cuh"

#include <vector>
#include <math.h>
#include <stdlib.h>

namespace qi {

// ---------------------------------------------------------------- P: half-band decimation by 2
// src: level l (with halo `src_halo`, length src_len incl. halo; level 0: halo 0), dst: level l+1 with MR_HALO.
// A CTA makes 1024 outputs: the source tile is split on the way into shared memory into its even samples (the
// centre taps) and its odd samples (all other taps), so a thread's four consecutive outputs need six 128-bit loads
//     out[q] = 0.5 * even[q] + sum_t c_t * (odd[q + t] + odd[q - t - 1])
// src rows must be 8-byte aligned, dst rows 16-byte aligned, dst_len a multiple of 4 (true for every level array).
constexpr int DEC_TILE = 1024, DEC_PAD = 8;
static_assert(QI_HB_MAX_TAPS <= DEC_PAD - 1, "decimator window");
__global__ void __launch_bounds__(256)
mr_decimate_kernel(const float* __restrict__ src, i64 src_stride, i64 src_len, int src_halo,
                   float* __restrict__ dst, i64 dst_stride, i64 dst_len, HbTaps taps) {
    __shared__ __align__(16) float s_even[DEC_TILE + 2 * DEC_PAD];
    __shared__ __align__(16) float s_odd[DEC_TILE + 2 * DEC_PAD + 4];
    const i64 c = blockIdx.y;
    const float* s = src + c * src_stride;
    const i64 i_base = (i64)blockIdx.x * DEC_TILE;                 // dst index of the tile's first output, q = i - MR_HALO
    const i64 k_base = 2 * (i_base - MR_HALO - DEC_PAD) + src_halo; // src index of slot 0 (even by construction)
    for (int j = threadIdx.x; j < DEC_TILE + 2 * DEC_PAD; j += blockDim.x) {
        const i64 k = k_base + 2 * j;
        float2 v = make_float2(0.0f, 0.0f);
        if (k >= 0 && k + 1 < src_len) v = *reinterpret_cast<const float2*>(s + k);
        else {
            if (k >= 0 && k < src_len) v.x = s[k];
            if (k + 1 >= 0 && k + 1 < src_len) v.y = s[k + 1];
        }
        s_even[j] = v.x;
        s_odd[j] = v.y;
    }
    if (threadIdx.x < 4) s_odd[DEC_TILE + 2 * DEC_PAD + threadIdx.x] = 0.0f;
    __syncthreads();
    const int j0 = 4 * threadIdx.x;                                // outputs j0 .. j0+3 of the tile; slot = j + DEC_PAD
    if (i_base + j0 >= dst_len) return;
    float od[20];                                                  // odd[j0 - 8 .. j0 + 11] <-> slots j0 .. j0 + 19
#pragma unroll
    for (int m = 0; m < 5; ++m) {
        const float4 v = *reinterpret_cast<const float4*>(s_odd + j0 + 4 * m);
        od[4 * m] = v.x; od[4 * m + 1] = v.y; od[4 * m + 2] = v.z; od[4 * m + 3] = v.w;
    }
    const float4 ev = *reinterpret_cast<const float4*>(s_even + j0 + DEC_PAD);
    const float e[4] = {ev.x, ev.y, ev.z, ev.w};
    float o[4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        float acc = 0.5f * e[r];
#pragma unroll
        for (int t = 0; t < QI_HB_MAX_TAPS; ++t)                   // taps beyond n[0] are stored as zeros
            acc += taps.c[0][t] * (od[8 + r + t] + od[8 + r - t - 1]);
        o[r] = acc;
    }
    *reinterpret_cast<float4*>(dst + c * dst_stride + i_base + j0) = make_float4(o[0], o[1], o[2], o[3]);
}

// ---------------------------------------------------------------- running sums of the record (edge rows, see MrDevBand)
// blk[c][0][j + 1] = sum of x over block j, blk[c][1][j + 1] = sum of (k - (N-1)/2) x[k] over block j  (fp64), and
// grp[c][j * 256 + t] = (L0, L1) = (sum_{m < 8t} a[m], sum_{m < 8t} (m + 1) a[m]) with a[m] = x[2048 j + m]: the block-local
// exclusive scans the edge expansion starts its 8 outputs from (see edge_add in qi_mr_expand.cuh).
// One 2048-sample block per call, 256 threads, z = the thread's samples a[8 tid .. 8 tid + 7].
struct PrefixScratch { double red[32]; float wtot[2][8]; };
QI_DEV void prefix_block(const float* z, i64 c, i64 j, i64 n_points, double* __restrict__ blk, i64 n_prefix,
                         float2* __restrict__ grp, PrefixScratch& sh) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float s0 = 0.0f, s1 = 0.0f;
    const float fi0 = (float)(8 * tid);
#pragma unroll
    for (int r = 0; r < 8; ++r) { s0 += z[r]; s1 = fmaf(fi0 + (float)(r + 1), z[r], s1); }
    float i0 = s0, i1 = s1;                              // inclusive scan of the thread totals over the warp
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const float u0 = __shfl_up_sync(0xffffffffu, i0, o), u1 = __shfl_up_sync(0xffffffffu, i1, o);
        if (lane >= o) { i0 += u0; i1 += u1; }
    }
    __syncthreads();                                     // the previous block of this CTA has left the scratch
    if (lane == 31) { sh.wtot[0][warp] = i0; sh.wtot[1][warp] = i1; }
    __syncthreads();
    float off0 = i0 - s0, off1 = i1 - s1;
    for (int w = 0; w < warp; ++w) { off0 += sh.wtot[0][w]; off1 += sh.wtot[1][w]; }
    grp[c * (n_points >> 3) + j * (MR_EDGE_BLOCK / 8) + tid] = make_float2(off0, off1);
    // block totals in fp64: sum a[m], sum (2048 j + m - cc) a[m] with sum (m + 1) a[m] = s1
    const double k0 = (double)(j * MR_EDGE_BLOCK) - 1.0 - 0.5 * (double)(n_points - 1);
    double d0 = (double)s0, d1 = k0 * (double)s0 + (double)s1;
    d0 = block_sum(d0, sh.red);
    d1 = block_sum(d1, sh.red);
    if (tid == 0) {
        double* row = blk + c * 2 * n_prefix;
        row[j + 1] = d0;
        row[n_prefix + j + 1] = d1;
    }
}
// ---------------------------------------------------------------- P: levels 1, 2 and 3 in one pass over the record
// The three finest levels are 7/8 of the pyramid's traffic when each level re-reads the one above it.  Here a CTA reads
// 8 * P3_T + 224 record samples once and leaves P3_T level-3 samples plus the level-1 / level-2 samples it owns
// (stored indices [4 P3_T j, 4 P3_T (j+1)) and [2 P3_T j, 2 P3_T (j+1))); the intermediate tiles live in shared memory,
// split into even and odd samples like the tile of mr_decimate_kernel.  Same arithmetic, same order, same zero
// extension as three runs of mr_decimate_kernel (a sample outside a level's stored range [-HALO, n + HALO) is zero), so
// the results are bit-identical to the level-by-level chain.  With edge rows (blk != nullptr) the CTA also makes the
// running sums of the two 2048-sample blocks [4096 j, 4096 (j+1)) it holds (prefix_block): no second pass over the record.
// Tile geometry (q = index at the level's own rate, first sample of a tile a multiple of 8):
//   level 3: q in [P3_T j - 16, + P3_T)            level 2: [2 P3_T j - 48, + 2 P3_T + 32)
//   level 1: [4 P3_T j - 112, + 4 P3_T + 96)       record : [8 P3_T j - 240, + 8 P3_T + 240)   (the last 16 samples:
//                                                            prefix sums only)
// so that output m of a tile sits at p = 8 + m of the tile above it: a thread makes 4 outputs from O[4g .. 4g + 19] and
// E[4g + 8 .. 4g + 11] (six 128-bit loads), g its group index.
constexpr int P3_T = 512;
constexpr int P3_N0 = 8 * P3_T + 240, P3_N1 = 4 * P3_T + 96, P3_N2 = 2 * P3_T + 32;
static_assert(QI_HB_MAX_TAPS == 7 && MR_HALO == 16, "tile geometry of mr_pyramid3_kernel");
static_assert(8 * P3_T == 2 * MR_EDGE_BLOCK, "two prefix blocks per CTA");

// 4 consecutive outputs of one half-band decimation from the even / odd arrays of the level above
QI_DEV void p3_group(const float* __restrict__ E, const float* __restrict__ O, int g, const HbTaps& taps, float* o) {
    float od[20];
#pragma unroll
    for (int m = 0; m < 5; ++m) {
        const float4 v = *reinterpret_cast<const float4*>(O + 4 * g + 4 * m);
        od[4 * m] = v.x; od[4 * m + 1] = v.y; od[4 * m + 2] = v.z; od[4 * m + 3] = v.w;
    }
    const float4 ev = *reinterpret_cast<const float4*>(E + 4 * g + 8);
    const float e[4] = {ev.x, ev.y, ev.z, ev.w};
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        float acc = 0.5f * e[r];
#pragma unroll
        for (int t = 0; t < QI_HB_MAX_TAPS; ++t)
            acc += taps.c[0][t] * (od[8 + r + t] + od[8 + r - t - 1]);
        o[r] = acc;
    }
}

__global__ void __launch_bounds__(256)
mr_pyramid3_kernel(const float* __restrict__ sig, i64 sig_stride, i64 n_points, float* __restrict__ l1,
                   float* __restrict__ l2, float* __restrict__ l3, i64 pyr_stride, HbTaps taps, double* __restrict__ blk,
                   i64 n_prefix, float2* __restrict__ grp) {
    __shared__ PrefixScratch sh;
    __shared__ __align__(16) float E0[P3_N0 / 2], O0[P3_N0 / 2];
    __shared__ __align__(16) float E1[P3_N1 / 2], O1[P3_N1 / 2];
    __shared__ __align__(16) float E2[P3_N2 / 2], O2[P3_N2 / 2];
    const i64 c = blockIdx.y, j = blockIdx.x;
    const float* x = sig + c * sig_stride;
    // record tile: all loads of a thread in flight before the first store
    {
        const i64 k0 = 8 * (i64)P3_T * j - 240;
        constexpr int LU = (P3_N0 / 2 + 255) / 256;
        float2 v[LU];
#pragma unroll
        for (int u = 0; u < LU; ++u) {
            const int s = threadIdx.x + 256 * u;
            const i64 k = k0 + 2 * s;
            v[u] = make_float2(0.0f, 0.0f);
            if (s < P3_N0 / 2) {
                if (k >= 0 && k + 1 < n_points) v[u] = *reinterpret_cast<const float2*>(x + k);
                else {
                    if (k >= 0 && k < n_points) v[u].x = x[k];
                    if (k + 1 >= 0 && k + 1 < n_points) v[u].y = x[k + 1];
                }
            }
        }
#pragma unroll
        for (int u = 0; u < LU; ++u) {
            const int s = threadIdx.x + 256 * u;
            if (s < P3_N0 / 2) { E0[s] = v[u].x; O0[s] = v[u].y; }
        }
    }
    __syncthreads();
    if (blk) {
        // record sample 4096 j + 2048 b + 8 t + r sits at tile offset 240 + 2048 b + 8 t + r: four even, four odd slots
        for (int b = 0; b < 2; ++b) {
            const i64 jb = 2 * j + b;
            if (jb >= n_prefix - 1) break;                           // uniform over the CTA
            const int s0 = 120 + 1024 * b + 4 * threadIdx.x;
            const float4 ev = *reinterpret_cast<const float4*>(E0 + s0), ov = *reinterpret_cast<const float4*>(O0 + s0);
            const float z[8] = {ev.x, ov.x, ev.y, ov.y, ev.z, ov.z, ev.w, ov.w};
            prefix_block(z, c, jb, n_points, blk, n_prefix, grp, sh);
        }
    }
    // level 1: stored index i = q + HALO, q = 4 P3_T j - 112 + 4 g + r; owned from i = 4 P3_T j on
    {
        const i64 len = (n_points >> 1) + 2 * MR_HALO;
        float* dst = l1 + c * pyr_stride;
        for (int g = threadIdx.x; g < P3_N1 / 4; g += 256) {
            float o[4];
            p3_group(E0, O0, g, taps, o);
            const i64 i = 4 * (i64)P3_T * j - 112 + MR_HALO + 4 * g;
            if (i < 0 || i >= len) { o[0] = 0.0f; o[1] = 0.0f; o[2] = 0.0f; o[3] = 0.0f; }   // len and i are multiples of 4
            *reinterpret_cast<float2*>(E1 + 2 * g) = make_float2(o[0], o[2]);
            *reinterpret_cast<float2*>(O1 + 2 * g) = make_float2(o[1], o[3]);
            if (4 * g >= 96 && i >= 0 && i < len) *reinterpret_cast<float4*>(dst + i) = make_float4(o[0], o[1], o[2], o[3]);
        }
    }
    __syncthreads();
    {
        const i64 len = (n_points >> 2) + 2 * MR_HALO;
        float* dst = l2 + c * pyr_stride;
        for (int g = threadIdx.x; g < P3_N2 / 4; g += 256) {
            float o[4];
            p3_group(E1, O1, g, taps, o);
            const i64 i = 2 * (i64)P3_T * j - 48 + MR_HALO + 4 * g;
            if (i < 0 || i >= len) { o[0] = 0.0f; o[1] = 0.0f; o[2] = 0.0f; o[3] = 0.0f; }
            *reinterpret_cast<float2*>(E2 + 2 * g) = make_float2(o[0], o[2]);
            *reinterpret_cast<float2*>(O2 + 2 * g) = make_float2(o[1], o[3]);
            if (4 * g >= 32 && i >= 0 && i < len) *reinterpret_cast<float4*>(dst + i) = make_float4(o[0], o[1], o[2], o[3]);
        }
    }
    __syncthreads();
    {
        const i64 len = (n_points >> 3) + 2 * MR_HALO;
        float* dst = l3 + c * pyr_stride;
        for (int g = threadIdx.x; g < P3_T / 4; g += 256) {
            float o[4];
            p3_group(E2, O2, g, taps, o);
            const i64 i = (i64)P3_T * j + 4 * g;
            if (i < len) *reinterpret_cast<float4*>(dst + i) = make_float4(o[0], o[1], o[2], o[3]);
        }
    }
}

// ---------------------------------------------------------------- T: kernel tables
// One CTA per band: sample kappa[d] = 2^l * amp * exp(-t^2/2s^2) * exp(i*omega*t), t = 2^l d - 1/2, on the circular
// lag grid of F points, keep |d| <= half_w and |t| <= (N-1)/2, forward FFT in shared memory, store * 1/F.
__global__ void __launch_bounds__(256)
mr_table_kernel(const MrDevBand* __restrict__ bands, i64 n_points, int half_w_cap, cplx<float>* __restrict__ tables) {
    QI_DYN_SMEM(smem_raw);
    const MrDevBand b = bands[blockIdx.x];
    const int F = 1 << b.logF;
    cplx<float>* tile = reinterpret_cast<cplx<float>*>(smem_raw);       // [F][2]
    cplx<float>* tw = tile + (size_t)F * 2;
    fill_twiddles<float>(tw, b.logF);
    const double step = (double)(1ll << b.conv_level);
    const double tmax = 0.5 * (double)(n_points - 1);
    // time support kept: 5.2 sigma (3e-6 of the peak) or the whole block half for record-long atoms
    int half_w = (int)ceil(5.2 * b.scale / step) + 1;
    if (half_w > half_w_cap) half_w = half_w_cap;
    for (int p = threadIdx.x; p < F; p += blockDim.x) {
        const int d = p < F / 2 ? p : p - F;
        double re = 0.0, im = 0.0;
        const double t = step * (double)d - 0.5;
        if (d >= -half_w && d <= half_w && fabs(t) <= tmax) {
            const double u = t / b.scale;
            const double env = step * b.amp * exp(-0.5 * u * u);
            double s, c;
            sincos(b.omega * t, &s, &c);
            re = env * c; im = env * s;
            if (b.flags & MR_FLAG_EDGE_SRC) { re -= step * b.edge_ar; im -= step * b.edge_beta * t; }
        }
        tile[p * 2] = mk<float>((float)re, (float)im);
    }
    __syncthreads();
    tile_fft<float, FFT_FWD>(tile, tw, b.logF, 1, 2);
    const float inv = 1.0f / (float)F;
    for (int p = threadIdx.x; p < F; p += blockDim.x)       // 2048-point tables: the warp order of mr_level2k_kernel
        tables[b.table_off + (F == L2K_F ? l2k_tab_slot(p) : p)] = tile[p * 2] * inv;
}

// ---------------------------------------------------------------- A: overlap-save level convolution (generic)
// Any block length / one block per column; used for the deepest level (one 4096-point block holds the whole level)
// and for levels whose kernels need 4096-point blocks.  The 2048-point fast path is qi_mr_level2k.cuh.
__global__ void __launch_bounds__(1024)
mr_level_kernel(const float* __restrict__ x, MrLevelGeom g, const MrDevBand* __restrict__ bands,
                const cplx<float>* __restrict__ tables, cplx<float>* __restrict__ wbuf,
                float* __restrict__ out_power, cplx<float>* __restrict__ out_complex, double* __restrict__ band_sum) {
    QI_DYN_SMEM(smem_raw);
    const int F = 1 << g.logF;
    const int TC = g.TC, TP = TC + 1;
    cplx<float>* tile_x = reinterpret_cast<cplx<float>*>(smem_raw);
    cplx<float>* tile_y = tile_x + (size_t)F * TP;
    cplx<float>* tw = tile_y + (size_t)F * TP;
    double* scratch = reinterpret_cast<double*>(tw + F);
    const i64 chan = blockIdx.y;
    const i64 blk0 = (i64)blockIdx.x * TC;
    const int V = F - g.wk;
    const int logTC = 31 - __clz(TC);
    const float* xs = x + chan * g.x_stride;

    fill_twiddles<float>(tw, g.logF);
    for (int idx = threadIdx.x; idx < F * TC; idx += blockDim.x) {
        const int p = idx & (F - 1);
        const int c = idx >> g.logF;
        const i64 blk = blk0 + c;
        float v = 0.0f;
        if (blk < g.n_blocks) {
            const i64 q = g.q_first + blk * V - g.wk / 2 + p;
            const i64 k = q + g.x_halo;
            if (k >= 0 && k < g.x_len) v = xs[k];
        }
        tile_x[p * TP + c] = mk<float>(v, 0.0f);
    }
    __syncthreads();
    tile_fft<float, FFT_FWD>(tile_x, tw, g.logF, TC, TP);

    // grid.z splits the level's bands over CTAs (each repeats the cheap forward transform): the deepest level is one
    // block per channel with a dozen bands, which would otherwise be a dozen serial inverse FFTs on 8 SMs
    const int per_z = (g.band_count + (int)gridDim.z - 1) / (int)gridDim.z;
    const int bi_end = min(g.band_count, ((int)blockIdx.z + 1) * per_z);
    for (int bi = (int)blockIdx.z * per_z; bi < bi_end; ++bi) {
        const int b = g.band_first + bi;
        const MrDevBand band = bands[b];
        const cplx<float>* K = tables + band.table_off;
        for (int idx = threadIdx.x; idx < F * TC; idx += blockDim.x) {
            const int c = idx & (TC - 1);
            const int r = idx >> logTC;
            tile_y[r * TP + c] = tile_x[r * TP + c] * K[F == L2K_F ? l2k_tab_slot(r) : r];
        }
        __syncthreads();
        tile_fft<float, FFT_INV>(tile_y, tw, g.logF, TC, TP);
        float acc_f = 0.0f;
        for (int c = 0; c < TC; ++c) {
            const i64 blk = blk0 + c;
            if (blk >= g.n_blocks) break;
            const i64 o0 = blk * V;                 // output ordinal of this block's first valid sample
            const cplx<float>* ycol = tile_y + (g.wk / 2) * TP + c;
            if (g.level == 0) {
                const i64 cell0 = (chan * g.n_bands + b) * g.n_points + o0;
                for (int pv = threadIdx.x; pv < V; pv += blockDim.x) {     // lanes along the output index
                    if (o0 + pv < g.n_out) {
                        const cplx<float> y = ycol[pv * TP];
                        const float pw = norm2(y);
                        if (out_power) out_power[cell0 + pv] = pw;
                        if (out_complex) out_complex[cell0 + pv] = y;
                        acc_f += pw;
                    }
                }
            } else {
                cplx<float>* wdst = wbuf + band.w_off + chan * band.w_stride + o0;
                for (int pv = threadIdx.x; pv < V; pv += blockDim.x) {
                    if (o0 + pv < g.n_out) {
                        const cplx<float> y = ycol[pv * TP];
                        wdst[pv] = y;
                        const i64 q = g.q_first + o0 + pv;             // raw sum over the record proper, see mr_total_kernel
                        if (q >= 0 && q < g.n_level) acc_f += norm2(y);
                    }
                }
            }
        }
        double acc = (double)acc_f;
        if (band_sum) {
            acc = block_sum(acc, scratch);
            if (threadIdx.x == 0) atomicAdd(&band_sum[chan * g.n_bands + b], acc);
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------- running sums of the record: block scan
// in-place inclusive scan of each of the 2 C rows (entry 0 = 0): row[j] = sum over the blocks before block j
__global__ void __launch_bounds__(1024)
mr_prefix_scan_kernel(double* __restrict__ blk, i64 n_prefix) {
    __shared__ double part[1024];
    double* row = blk + (i64)blockIdx.x * n_prefix;
    const i64 per = (n_prefix + blockDim.x - 1) / blockDim.x;
    const i64 i0 = (i64)threadIdx.x * per, i1 = i0 + per < n_prefix ? i0 + per : n_prefix;
    double s = 0.0;
    for (i64 i = i0; i < i1; ++i) s += i ? row[i] : 0.0;
    part[threadIdx.x] = s;
    __syncthreads();
    for (int o = 1; o < (int)blockDim.x; o <<= 1) {           // Hillis-Steele over the per-thread sums
        const double u = (int)threadIdx.x >= o ? part[threadIdx.x - o] : 0.0;
        __syncthreads();
        part[threadIdx.x] += u;
        __syncthreads();
    }
    double run = part[threadIdx.x] - s;
    for (i64 i = i0; i < i1; ++i) { run += i ? row[i] : 0.0; row[i] = run; }
}

// ---------------------------------------------------------------- host driver
struct MrPlan {
    int cap;                         // deepest level
    std::vector<i64> lvl_off, lvl_len;   // pyramid arrays (levels 1..cap), float elements per channel / offsets
    std::vector<MrDevBand> bands;
    std::vector<int> expand_list;       // bands with level >= 1 (final expand launch)
    std::vector<int> deep_list;         // bands with level > MR_LMID (first brought to level MR_LMID)
    std::vector<MrLevelGeom> levels;
    int n_edge;                         // edge rows = the first n_edge bands; their source bands are B .. B + n_edge - 1
    i64 n_prefix;
    size_t off_bands, off_list, off_deep, off_tw, off_pyr, off_tables, off_w, off_mid, off_prefix, off_group, total;
    i64 pyr_per_chan, w_total, mid_total;
};

static HbTaps make_taps() {
    HbTaps t;
    for (int j = 0; j < QI_HB_CLASSES; ++j) {
        t.n[j] = qi_hb_ntaps[j];
        for (int i = 0; i < QI_HB_MAX_TAPS; ++i) t.c[j][i] = (float)qi_hb_taps[j][i];
    }
    return t;
}

// allow_env: bands of the levels 1 .. cap-1 may be stored as demodulated envelopes one level deeper (power / information
// outputs only; the complex TFR needs the carrier).  The workspace query plans without it (an upper bound).
static int mr_plan(i64 C, i64 N, const QiMrBand* hb, int B, MrPlan& pl, bool allow_env = false) {
    int logN = 0;
    while ((1ll << logN) < N) ++logN;
    if ((1ll << logN) != N || logN < 13 || logN > 30) return QI_ERR_UNSUPPORTED;
    pl.cap = logN - 10;
    if (pl.cap > MR_MAX_LEVEL) return QI_ERR_UNSUPPORTED;
    // bands must come sorted by ascending frequency => non-increasing level
    for (int b = 0; b < B; ++b) {
        if (hb[b].level < 0 || hb[b].level > pl.cap) return QI_ERR_ARG;
        if (b && hb[b].level > hb[b - 1].level) return QI_ERR_ARG;
    }
    // pyramid arrays
    pl.lvl_off.assign(pl.cap + 1, 0);
    pl.lvl_len.assign(pl.cap + 1, 0);
    i64 off = 0;
    for (int l = 1; l <= pl.cap; ++l) {
        pl.lvl_len[l] = (N >> l) + 2 * MR_HALO;
        pl.lvl_off[l] = off;
        off += (pl.lvl_len[l] + 63) / 64 * 64;
    }
    pl.pyr_per_chan = off;
    // edge rows: record-long atoms (they sit at the deepest level, at the low end of the table)
    pl.n_edge = 0;
    while (pl.n_edge < B && hb[pl.n_edge].level == pl.cap && (double)N / hb[pl.n_edge].scale < MR_EDGE_NS) ++pl.n_edge;
    const int E = pl.n_edge;
    pl.n_prefix = N / MR_EDGE_BLOCK + 1;
    // bands, tables, decimated outputs
    pl.bands.resize(B + E);
    pl.expand_list.clear();
    pl.deep_list.clear();
    pl.levels.clear();
    i64 toff = 0, woff = 0, moff = 0;
    for (int l = pl.cap; l >= 0; --l) {
        int first = -1, count = 0;
        double smax = 0.0;
        for (int b = 0; b < B; ++b)
            if (hb[b].level == l) { if (first < 0) first = b; ++count; smax = fmax(smax, hb[b].scale / (double)(1ll << l)); }
        if (!count) continue;
        MrLevelGeom g;
        g.level = l; g.band_first = first; g.band_count = count; g.n_bands = B;
        g.n_points = N; g.n_level = N >> l;
        g.x_halo = l ? MR_HALO : 0;
        g.x_len = l ? pl.lvl_len[l] : N;
        g.q_first = l ? -MR_HALO : 0;
        g.n_out = l ? (N >> l) + 2 * MR_HALO : N;
        if (l == pl.cap) {
            // record-long (possibly truncated) atoms: one block holds the whole level
            g.wk = (int)(2 * (g.n_level + 2 * MR_HALO));
            g.logF = 12;
            if ((1 << g.logF) - g.wk < g.n_out) return QI_ERR_UNSUPPORTED;
        } else {
            // half a multiple of 16 -> V a multiple of 32: every plane store of the 2048-point kernel is sector aligned
            const int half = ((int)ceil(5.2 * smax) + 1 + 15) & ~15;
            g.wk = 2 * half;
            g.logF = g.wk <= 768 ? 11 : 12;
            if (g.wk > 3072) return QI_ERR_UNSUPPORTED;
        }
        g.TC = 1;
        g.no_sums = 0;
        // Envelope decimation.  The band output y_b at level l is analytic with support |theta - omega_l| <= 4.8/s_l, so
        // its even samples are alias free, and times exp(-i omega_d q) they form a LOW-PASS signal at level l + 1 that
        // the real-coefficient interpolators of E handle like any other level-(l+1) band: half the inverse FFT, half the
        // decimated traffic, one octave less for the x2/x4 interpolators.  |.|^2 does not see the demodulation.
        // omega_d is a multiple of 2 pi / 64 (exact phases from a 64-entry table).
        g.env = 0;
        std::vector<int> demod(count, 0);
        if (allow_env && l >= 1 && l < pl.cap && g.logF == L2K_LOGF && count <= L2K_MAXB) {
            g.env = 1;
            for (int b = first; b < first + count; ++b) {
                const double wc = hb[b].omega * (double)(1ll << (l + 1));             // centre at level l + 1
                const int kd = (int)llround(wc * 64.0 / (2.0 * M_PI));
                const double dev = fabs(wc - 2.0 * M_PI * kd / 64.0);
                // QI_MR_ENV_KAPPA: measurement override of the envelope half-width (see DESIGN.md, "what is next")
                static const double env_kappa = getenv("QI_MR_ENV_KAPPA") ? atof(getenv("QI_MR_ENV_KAPPA")) : 4.8;
                const double halfbw = env_kappa / (hb[b].scale / (double)(1ll << (l + 1)));
                if (halfbw + dev > 0.98 * M_PI / 2.0 || wc + halfbw >= 2.0 * M_PI) g.env = 0;
                demod[b - first] = kd & 63;
            }
        }
        if (g.env) { g.q_first = -2 * MR_HALO; g.n_out = (N >> l) + 4 * MR_HALO; }
        const int V = (1 << g.logF) - g.wk;
        g.n_blocks = (g.n_out + V - 1) / V;
        pl.levels.push_back(g);
        const int lout = l + g.env;
        auto add_band = [&](int idx, int b, int flags) {
            MrDevBand d;
            d.omega = hb[b].omega; d.scale = hb[b].scale; d.amp = hb[b].amp; d.logF = g.logF;
            d.edge_ar = 0.0; d.edge_beta = 0.0; d.out_row = b; d.flags = flags;
            if (flags & MR_FLAG_EDGE_SRC) {
                // last sample of the N-sample atom, g[N-1] = amp exp(-cc^2 / 2 s^2) exp(i omega cc), cc = (N-1)/2
                const double cc = 0.5 * (double)(N - 1);
                const double env = hb[b].amp * exp(-0.5 * (cc / hb[b].scale) * (cc / hb[b].scale));
                d.edge_ar = env * cos(hb[b].omega * cc);
                d.edge_beta = env * sin(hb[b].omega * cc) / cc;
            }
            d.level = lout; d.conv_level = l; d.demod = g.env ? demod[b - first] : 0;
            d.table_off = toff; toff += (1ll << g.logF);
            d.w_off = 0; d.w_stride = 0; d.mid_off = 0; d.mid_stride = 0;
            if (l) {
                d.w_stride = ((N >> lout) + 2 * MR_HALO + 63) / 64 * 64;
                d.w_off = woff; woff += d.w_stride * C;
                if (!(flags & MR_FLAG_EDGE_EST)) pl.expand_list.push_back(idx);
            }
            if (lout > MR_LMID) {
                d.mid_stride = ((N >> MR_LMID) + 2 * MR_HALO + 63) / 64 * 64;
                d.mid_off = moff; moff += d.mid_stride * C;
                if (!(flags & MR_FLAG_EDGE_SRC)) pl.deep_list.push_back(idx);   // sources have no estimate of their own
            }
            pl.bands[idx] = d;
        };
        // the edge source bands first: both lists keep the bands of one launch group contiguous
        if (l == pl.cap && E > 0) {
            MrLevelGeom ge = g;
            ge.band_first = B; ge.band_count = E; ge.no_sums = 1;
            pl.levels.push_back(ge);
            for (int b = 0; b < E; ++b) add_band(B + b, b, MR_FLAG_EDGE_SRC);
        }
        for (int b = first; b < first + count; ++b) add_band(b, b, (l == pl.cap && b < E) ? MR_FLAG_EDGE_EST : 0);
    }
    pl.w_total = woff;
    pl.mid_total = moff;
    size_t o = 0;
    pl.off_bands = o; o = align_up(o + sizeof(MrDevBand) * (size_t)(B + E), 256);
    pl.off_list = o; o = align_up(o + sizeof(int) * (size_t)(B + E + 1), 256);
    pl.off_deep = o; o = align_up(o + sizeof(int) * (size_t)(B + E + 1), 256);
    pl.off_prefix = o; o = align_up(o + sizeof(double) * 2 * (size_t)pl.n_prefix * (size_t)C * (E > 0 ? 1 : 0), 256);
    pl.off_group = o; o = align_up(o + sizeof(float2) * (size_t)(N / 8) * (size_t)C * (E > 0 ? 1 : 0), 256);
    pl.off_tw = o; o = align_up(o + sizeof(float4) * (size_t)L2K_TW_TOTAL, 256);
    pl.off_pyr = o; o = align_up(o + sizeof(float) * (size_t)pl.pyr_per_chan * C, 256);
    pl.off_tables = o; o = align_up(o + sizeof(cplx<float>) * (size_t)toff, 256);
    pl.off_w = o; o = align_up(o + sizeof(cplx<float>) * (size_t)woff, 256);
    pl.off_mid = o; o = align_up(o + sizeof(cplx<float>) * (size_t)moff, 256);
    pl.total = o;
    return QI_OK;
}

// Band-power estimates and the per-record total that normalises the pdf, needed before the planes are written.
// band_sum_est arrives holding the RAW sums  sum_{q < N/h} |w(q)|^2  of every band with level >= 1, accumulated by
// the kernel that produced its decimated output w at level min(L, MR_LMID) (h = 2^that level).  With P = |w|^2
// band-limited below that level's Nyquist rate,
//     sum_{n<N} P(n) ~= h * sum_q P(h q) + (h-1)/2 (P(N) - P(0)) - (h^2-1)/12 (P'(N) - P'(0))      (Euler-Maclaurin,
// P' by central differences; deep bands use their level-MR_LMID copy: smaller h => smaller remainder).
// Level-0 bands enter with their exact sums.  total[c] = sum over bands.
__global__ void mr_total_kernel(const MrDevBand* __restrict__ bands, int B, i64 n_points,
                                const cplx<float>* __restrict__ wbuf, const cplx<float>* __restrict__ midbuf,
                                const double* __restrict__ band_sum, double* __restrict__ band_sum_est,
                                double* __restrict__ total) {
    __shared__ double scratch[32];
    const i64 c = blockIdx.x;
    double s = 0.0;
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        const MrDevBand band = bands[b];
        double est;
        if (band.level == 0) {
            est = band_sum[c * B + b];
        } else {
            const int lvl = band.level > MR_LMID ? MR_LMID : band.level;
            const i64 m = n_points >> lvl;
            const cplx<float>* w = (band.level > MR_LMID ? midbuf + band.mid_off + c * band.mid_stride
                                                          : wbuf + band.w_off + c * band.w_stride) + MR_HALO;
            const double h = (double)(1ll << lvl);
            const double p0 = norm2(w[0]), pn = norm2(w[m]);
            const double d0 = ((double)norm2(w[1]) - (double)norm2(w[-1])) / (2.0 * h);
            const double dn = ((double)norm2(w[m + 1]) - (double)norm2(w[m - 1])) / (2.0 * h);
            est = h * band_sum_est[c * B + b] + 0.5 * (h - 1.0) * (pn - p0) - (h * h - 1.0) / 12.0 * (dn - d0);
        }
        band_sum_est[c * B + b] = est;
        s += est;
    }
    s = block_sum(s, scratch);
    if (threadIdx.x == 0) total[c] = s;
}

// information plane + entropy sums of the rows the level-0 kernel wrote (their power is already in HBM)
__global__ void __launch_bounds__(256)
mr_info_rows_kernel(const float4* __restrict__ p, const double* __restrict__ total, int B, int b_first, i64 T4,
                    float eps, float4* __restrict__ o_info, double* __restrict__ ent_sum) {
    __shared__ double scratch[32];
    const i64 c = blockIdx.z;
    const int b = b_first + blockIdx.y;
    const i64 row = (c * B + b) * T4;
    const float inv = (float)(1.0 / total[c]);
    const i64 chunk = (T4 + gridDim.x - 1) / gridDim.x;
    const i64 t0 = (i64)blockIdx.x * chunk;
    const i64 t1 = t0 + chunk < T4 ? t0 + chunk : T4;
    double acc = 0.0;
    auto one = [&](const float4 v, i64 t) {
        const float d0 = fmaf(v.x, inv, eps), d1 = fmaf(v.y, inv, eps), d2 = fmaf(v.z, inv, eps), d3 = fmaf(v.w, inv, eps);
        const float i0 = -mr_fast_log2f(d0), i1 = -mr_fast_log2f(d1), i2 = -mr_fast_log2f(d2), i3 = -mr_fast_log2f(d3);
        o_info[row + t] = make_float4(i0, i1, i2, i3);
        acc += (double)((d0 * i0 + d1 * i1) + (d2 * i2 + d3 * i3));   // eps inside the weight, as in the fused expand pass
    };
    i64 t = t0 + threadIdx.x;
    for (; t + 3 * (i64)blockDim.x < t1; t += 4 * (i64)blockDim.x) {       // four independent 128-bit loads in flight
        const float4 v0 = p[row + t], v1 = p[row + t + blockDim.x];
        const float4 v2 = p[row + t + 2 * blockDim.x], v3 = p[row + t + 3 * blockDim.x];
        one(v0, t); one(v1, t + blockDim.x); one(v2, t + 2 * blockDim.x); one(v3, t + 3 * blockDim.x);
    }
    for (; t < t1; t += blockDim.x) one(p[row + t], t);
    acc = block_sum(acc, scratch);
    if (threadIdx.x == 0 && ent_sum) atomicAdd(&ent_sum[c * B + b], acc);
}

static int mr_run(const float* sig, i64 C, i64 N, i64 stride, const QiMrBand* hb, int B, float* out_power,
                  cplx<float>* out_complex, double* band_sum, float* out_info, double* entropy_sum,
                  double* band_sum_est, double* total_power, double eps, int phase, void* ws, size_t ws_bytes,
                  cudaStream_t st) {
    const bool fused = out_info != nullptr;
    if (fused && (!out_power || !band_sum || !band_sum_est || !total_power || out_complex)) return QI_ERR_ARG;
    if (!fused && phase != QI_MR_PHASE_ALL) return QI_ERR_ARG;
    MrPlan pl;
    int rc = mr_plan(C, N, hb, B, pl, /*allow_env=*/out_complex == nullptr);
    if (rc != QI_OK) return rc;
    if (ws_bytes < pl.total) return QI_ERR_WORKSPACE;
    if (C > 65535 || B > 65535) return QI_ERR_UNSUPPORTED;
    unsigned char* base = static_cast<unsigned char*>(ws);
    MrDevBand* d_bands = reinterpret_cast<MrDevBand*>(base + pl.off_bands);
    int* d_list = reinterpret_cast<int*>(base + pl.off_list);
    int* d_deep = reinterpret_cast<int*>(base + pl.off_deep);
    double* d_prefix = reinterpret_cast<double*>(base + pl.off_prefix);
    float2* d_group = reinterpret_cast<float2*>(base + pl.off_group);
    const int E = pl.n_edge;
    cplx<float>* midbuf = reinterpret_cast<cplx<float>*>(base + pl.off_mid);
    float4* tw2k = reinterpret_cast<float4*>(base + pl.off_tw);
    float* pyr = reinterpret_cast<float*>(base + pl.off_pyr);
    cplx<float>* tables = reinterpret_cast<cplx<float>*>(base + pl.off_tables);
    cplx<float>* wbuf = reinterpret_cast<cplx<float>*>(base + pl.off_w);
    const HbTaps taps = make_taps();

    stage_to_device(d_bands, pl.bands.data(), sizeof(MrDevBand) * (size_t)(B + E), st);
    if (!pl.expand_list.empty()) stage_to_device(d_list, pl.expand_list.data(), sizeof(int) * pl.expand_list.size(), st);
    if (!pl.deep_list.empty()) stage_to_device(d_deep, pl.deep_list.data(), sizeof(int) * pl.deep_list.size(), st);
    const bool do_front = phase != QI_MR_PHASE_EXPAND;      // tables, pyramid, level convolutions, estimates
    const bool do_back = phase != QI_MR_PHASE_ESTIMATE;     // expansion to the full rate
    if (do_front) {
        if (band_sum) cudaMemsetAsync(band_sum, 0, sizeof(double) * (size_t)C * B, st);
        if (band_sum_est) cudaMemsetAsync(band_sum_est, 0, sizeof(double) * (size_t)C * B, st);
    }
    if (do_back && entropy_sum) cudaMemsetAsync(entropy_sum, 0, sizeof(double) * (size_t)C * B, st);

    // T: kernel tables (one CTA per band)
    prof_set_category(QI_CAT_FFT_FWD);
    if (do_front) {
        const size_t smem = (size_t)4096 * 3 * sizeof(cplx<float>);
#ifndef QI_EMUL
        cudaFuncSetAttribute(mr_table_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
#endif
        QI_LAUNCH(mr_table_kernel, dim3((unsigned)(B + E)), dim3(256), smem, st, (const MrDevBand*)d_bands, N, 2047, tables);
        QI_LAUNCH(mr_twiddle2k_kernel, dim3((L2K_TW_TOTAL + 255) / 256), dim3(256), 0, st, tw2k);
    }
    // P: pyramid
    int first_level = 1;
    if (do_front) {                     // levels 1 - 3 in one pass over the record (cap >= 3: records of >= 2^13 samples)
        dim3 grid((unsigned)((pl.lvl_len[3] + P3_T - 1) / P3_T), (unsigned)C);
        QI_LAUNCH(mr_pyramid3_kernel, grid, dim3(256), 0, st, sig, stride, N, pyr + pl.lvl_off[1], pyr + pl.lvl_off[2],
                  pyr + pl.lvl_off[3], pl.pyr_per_chan, taps, E > 0 ? d_prefix : nullptr, pl.n_prefix, d_group);
        if (E > 0) QI_LAUNCH(mr_prefix_scan_kernel, dim3((unsigned)(2 * C)), dim3(1024), 0, st, d_prefix, pl.n_prefix);
        first_level = 4;
    }
    for (int l = first_level; do_front && l <= pl.cap; ++l) {
        const float* src = l == 1 ? sig : pyr + pl.lvl_off[l - 1];
        const i64 src_stride = l == 1 ? stride : pl.pyr_per_chan;
        const i64 src_len = l == 1 ? N : pl.lvl_len[l - 1];
        dim3 grid((unsigned)((pl.lvl_len[l] + DEC_TILE - 1) / DEC_TILE), (unsigned)C);
        QI_LAUNCH(mr_decimate_kernel, grid, dim3(256), 0, st, src, src_stride, src_len, l == 1 ? 0 : MR_HALO,
                  pyr + pl.lvl_off[l], pl.pyr_per_chan, pl.lvl_len[l], taps);
    }
    // A: level convolutions (deepest first; level 0 last so its epilogue traffic is contiguous in time).  Levels >= 1
    // whose grids are only a few CTAs are collected into merged launches.
    int level0_first = 0, level0_count = 0;
    MrMultiLevel multi;
    multi.n = 0;
    auto flush_multi = [&]() {
        if (!multi.n) return;
        prof_set_category(QI_CAT_INV_FIRST);
#ifndef QI_EMUL
        cudaFuncSetAttribute(mr_level2k_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L2K_SMEM);
#endif
        QI_LAUNCH(mr_level2k_multi_kernel, dim3((unsigned)multi.cta_end[multi.n - 1], (unsigned)C), dim3(L2K_THREADS),
                  L2K_SMEM, st, multi, (const MrDevBand*)d_bands, (const cplx<float>*)tables, (const float4*)tw2k, wbuf);
        multi.n = 0;
    };
    for (const MrLevelGeom& g0 : pl.levels) {
        if (g0.level == 0) { level0_first = g0.band_first; level0_count = g0.band_count; }
        if (!do_front) continue;
        MrLevelGeom g = g0;
        const float* x = g.level ? pyr + pl.lvl_off[g.level] : sig;
        g.x_stride = g.level ? pl.pyr_per_chan : stride;
        const int F = 1 << g.logF;
        prof_set_category(g.level ? QI_CAT_INV_FIRST : QI_CAT_INV_MID);
        // level 0: exact band sums; levels 1..MR_LMID in the fused mode: raw sums for the power estimate
        double* sum_dst = g.level == 0 ? band_sum : ((fused && g.level + g.env <= MR_LMID) ? band_sum_est : nullptr);
        if (g.no_sums) sum_dst = nullptr;
        if (g.logF == L2K_LOGF && g.band_count <= L2K_MAXB) {
            // 2048-point blocks: pairs of blocks per CTA, a few pairs in sequence so the twiddle copy is amortised
            const i64 pairs = (g.n_blocks + 1) / 2;
            i64 ppc = pairs * C / (148 * 2 * 8);
            ppc = ppc < 1 ? 1 : (ppc > 4 ? 4 : ppc);
            const i64 ctas = (pairs + ppc - 1) / ppc;
            if (g.level > 0 && ctas * C <= 148 * 2) {            // less than one wave: goes into a merged launch
                const int i = multi.n++;
                multi.g[i] = g; multi.x[i] = x; multi.sum[i] = sum_dst; multi.ppc[i] = (int)ppc;
                multi.cta_end[i] = (i ? multi.cta_end[i - 1] : 0) + (int)ctas;
                if (multi.n == L2K_MULTI) flush_multi();
                continue;
            }
            flush_multi();
            dim3 grid2((unsigned)ctas, (unsigned)C);
#ifndef QI_EMUL
            cudaFuncSetAttribute(mr_level2k_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L2K_SMEM);
            cudaFuncSetAttribute(mr_level2k_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L2K_SMEM);
#endif
            if (g.env)
                QI_LAUNCH((mr_level2k_kernel<true>), grid2, dim3(L2K_THREADS), L2K_SMEM, st, x, g, (const MrDevBand*)d_bands,
                          (const cplx<float>*)tables, (const float4*)tw2k, wbuf, out_power, out_complex, sum_dst, (int)ppc);
            else
                QI_LAUNCH((mr_level2k_kernel<false>), grid2, dim3(L2K_THREADS), L2K_SMEM, st, x, g, (const MrDevBand*)d_bands,
                          (const cplx<float>*)tables, (const float4*)tw2k, wbuf, out_power, out_complex, sum_dst, (int)ppc);
            continue;
        }
        const i64 gx = (g.n_blocks + g.TC - 1) / g.TC;
        const int gz = gx * C < 148 ? g.band_count : 1;           // few blocks: spread the bands instead
        dim3 grid((unsigned)gx, (unsigned)C, (unsigned)gz);
        const size_t smem = ((size_t)F * (g.TC + 1) * 2 + F) * sizeof(cplx<float>) + 256;
#ifndef QI_EMUL
        cudaFuncSetAttribute(mr_level_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
#endif
        QI_LAUNCH(mr_level_kernel, grid, dim3(1024), smem, st, x, g, (const MrDevBand*)d_bands,
                  (const cplx<float>*)tables, wbuf, out_power, out_complex, sum_dst);
    }
    if (do_front) flush_multi();
    // E: expand -- deep bands first to level MR_LMID (1/32 of the cells), then everything to the full rate
    MrExpandArgs ea;
    ea.bands = d_bands; ea.n_bands = B; ea.n_points = N; ea.wbuf = wbuf; ea.midbuf = midbuf;
    ea.out_power = out_power; ea.out_complex = out_complex; ea.band_sum = band_sum;
    ea.out_info = out_info; ea.band_sum_est = band_sum_est; ea.entropy_sum = entropy_sum;
    ea.total_power = total_power; ea.eps = (float)eps;
    ea.x = sig; ea.x_stride = stride; ea.prefix = d_prefix; ea.n_prefix = pl.n_prefix; ea.group_prefix = d_group;
    // both lists are ordered deepest level first, so the bands sharing a polyphase factor 2^k are contiguous
    auto launch_groups = [&](const std::vector<int>& list, const int* d_idx, int dst_level, i64 n_dst, int mode) {
        size_t pos = 0;
        while (pos < list.size()) {
            const int lr0 = pl.bands[list[pos]].level - dst_level;
            const int k = lr0 < 3 ? lr0 : 3;
            // edge source bands form their own group at the full rate (the running sums are added there)
            const bool edge = mode != MR_MODE_MID && (pl.bands[list[pos]].flags & MR_FLAG_EDGE_SRC);
            size_t end = pos;
            while (end < list.size() && end - pos < (size_t)MR_EXPAND_MAXB) {
                const int lr = pl.bands[list[end]].level - dst_level;
                if ((lr < 3 ? lr : 3) != k) break;
                if ((mode != MR_MODE_MID && (pl.bands[list[end]].flags & MR_FLAG_EDGE_SRC)) != edge) break;
                ++end;
            }
            ea.band_list = d_idx + pos;
            MrBandBlob blob;
            for (size_t i = pos; i < end; ++i) blob.b[i - pos] = pl.bands[list[i]];
            const i64 tile = (i64)MR_SEGQ << 3;          // per CTA, for every k (see mr_expand_kernel)
            dim3 grid((unsigned)((n_dst + tile - 1) / tile), (unsigned)(end - pos), (unsigned)C);
            if (edge) {             // record-long atoms live at level >= 3: always the x8 interpolator
                if (mode == MR_MODE_POWER) QI_LAUNCH((mr_expand_kernel<MR_MODE_POWER, false, true>), grid, dim3(256), 0, st, ea, taps, blob);
                else QI_LAUNCH((mr_expand_kernel<MR_MODE_POWER_INFO, false, true>), grid, dim3(256), 0, st, ea, taps, blob);
            } else if (k < 3) {
                if (mode == MR_MODE_MID) QI_LAUNCH((mr_expand_kernel<MR_MODE_MID, true>), grid, dim3(256), 0, st, ea, taps, blob);
                else if (mode == MR_MODE_POWER) QI_LAUNCH((mr_expand_kernel<MR_MODE_POWER, true>), grid, dim3(256), 0, st, ea, taps, blob);
                else QI_LAUNCH((mr_expand_kernel<MR_MODE_POWER_INFO, true>), grid, dim3(256), 0, st, ea, taps, blob);
            } else {
                if (mode == MR_MODE_MID) QI_LAUNCH((mr_expand_kernel<MR_MODE_MID, false>), grid, dim3(256), 0, st, ea, taps, blob);
                else if (mode == MR_MODE_POWER) QI_LAUNCH((mr_expand_kernel<MR_MODE_POWER, false>), grid, dim3(256), 0, st, ea, taps, blob);
                else QI_LAUNCH((mr_expand_kernel<MR_MODE_POWER_INFO, false>), grid, dim3(256), 0, st, ea, taps, blob);
            }
            pos = end;
        }
    };
    if (do_front) {
        prof_set_category(QI_CAT_INV_FIRST);
        // level-MR_LMID pass of the deep bands: only the band-power estimates need it (the expansion reads the bands' own samples)
        if (fused && !pl.deep_list.empty())
            launch_groups(pl.deep_list, d_deep, MR_LMID, (N >> MR_LMID) + 2 * MR_HALO, MR_MODE_MID);
        if (fused) {
            // raw sums are in band_sum_est (level kernels / the MID pass); finish the estimates and the totals
            QI_LAUNCH(mr_total_kernel, dim3((unsigned)C), dim3(128), 0, st, (const MrDevBand*)d_bands, B, N,
                      (const cplx<float>*)wbuf, (const cplx<float>*)midbuf, (const double*)band_sum, band_sum_est,
                      total_power);
        }
    }
    if (do_back) {
        prof_set_category(QI_CAT_INV_LAST);
        if (!pl.expand_list.empty())
            launch_groups(pl.expand_list, d_list, 0, N, fused ? MR_MODE_POWER_INFO : MR_MODE_POWER);
        if (fused && level0_count > 0) {
            prof_set_category(QI_CAT_INFO);
            const i64 T4 = N / 4;
            i64 splits = (148 * 8 * 16 + (i64)level0_count * C - 1) / ((i64)level0_count * C);
            if (splits > (T4 + 8191) / 8192) splits = (T4 + 8191) / 8192;
            if (splits < 1) splits = 1;
            dim3 grid((unsigned)splits, (unsigned)level0_count, (unsigned)C);
            QI_LAUNCH(mr_info_rows_kernel, grid, dim3(256), 0, st, reinterpret_cast<const float4*>(out_power),
                      (const double*)total_power, B, level0_first, T4, (float)eps, reinterpret_cast<float4*>(out_info),
                      entropy_sum);
        }
    }
    prof_set_category(QI_CAT_OTHER);
    return check_cuda("qi_cwt_multirate");
}

}  // namespace qi

extern "C" {

size_t qi_cwt_multirate_workspace_bytes(int64_t C, int64_t N, const QiMrBand* bands, int B) {
    if (C <= 0 || N <= 0 || B <= 0 || !bands) return 0;
    qi::MrPlan pl;
    if (qi::mr_plan(C, N, bands, B, pl, false) != QI_OK) return 0;
    qi::MrPlan pe;
    if (qi::mr_plan(C, N, bands, B, pe, true) != QI_OK) return 0;
    return pl.total > pe.total ? pl.total : pe.total;
}

int qi_cwt_multirate(const void* sig, int64_t C, int64_t N, int64_t stride, const QiMrBand* bands, int B,
                     void* out_power, void* out_complex, double* band_sum, void* out_info, double* entropy_sum,
                     double* band_sum_est, double* total_power, double eps, int phase, void* ws, size_t ws_bytes,
                     void* stream) {
    if (!sig || !bands || !ws || C <= 0 || N <= 0 || B <= 0 || stride < N) return QI_ERR_ARG;
    // vector loads / 256-bit plane stores: records 16-byte aligned with a stride that is a multiple of 4 samples (the
    // edge rows read the record as float4 in mr_expand_kernel), planes 32-byte aligned
    if (((uintptr_t)sig & 15) || (stride & 3) || ((uintptr_t)out_power & 31) || ((uintptr_t)out_info & 31) ||
        ((uintptr_t)out_complex & 31))
        return QI_ERR_ARG;
    if (!out_power && !out_complex && !band_sum) return QI_ERR_ARG;
    if (phase < QI_MR_PHASE_ALL || phase > QI_MR_PHASE_EXPAND) return QI_ERR_ARG;
    return qi::mr_run(static_cast<const float*>(sig), C, N, stride, bands, B, static_cast<float*>(out_power),
                      static_cast<qi::cplx<float>*>(out_complex), band_sum, static_cast<float*>(out_info),
                      entropy_sum, band_sum_est, total_power, eps, phase, ws, ws_bytes,
                      static_cast<cudaStream_t>(stream));
}

}  // extern "C"
