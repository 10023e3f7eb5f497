// TEST INFRASTRUCTURE ONLY: runs the level-convolution kernel of qi_mr_level2k.cuh on the CPU emulator with a
// caller-made geometry and caller-made band tables (one channel), for tests/test_level2k_radix16.py.
#include "qi_mr_level2k.cuh"

using namespace qi;

extern "C" int l2k_run(const float* x, int64_t x_len, int x_halo, int64_t q_first, int level, int env,
                       int64_t n_points, int64_t n_level, int64_t n_out, int64_t n_blocks, int wk, int band_count,
                       const float* tables, const int* demod, int pairs_per_cta, float* out_power, float* out_complex,
                       float* wbuf, int64_t w_stride, double* band_sum) {
    if (band_count > L2K_MAXB || wk % 2) return 1;
    std::vector<float4> tw(L2K_TW_TOTAL);
    float4* twd = tw.data();                               // the launch captures by value: pass the pointer
    QI_LAUNCH(mr_twiddle2k_kernel, dim3((L2K_TW_TOTAL + 255) / 256), dim3(256), 0, 0, twd);
    std::vector<MrDevBand> bands(band_count);
    for (int b = 0; b < band_count; ++b) {
        MrDevBand d = {};
        d.level = env ? level + 1 : level;
        d.conv_level = level;
        d.demod = demod[b];
        d.logF = L2K_LOGF;
        d.table_off = (long long)b * L2K_F;
        d.w_off = (long long)b * w_stride;
        d.w_stride = w_stride;
        bands[b] = d;
    }
    MrLevelGeom g = {};
    g.level = level; g.logF = L2K_LOGF; g.TC = 0;
    g.band_first = 0; g.band_count = band_count; g.n_bands = band_count;
    g.wk = wk; g.n_points = n_points; g.n_level = n_level; g.q_first = q_first; g.n_out = n_out; g.n_blocks = n_blocks;
    g.x_stride = x_len; g.x_len = x_len; g.x_halo = x_halo; g.env = env; g.no_sums = 0;
    const dim3 grid((unsigned)((n_blocks + 2 * pairs_per_cta - 1) / (2 * pairs_per_cta)), 1);
    // the caller's tables are in bit-reversed bin order; the kernel reads them in the warp order of mr_table_kernel
    std::vector<cplx<float>> perm((size_t)band_count * L2K_F);
    for (int b = 0; b < band_count; ++b)
        for (int r = 0; r < L2K_F; ++r)
            perm[(size_t)b * L2K_F + l2k_tab_slot(r)] = mk<float>(tables[2 * ((size_t)b * L2K_F + r)],
                                                                  tables[2 * ((size_t)b * L2K_F + r) + 1]);
    const cplx<float>* tab = perm.data();
    cplx<float>* wb = reinterpret_cast<cplx<float>*>(wbuf);
    cplx<float>* oc = reinterpret_cast<cplx<float>*>(out_complex);
    const float4* twp = tw.data();
    const MrDevBand* bp = bands.data();
    if (level == 0 && !env)
        QI_LAUNCH((mr_level2k_kernel<false>), grid, dim3(L2K_THREADS), L2K_SMEM, 0, x, g, bp, tab, twp, wb, out_power, oc,
                  band_sum, pairs_per_cta);
    else
        QI_LAUNCH((mr_level2k_kernel<true>), grid, dim3(L2K_THREADS), L2K_SMEM, 0, x, g, bp, tab, twp, wb, out_power, oc,
                  band_sum, pairs_per_cta);
    return 0;
}
