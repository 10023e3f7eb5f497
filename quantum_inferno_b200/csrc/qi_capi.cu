// qi_capi.cu -- extern "C" boundary of libqi_b200.so (see include/qi_b200.h).
#include "qi_fft.cuh"
#include "qi_host.h"

#include <string.h>
#include <atomic>
#include <mutex>
#include <vector>

namespace qi {

thread_local char g_last_cuda_error[256] = {0};

// ---------------------------------------------------------------- launch accounting / event timing
#ifndef QI_EMUL
namespace {
struct ProfRec { cudaEvent_t a, b; int cat; };
std::mutex g_prof_mu;
std::vector<ProfRec> g_prof_recs;
std::atomic<long long> g_launches{0};
std::atomic<int> g_prof_on{0};
thread_local int g_prof_cat = QI_CAT_OTHER;
thread_local cudaEvent_t g_prof_pending = nullptr;
}  // namespace
void prof_set_category(int cat) { g_prof_cat = cat; }
void prof_begin(cudaStream_t st) {
    g_launches.fetch_add(1);
    if (!g_prof_on.load()) return;
    cudaEventCreate(&g_prof_pending);
    cudaEventRecord(g_prof_pending, st);
}
void prof_end(cudaStream_t st) {
    if (!g_prof_pending) return;
    ProfRec r;
    r.a = g_prof_pending; r.cat = g_prof_cat;
    g_prof_pending = nullptr;
    cudaEventCreate(&r.b);
    cudaEventRecord(r.b, st);
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof_recs.push_back(r);
}
#endif

#ifdef QI_EMUL
void stage_to_device(void* dst, const void* src, size_t bytes, cudaStream_t) { memcpy(dst, src, bytes); }
#else
// The table travels in the kernel's parameter space and a few threads write it out: no copy engine is involved, so the
// transfer can never queue behind a bulk host->device copy that another stream has in flight (measured: with
// cudaMemcpyAsync the first kernel of a call waited for the WHOLE 128 MB record copy of the next channel group).
namespace {
struct StageBlob { unsigned q[768]; };                // 3 KB per launch, inside the 4 KB parameter space
__global__ void stage_blob_kernel(StageBlob blob, unsigned* __restrict__ dst, int n4) {
    for (int i = threadIdx.x; i < n4; i += blockDim.x) dst[i] = blob.q[i];
}
}  // namespace
void stage_to_device(void* dst, const void* src, size_t bytes, cudaStream_t st) {
    // every table of this library is an array of 4- or 8-byte fields: whole 32-bit words
    const unsigned char* s = static_cast<const unsigned char*>(src);
    unsigned char* d = static_cast<unsigned char*>(dst);
    while (bytes > 0) {
        const size_t chunk = bytes < sizeof(StageBlob) ? bytes : sizeof(StageBlob);
        StageBlob blob;
        memcpy(&blob, s, chunk);
        stage_blob_kernel<<<1, 256, 0, st>>>(blob, reinterpret_cast<unsigned*>(d), (int)((chunk + 3) / 4));
        s += chunk; d += chunk; bytes -= chunk;
    }
}
#endif

int check_cuda(const char* where) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        snprintf(g_last_cuda_error, sizeof(g_last_cuda_error), "%s: %s", where, cudaGetErrorString(e));
        return QI_ERR_CUDA;
    }
    return QI_OK;
}

template <typename T>
static int fft_c2c_impl(const void* in, void* out, i64 batch, int log2n, int inverse, cudaStream_t st) {
    const FftPlan plan = make_plan(log2n, (int)sizeof(cplx<T>));
    const i64 n = 1ll << log2n;
    const SrcComplex<T> src{static_cast<const cplx<T>*>(in), n};
    cplx<T>* dstp = static_cast<cplx<T>*>(out);
    if (!inverse) {
        forward_passes<T>(plan, batch, src, dstp, n, st);
    } else {
        inverse_passes<T>(plan, batch, src, DstComplex<T>{dstp, n, (T)(1.0 / (double)n)}, 0, false, dstp, n, st);
        prof_set_category(QI_CAT_OTHER);
    }
    return check_cuda("qi_fft_c2c");
}

// natural-order one-sided spectrum out of the bit-reversed full spectrum
template <typename T>
__global__ void half_spectrum_gather_kernel(const cplx<T>* spec, int logn, cplx<T>* out) {
    const i64 n = 1ll << logn;
    const i64 k = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    const i64 m = blockIdx.y;
    if (k > n / 2) return;
    out[m * (n / 2 + 1) + k] = spec[m * n + (i64)brev_bits((unsigned)k, logn)];
}

template <typename T>
static int rfft_impl(const void* sig, i64 M, i64 n, i64 stride, void* out, void* ws, size_t ws_bytes, cudaStream_t st) {
    int logn = 0;
    while ((1ll << logn) < n) ++logn;
    if ((1ll << logn) != n) return QI_ERR_ARG;
    if (ws_bytes < sizeof(cplx<T>) * (size_t)M * n) return QI_ERR_WORKSPACE;
    if (M > 65535) return QI_ERR_UNSUPPORTED;
    cplx<T>* spec = static_cast<cplx<T>*>(ws);
    const FftPlan plan = make_plan(logn, (int)sizeof(cplx<T>));
    forward_passes<T>(plan, M, SrcRealPad<T>{static_cast<const T*>(sig), stride, n}, spec, n, st);
    dim3 grid((unsigned)((n / 2 + 1 + 255) / 256), (unsigned)M);
    QI_LAUNCH((half_spectrum_gather_kernel<T>), grid, dim3(256), 0, st, (const cplx<T>*)spec, logn, static_cast<cplx<T>*>(out));
    return check_cuda("qi_rfft");
}

}  // namespace qi

extern "C" {

int qi_rfft(const void* sig, int64_t M, int64_t n, int64_t stride, int dtype, void* out, void* ws, size_t ws_bytes,
            void* stream) {
    if (!sig || !out || !ws || M <= 0 || n <= 0 || stride < n) return QI_ERR_ARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (dtype == QI_F32) return qi::rfft_impl<float>(sig, M, n, stride, out, ws, ws_bytes, st);
    if (dtype == QI_F64) return qi::rfft_impl<double>(sig, M, n, stride, out, ws, ws_bytes, st);
    return QI_ERR_ARG;
}

int qi_abi_version(void) { return QI_ABI_VERSION; }

#ifndef QI_EMUL
int64_t qi_launch_count(void) { return qi::g_launches.load(); }
int qi_profile_enable(int on) { qi::g_prof_on.store(on ? 1 : 0); return QI_OK; }
int qi_profile_read(double* total_ms, int64_t* launches) {
    if (!total_ms || !launches) return QI_ERR_ARG;
    for (int i = 0; i < QI_N_CATEGORIES; ++i) { total_ms[i] = 0.0; launches[i] = 0; }
    std::lock_guard<std::mutex> lk(qi::g_prof_mu);
    for (auto& r : qi::g_prof_recs) {
        cudaEventSynchronize(r.b);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, r.a, r.b);
        if (r.cat >= 0 && r.cat < QI_N_CATEGORIES) { total_ms[r.cat] += ms; launches[r.cat] += 1; }
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
    }
    qi::g_prof_recs.clear();
    return qi::check_cuda("qi_profile_read");
}
#else
int64_t qi_launch_count(void) { return 0; }
int qi_profile_enable(int) { return QI_OK; }
int qi_profile_read(double* total_ms, int64_t* launches) {
    for (int i = 0; i < QI_N_CATEGORIES; ++i) { if (total_ms) total_ms[i] = 0.0; if (launches) launches[i] = 0; }
    return QI_OK;
}
#endif

const char* qi_error_string(int code) {
    switch (code) {
        case QI_OK: return "ok";
        case QI_ERR_ARG: return "invalid argument";
        case QI_ERR_WORKSPACE: return "workspace too small";
        case QI_ERR_CUDA: return "CUDA error";
        case QI_ERR_UNSUPPORTED: return "unsupported configuration";
        default: return "unknown error";
    }
}

const char* qi_last_cuda_error(void) { return qi::g_last_cuda_error; }

int qi_fft_c2c(const void* in, void* out, int64_t batch, int log2n, int inverse, int dtype, void* stream) {
    if (!in || !out || batch <= 0 || log2n < 0 || log2n > 30) return QI_ERR_ARG;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (dtype == QI_F32) return qi::fft_c2c_impl<float>(in, out, batch, log2n, inverse, st);
    if (dtype == QI_F64) return qi::fft_c2c_impl<double>(in, out, batch, log2n, inverse, st);
    return QI_ERR_ARG;
}

}  // extern "C"
