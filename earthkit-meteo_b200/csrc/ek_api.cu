// ek_api.cu -- library-level entry points: version, errors, launch configuration, the field partitioner
// and the host-buffer pipeline.
#include <cstring>
#include <vector>

#include "ek_launch.cuh"

namespace ek {

std::atomic<int> g_ctas_per_sm{16};
std::atomic<uint64_t> g_launches{0};

static thread_local char t_err[512] = "";

int set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(t_err, sizeof(t_err), fmt, ap);
    va_end(ap);
    return code;
}

int sm_count_current_device() {
    static std::atomic<int> cache[64];
    int dev = -1;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0) return -1;
    if (dev < 64) {
        int v = cache[dev].load(std::memory_order_relaxed);
        if (v > 0) return v;
    }
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return -1;
    if (dev < 64) cache[dev].store(sms, std::memory_order_relaxed);
    return sms;
}

}  // namespace ek

using namespace ek;

extern "C" EK_EXPORT int ek_thermo_version(void) { return EK_THERMO_VERSION; }
extern "C" EK_EXPORT const char* ek_thermo_last_error(void) { return t_err; }
extern "C" EK_EXPORT uint64_t ek_thermo_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

extern "C" EK_EXPORT int ek_thermo_set_launch_config(int threads, int ctas_per_sm) {
    if (threads != 0 && threads != kThreads) return set_error(EK_ERR_ARG, "threads=%d: the CTA size is fixed at build time (%d)", threads, kThreads);
    if (ctas_per_sm != 0) {
        if (ctas_per_sm < 1 || ctas_per_sm > 4096) return set_error(EK_ERR_ARG, "ctas_per_sm=%d out of range", ctas_per_sm);
        g_ctas_per_sm.store(ctas_per_sm);
    }
    return EK_OK;
}

// Contiguous, aligned shards of a flat index range (SURVEY.md §8(e)): the first (units % world) ranks get
// one extra unit of `align` points; the last shard absorbs the sub-unit remainder.
extern "C" EK_EXPORT int ek_thermo_shard_range(int64_t n, int world, int rank, int64_t align, int64_t* begin, int64_t* end) {
    if (n < 0 || world < 1 || rank < 0 || rank >= world || align < 1 || !begin || !end)
        return set_error(EK_ERR_ARG, "shard_range: bad arguments n=%lld world=%d rank=%d align=%lld", (long long)n, world, rank, (long long)align);
    const int64_t units = n / align;
    const int64_t base = units / world, extra = units % world;
    const int64_t b = (rank * base + (rank < extra ? rank : extra)) * align;
    int64_t e = b + (base + (rank < extra ? 1 : 0)) * align;
    if (rank == world - 1) e = n;
    *begin = b;
    *end = e;
    return EK_OK;
}

// defined in ek_ops_fused_*.cu / ek_hybrid.cu (so the suite kernels are instantiated in one translation unit only)
template <typename T> int ek_suite_launch_tqp(const ek_operand* ins, void* const* outs, uint32_t mask, int ept_method, int64_t n, void* stream);
template <typename T> int ek_suite_launch_ttdp(const ek_operand* ins, void* const* outs, uint32_t mask, int ept_method, int64_t n, void* stream);
template <typename T>
int ek_suite_launch_hybrid(const void* t, const void* q, const void* sp, const void* A, const void* B, int nlev, int64_t npl, void* const* outs,
                           uint32_t out_mask, int ept_method, void* stream);
template <typename T>
int ek_suite_launch_hybrid_geo(const void* t, const void* q, const void* sp, const void* zs, const void* A, const void* B, int nlev, int64_t npl,
                               void* const* outs, uint32_t out_mask, int ept_method, int top_toa, double alpha_top, void* const* cols,
                               int height_mode, void* stream);

// ---- host-buffer pipeline ---------------------------------------------------------------------------
namespace {
// The pipeline's streams.  The destructor drains them before destroying them: on an error path earlier chunks' async
// copies may still be reading or writing the caller's host buffers, and the caller is free to release those as soon as
// the entry point returns.
struct StreamSet {
    std::vector<cudaStream_t> s;
    ~StreamSet() {
        for (auto st : s) cudaStreamSynchronize(st);
        for (auto st : s) cudaStreamDestroy(st);
    }
    int create(int n) {
        for (int i = 0; i < n; ++i) {
            cudaStream_t st;
            cudaError_t e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
            if (e != cudaSuccess) return set_error((int)e, "host pipeline: cudaStreamCreate: %s", cudaGetErrorString(e));
            s.push_back(st);
        }
        return EK_OK;
    }
    int drain() {
        for (auto st : s) {
            cudaError_t e = cudaStreamSynchronize(st);
            if (e != cudaSuccess) return set_error((int)e, "host pipeline: stream sync: %s", cudaGetErrorString(e));
        }
        return EK_OK;
    }
};

int count_outputs(const char* what, void* const* h_outs, uint32_t out_mask, int* n_out, bool allow_none = false) {
    if ((out_mask == 0 && !allow_none) || out_mask >= (1u << S_NSLOTS)) return set_error(EK_ERR_ARG, "%s: out_mask=0x%x", what, out_mask);
    *n_out = 0;
    for (int k = 0; k < S_NSLOTS; ++k)
        if ((out_mask >> k) & 1u) {
            if (!h_outs[k]) return set_error(EK_ERR_ARG, "%s: output %d requested but its buffer is NULL", what, k);
            ++*n_out;
        }
    return EK_OK;
}
}  // namespace

template <typename T>
static int impl_host_suite(int kind, const void* h_a, const void* h_b, const void* h_c, void* const* h_outs, uint32_t out_mask, int ept_method,
                           int64_t n, void* workspace, size_t workspace_bytes, int n_slots) {
    if (kind != 0 && kind != 1) return set_error(EK_ERR_ENUM, "host_suite: kind=%d", kind);
    if (!h_a || !h_b || !h_c || !h_outs || !workspace) return set_error(EK_ERR_ARG, "host_suite: NULL buffer");
    if (n < 0 || n_slots < 1 || n_slots > 16) return set_error(EK_ERR_ARG, "host_suite: n=%lld n_slots=%d", (long long)n, n_slots);
    int n_out = 0;
    if (int rc = count_outputs("host_suite", h_outs, out_mask, &n_out)) return rc;
    if (n == 0) return EK_OK;
    if (!aligned16(workspace)) return set_error(EK_ERR_ARG, "host_suite: workspace must be 16-byte aligned");
    const int n_arr = 3 + n_out;
    int64_t chunk = (int64_t)(workspace_bytes / ((size_t)n_slots * n_arr * sizeof(T)));
    chunk -= chunk % 4096;  // keeps every sub-buffer 16-byte aligned and tiles whole
    if (chunk <= 0) return set_error(EK_ERR_PIPE, "host_suite: workspace of %zu bytes is too small for %d slots", workspace_bytes, n_slots);
    if (chunk > n) chunk = ((n + 4095) / 4096) * 4096;

    StreamSet ss;
    if (int rc = ss.create(n_slots)) return rc;
    const T* hin[3] = {static_cast<const T*>(h_a), static_cast<const T*>(h_b), static_cast<const T*>(h_c)};
    T* ws = static_cast<T*>(workspace);
    int64_t done = 0;
    for (int64_t c = 0; done < n; ++c, done += chunk) {
        const int slot = (int)(c % n_slots);
        cudaStream_t st = ss.s[slot];
        const int64_t m = (n - done) < chunk ? (n - done) : chunk;
        T* base = ws + (int64_t)slot * n_arr * chunk;
        ek_operand ins[3];
        for (int k = 0; k < 3; ++k) {
            T* d = base + (int64_t)k * chunk;
            cudaError_t e = cudaMemcpyAsync(d, hin[k] + done, (size_t)m * sizeof(T), cudaMemcpyHostToDevice, st);
            if (e != cudaSuccess) return set_error((int)e, "host_suite: H2D copy: %s", cudaGetErrorString(e));
            ins[k].ptr = d;
            ins[k].value = 0.0;
        }
        void* douts[S_NSLOTS];
        int j = 0;
        for (int k = 0; k < S_NSLOTS; ++k) douts[k] = ((out_mask >> k) & 1u) ? (void*)(base + (int64_t)(3 + j++) * chunk) : nullptr;
        int rc = kind == 0 ? ek_suite_launch_tqp<T>(ins, douts, out_mask, ept_method, m, st) : ek_suite_launch_ttdp<T>(ins, douts, out_mask, ept_method, m, st);
        if (rc != EK_OK) return rc;
        for (int k = 0; k < S_NSLOTS; ++k)
            if (douts[k]) {
                cudaError_t e = cudaMemcpyAsync(static_cast<T*>(h_outs[k]) + done, douts[k], (size_t)m * sizeof(T), cudaMemcpyDeviceToHost, st);
                if (e != cudaSuccess) return set_error((int)e, "host_suite: D2H copy: %s", cudaGetErrorString(e));
            }
    }
    return ss.drain();
}
EK_API(host_suite,
       (int kind, const void* h_a, const void* h_b, const void* h_c, void* const* h_outs, uint32_t out_mask, int ept_method, int64_t n,
        void* workspace, size_t workspace_bytes, int n_slots),
       (kind, h_a, h_b, h_c, h_outs, out_mask, ept_method, n, workspace, workspace_bytes, n_slots))

// The hybrid-level suite fed from HOST arrays: t, q and every output are [nlev, npl] host arrays, sp is [npl], A / B the
// nlev + 1 half-level coefficients.  The pressure field never exists on either side of PCIe: 16 + 8/nlev bytes per point
// travel to the device instead of 24.  Chunks are column ranges of all levels; each array of a chunk moves as one 2-D
// copy (nlev rows of chunk-columns, host pitch npl).  With column outputs (h_cols: thickness, z, height; NULL or any entry
// NULL for none) the chunks run the suite + geopotential kernel instead, and zs travels as one more [npl] row when an output
// needs it.
template <typename T>
static int host_suite_tq_hybrid(const char* what, const void* h_t, const void* h_q, const void* h_sp, const void* h_zs, const void* h_A,
                                const void* h_B, int nlev, int64_t npl, void* const* h_outs, uint32_t out_mask, int ept_method, int top_toa,
                                double alpha_top, void* const* h_cols, int height_mode, void* workspace, size_t workspace_bytes, int n_slots) {
    if (!h_t || !h_q || !h_sp || !h_A || !h_B || !h_outs || !workspace) return set_error(EK_ERR_ARG, "%s: NULL buffer", what);
    if (nlev < 1 || npl < 0 || n_slots < 1 || n_slots > 16) return set_error(EK_ERR_ARG, "%s: nlev=%d npl=%lld n_slots=%d", what, nlev, (long long)npl, n_slots);
    int n_col = 0;
    for (int k = 0; k < 3; ++k) n_col += (h_cols && h_cols[k]) ? 1 : 0;
    const bool geo = n_col > 0;
    if (geo && h_cols[2] && (height_mode < EK_HM_THICKNESS || height_mode > EK_HM_GEOM_GROUND))
        return set_error(EK_ERR_ENUM, "%s: invalid height mode %d", what, height_mode);
    const bool zs_row = geo && (h_cols[1] || (h_cols[2] && height_mode != EK_HM_THICKNESS && height_mode != EK_HM_GH_GROUND));
    if (zs_row && !h_zs) return set_error(EK_ERR_ARG, "%s: this output needs the surface geopotential zs", what);
    int n_out = 0;
    if (int rc = count_outputs(what, h_outs, out_mask, &n_out, geo)) return rc;
    if (npl == 0) return EK_OK;
    if (!aligned16(workspace)) return set_error(EK_ERR_ARG, "%s: workspace must be 16-byte aligned", what);
    const size_t coef = (((size_t)(nlev + 1) * sizeof(T) + 255u) / 256u) * 256u;  // A, then B, at the start of the workspace
    if (workspace_bytes <= 2 * coef) return set_error(EK_ERR_PIPE, "%s: workspace of %zu bytes is too small", what, workspace_bytes);
    // device rows of one chunk: t, q, outputs, column outputs (nlev each) + sp (+ zs)
    const int64_t rows = (int64_t)(2 + n_out + n_col) * nlev + 1 + (zs_row ? 1 : 0);
    int64_t chunk = (int64_t)((workspace_bytes - 2 * coef) / ((size_t)n_slots * rows * sizeof(T)));
    chunk -= chunk % 1024;  // whole vectors, 16-byte aligned rows
    if (chunk <= 0) return set_error(EK_ERR_PIPE, "%s: workspace of %zu bytes is too small for %d slots of %d levels", what, workspace_bytes, n_slots, nlev);
    if (chunk > npl) chunk = ((npl + 1023) / 1024) * 1024;

    StreamSet ss;
    if (int rc = ss.create(n_slots)) return rc;
    unsigned char* wsb = static_cast<unsigned char*>(workspace);
    T* dA = reinterpret_cast<T*>(wsb);
    T* dB = reinterpret_cast<T*>(wsb + coef);
    T* ws = reinterpret_cast<T*>(wsb + 2 * coef);
    cudaEvent_t coef_ready;
    cudaError_t e = cudaEventCreateWithFlags(&coef_ready, cudaEventDisableTiming);
    if (e != cudaSuccess) return set_error((int)e, "%s: cudaEventCreate: %s", what, cudaGetErrorString(e));
    struct EventGuard {
        cudaEvent_t ev;
        ~EventGuard() { cudaEventDestroy(ev); }
    } guard{coef_ready};
    e = cudaMemcpyAsync(dA, h_A, (size_t)(nlev + 1) * sizeof(T), cudaMemcpyHostToDevice, ss.s[0]);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dB, h_B, (size_t)(nlev + 1) * sizeof(T), cudaMemcpyHostToDevice, ss.s[0]);
    if (e == cudaSuccess) e = cudaEventRecord(coef_ready, ss.s[0]);
    if (e != cudaSuccess) return set_error((int)e, "%s: coefficient copy: %s", what, cudaGetErrorString(e));
    const size_t hpitch = (size_t)npl * sizeof(T);
    int64_t done = 0;
    for (int64_t c = 0; done < npl; ++c, done += chunk) {
        const int slot = (int)(c % n_slots);
        cudaStream_t st = ss.s[slot];
        const int64_t m = (npl - done) < chunk ? (npl - done) : chunk;
        const size_t dpitch = (size_t)m * sizeof(T);  // the device copy of a chunk is a dense [nlev, m] array
        T* base = ws + (int64_t)slot * rows * chunk;
        T* d_t = base;
        T* d_q = base + (int64_t)nlev * chunk;
        T* d_sp = base + (int64_t)2 * nlev * chunk;
        if (c < n_slots && slot != 0) {
            e = cudaStreamWaitEvent(st, coef_ready, 0);
            if (e != cudaSuccess) return set_error((int)e, "%s: stream wait: %s", what, cudaGetErrorString(e));
        }
        e = cudaMemcpy2DAsync(d_t, dpitch, static_cast<const T*>(h_t) + done, hpitch, dpitch, (size_t)nlev, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpy2DAsync(d_q, dpitch, static_cast<const T*>(h_q) + done, hpitch, dpitch, (size_t)nlev, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_sp, static_cast<const T*>(h_sp) + done, dpitch, cudaMemcpyHostToDevice, st);
        T* d_zs = zs_row ? d_sp + chunk : nullptr;
        if (e == cudaSuccess && zs_row) e = cudaMemcpyAsync(d_zs, static_cast<const T*>(h_zs) + done, dpitch, cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) return set_error((int)e, "%s: H2D copy: %s", what, cudaGetErrorString(e));
        void* douts[S_NSLOTS];
        int j = 0;
        T* d_out0 = d_sp + (zs_row ? 2 : 1) * chunk;
        for (int k = 0; k < S_NSLOTS; ++k) douts[k] = ((out_mask >> k) & 1u) ? (void*)(d_out0 + (int64_t)(j++) * nlev * chunk) : nullptr;
        void* dcols[3];
        for (int k = 0; k < 3; ++k) dcols[k] = (geo && h_cols[k]) ? (void*)(d_out0 + (int64_t)(j++) * nlev * chunk) : nullptr;
        int rc = geo ? ek_suite_launch_hybrid_geo<T>(d_t, d_q, d_sp, d_zs, dA, dB, nlev, m, douts, out_mask, ept_method, top_toa, alpha_top, dcols,
                                                     height_mode, st)
                     : ek_suite_launch_hybrid<T>(d_t, d_q, d_sp, dA, dB, nlev, m, douts, out_mask, ept_method, st);
        if (rc != EK_OK) return rc;
        for (int k = 0; k < S_NSLOTS + 3; ++k) {
            void* h = k < S_NSLOTS ? h_outs[k] : (geo ? h_cols[k - S_NSLOTS] : nullptr);
            void* d = k < S_NSLOTS ? douts[k] : dcols[k - S_NSLOTS];
            if (d) {
                e = cudaMemcpy2DAsync(static_cast<T*>(h) + done, hpitch, d, dpitch, dpitch, (size_t)nlev, cudaMemcpyDeviceToHost, st);
                if (e != cudaSuccess) return set_error((int)e, "%s: D2H copy: %s", what, cudaGetErrorString(e));
            }
        }
    }
    return ss.drain();
}

template <typename T>
static int impl_host_suite_tq_hybrid(const void* h_t, const void* h_q, const void* h_sp, const void* h_A, const void* h_B, int nlev, int64_t npl,
                                     void* const* h_outs, uint32_t out_mask, int ept_method, void* workspace, size_t workspace_bytes,
                                     int n_slots) {
    return host_suite_tq_hybrid<T>("host_suite_tq_hybrid", h_t, h_q, h_sp, nullptr, h_A, h_B, nlev, npl, h_outs, out_mask, ept_method, 0, 0.0,
                                   nullptr, 0, workspace, workspace_bytes, n_slots);
}
EK_API(host_suite_tq_hybrid,
       (const void* h_t, const void* h_q, const void* h_sp, const void* h_A, const void* h_B, int nlev, int64_t npl, void* const* h_outs,
        uint32_t out_mask, int ept_method, void* workspace, size_t workspace_bytes, int n_slots),
       (h_t, h_q, h_sp, h_A, h_B, nlev, npl, h_outs, out_mask, ept_method, workspace, workspace_bytes, n_slots))

template <typename T>
static int impl_host_suite_tq_hybrid_geo(const void* h_t, const void* h_q, const void* h_sp, const void* h_zs, const void* h_A, const void* h_B,
                                         int nlev, int64_t npl, void* const* h_outs, uint32_t out_mask, int ept_method, int top_toa,
                                         double alpha_top, void* h_thickness, void* h_z, void* h_height, int height_mode, void* workspace,
                                         size_t workspace_bytes, int n_slots) {
    const char* what = "host_suite_tq_hybrid_geo";
    if (!h_thickness && !h_z && !h_height) return set_error(EK_ERR_ARG, "%s: no column output given (use host_suite_tq_hybrid)", what);
    void* const cols[3] = {h_thickness, h_z, h_height};
    return host_suite_tq_hybrid<T>(what, h_t, h_q, h_sp, h_zs, h_A, h_B, nlev, npl, h_outs, out_mask, ept_method, top_toa, alpha_top, cols,
                                   height_mode, workspace, workspace_bytes, n_slots);
}
EK_API(host_suite_tq_hybrid_geo,
       (const void* h_t, const void* h_q, const void* h_sp, const void* h_zs, const void* h_A, const void* h_B, int nlev, int64_t npl,
        void* const* h_outs, uint32_t out_mask, int ept_method, int top_toa, double alpha_top, void* h_thickness, void* h_z, void* h_height,
        int height_mode, void* workspace, size_t workspace_bytes, int n_slots),
       (h_t, h_q, h_sp, h_zs, h_A, h_B, nlev, npl, h_outs, out_mask, ept_method, top_toa, alpha_top, h_thickness, h_z, h_height, height_mode,
        workspace, workspace_bytes, n_slots))
