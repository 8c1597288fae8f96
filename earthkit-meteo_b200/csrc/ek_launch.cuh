// ek_launch.cuh -- host side of a launch: argument checks, grid sizing, error reporting.
#pragma once
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <mutex>

#include "../../include/ek_thermo.h"
#include "ek_thermo_kernels.cuh"

#define EK_EXPORT __attribute__((visibility("default")))

namespace ek {

// defined in ek_api.cu
int set_error(int code, const char* fmt, ...);
int sm_count_current_device();
extern std::atomic<int> g_ctas_per_sm;
extern std::atomic<uint64_t> g_launches;

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Dynamic shared memory of a launch: the lean float64 tables; float32 kernels use none.
template <typename T> constexpr unsigned smem_for() { return sizeof(T) == 8 ? kSmemBytes : 0u; }

// Shared-memory attributes of a kernel instantiation on the current device: a carve-out that holds kMinCtas CTAs' worth of
// `smem_bytes`, so the tables never lower the occupancy the register budget was chosen for (the driver's default carve-out
// heuristic may pick a smaller one), and, above the 48 KiB default, the dynamic shared memory limit of the function.  `Kernel` is
// the address of the __global__ instantiation.  The hybrid kernels' size grows with the level count, so the attributes are set
// again whenever a request exceeds the largest one configured so far on that device; they only ever grow.  Raising them is
// serialised: with two callers raising at once, the smaller setting must not land after the larger one and break its launches.
template <auto Kernel> inline int prepare_smem(unsigned smem_bytes) {
    if (smem_bytes == 0) return EK_OK;
    constexpr int kDevs = 64;
    static std::atomic<unsigned> configured[kDevs];  // per device: the largest smem_bytes the attributes hold
    static std::mutex raising;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0) return EK_OK;  // no current device: the launch reports it
    std::atomic<unsigned>* have = dev < kDevs ? &configured[dev] : nullptr;
    if (have && have->load(std::memory_order_acquire) >= smem_bytes) return EK_OK;
    std::lock_guard<std::mutex> lock(raising);
    if (have && have->load(std::memory_order_acquire) >= smem_bytes) return EK_OK;
    const unsigned want = kMinCtas * (smem_bytes + 1024u);  // + the per-CTA reservation
    int pct = (int)((want * 100u + 228u * 1024u - 1u) / (228u * 1024u));
    if (pct > 100) pct = 100;
    cudaFuncSetAttribute(Kernel, cudaFuncAttributePreferredSharedMemoryCarveout, pct);  // a hint: the launch works without it
    (void)cudaGetLastError();
    if (smem_bytes > 48u * 1024u) {
        const cudaError_t err = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
        if (err != cudaSuccess) {
            (void)cudaGetLastError();
            return set_error((int)err, "cannot allow %u bytes of dynamic shared memory: %s", smem_bytes, cudaGetErrorString(err));
        }
    }
    if (have) {  // max, not store: the value only grows
        unsigned cur = have->load(std::memory_order_relaxed);
        while (cur < smem_bytes && !have->compare_exchange_weak(cur, smem_bytes, std::memory_order_release, std::memory_order_relaxed)) {
        }
    }
    return EK_OK;
}

// prepare_smem + launch of a kernel with the standard CTA size and the dtype's dynamic shared memory; nonzero: not launched
template <auto Kernel, typename... Args> inline int launch_kernel_smem(int blocks, cudaStream_t st, unsigned smem, Args... args) {
    if (int rc = prepare_smem<Kernel>(smem)) return rc;
    Kernel<<<blocks, kThreads, smem, st>>>(args...);
    return EK_OK;
}
template <auto Kernel, typename T, typename... Args> inline int launch_kernel(int blocks, cudaStream_t st, Args... args) {
    return launch_kernel_smem<Kernel>(blocks, st, smem_for<T>(), args...);
}

// Launch of a streaming kernel that orders itself behind its predecessor in the stream with pdl_acquire() (ek_thermo_kernels.cuh):
// the programmatic-serialization attribute lets it be scheduled while the predecessor drains.  ONLY for kernels that call
// pdl_acquire() before their first access to a field -- without it the attribute would remove the stream dependency.
template <auto Kernel, typename... Args>
inline int launch_streaming(unsigned blocks, unsigned smem, cudaStream_t st, Args... args) {
    if (int rc = prepare_smem<Kernel>(smem)) return rc;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(blocks);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaLaunchKernelEx(&cfg, Kernel, args...);
    return EK_OK;
}

// Launch Op over n points.  ins[k].ptr == NULL means broadcast scalar ins[k].value; outs[o] == NULL means
// "output o not wanted" (P.out_mask must agree).
template <class Op, class OpE, typename T>
int launch(const char* what, const ek_operand* ins, void* const* outs, int64_t n, Params P, void* stream) {
    if (n < 0) return set_error(EK_ERR_ARG, "%s: n=%lld must be >= 0", what, (long long)n);
    InArgs<Op::NIN> in;
    OutArgs<Op::NOUT> out;
    int vec_ok = 1;
    for (int k = 0; k < Op::NIN; ++k) {
        in.p[k] = ins[k].ptr;
        in.s[k] = ins[k].value;
        if (ins[k].ptr) {
            if (!aligned16(ins[k].ptr)) vec_ok = 0;
            if (reinterpret_cast<uintptr_t>(ins[k].ptr) % sizeof(T))
                return set_error(EK_ERR_ARG, "%s: input %d is not aligned to its element size", what, k);
        }
    }
    uint32_t mask = 0;
    for (int o = 0; o < Op::NOUT; ++o) {
        out.p[o] = outs[o];
        if (outs[o]) {
            mask |= 1u << o;
            if (!aligned16(outs[o])) vec_ok = 0;
            if (reinterpret_cast<uintptr_t>(outs[o]) % sizeof(T))
                return set_error(EK_ERR_ARG, "%s: output %d is not aligned to its element size", what, o);
        }
    }
    if (mask == 0) return set_error(EK_ERR_ARG, "%s: no output buffer given", what);
    P.out_mask = mask;
    if (n == 0) return EK_OK;

    constexpr int threads = kThreads;
    constexpr int unroll = UnrollOf<Op>::value;
    const int64_t tile = (int64_t)threads * Vec16<T>::N * unroll;
    const int64_t ntiles = n / tile;
    const int64_t tail_blocks = ((n - ntiles * tile) + threads - 1) / threads;
    const int sms = sm_count_current_device();
    if (sms <= 0) return set_error(EK_ERR_ARG, "%s: no CUDA device is current", what);
    int64_t cap = (int64_t)sms * g_ctas_per_sm.load(std::memory_order_relaxed);
    // small fields (a few tiles per resident CTA, e.g. one ERA5 level): exactly one resident wave -- every CTA copies the lean
    // tables once and walks its 2-3 tiles back to back instead of a second, partial wave of CTAs queueing behind the first
    // (theta + rh on 1 M points, graph replay: 14.4 -> 12.3 us; profiles/r02_kbench_era5_ctas.log)
    const int64_t wave = (int64_t)sms * MinCtasOf<Op>::value;
    if (ntiles <= 8 * wave && wave < cap) cap = wave;
    int64_t blocks = ntiles > tail_blocks ? ntiles : tail_blocks;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;

    if (int rc = launch_streaming<&ew_kernel<Op, OpE, T, unroll>>((unsigned)blocks, smem_for<T>(), static_cast<cudaStream_t>(stream), in, out, n, P, vec_ok))
        return rc;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return set_error((int)err, "%s: kernel launch failed: %s", what, cudaGetErrorString(err));
    return EK_OK;
}

// Op over n_seg separate fields of n_per_seg points each in one launch (ew_batch_kernel).  ins[k]: host array of n_seg device
// pointers, or NULL for the broadcast scalar scalars[k]; outs[o]: host array of n_seg device pointers, or NULL when output o
// is not wanted.  last_scalars: NULL, or n_seg numbers -- the LAST input as one broadcast scalar per segment (then ins[NIN-1] must
// be NULL).  More than kBatchMaxSeg segments take one launch per kBatchMaxSeg.
template <class Op, class OpE, typename T>
int launch_batch(const char* what, int n_seg, const void* const* const* ins, const double* scalars, const double* last_scalars,
                 void* const* const* outs, int64_t n_per_seg, Params P, void* stream) {
    if (n_seg < 0 || n_per_seg < 0) return set_error(EK_ERR_ARG, "%s: n_seg=%d n_per_seg=%lld", what, n_seg, (long long)n_per_seg);
    uint32_t in_mask = 0, out_mask = 0;
    for (int k = 0; k < Op::NIN; ++k)
        if (ins[k]) in_mask |= 1u << k;
    for (int o = 0; o < Op::NOUT; ++o)
        if (outs[o]) out_mask |= 1u << o;
    if (out_mask == 0) return set_error(EK_ERR_ARG, "%s: no output buffer given", what);
    if (last_scalars && ins[Op::NIN - 1]) return set_error(EK_ERR_ARG, "%s: the last input is given both as fields and as per-segment scalars", what);
    P.out_mask = out_mask;
    if (n_seg == 0 || n_per_seg == 0) return EK_OK;
    const int sms = sm_count_current_device();
    if (sms <= 0) return set_error(EK_ERR_ARG, "%s: no CUDA device is current", what);
    constexpr int unroll = UnrollOf<Op>::value;
    const int64_t tile = (int64_t)kThreads * Vec16<T>::N * unroll;
    for (int s0 = 0; s0 < n_seg; s0 += kBatchMaxSeg) {
        BatchArgs<Op::NIN, Op::NOUT> B;
        B.n_seg = n_seg - s0 < kBatchMaxSeg ? n_seg - s0 : kBatchMaxSeg;
        B.in_mask = in_mask;
        B.out_mask = out_mask;
        B.last_per_seg = last_scalars ? 1 : 0;
        for (int j = 0; j < B.n_seg; ++j) B.s_last[j] = last_scalars ? last_scalars[s0 + j] : 0.0;
        int vec_ok = 1;  // tiles start at multiples of the vector length inside every segment: only the segment pointers must be 16-byte aligned
        for (int k = 0; k < Op::NIN; ++k) {
            B.s[k] = scalars ? scalars[k] : 0.0;
            for (int j = 0; j < B.n_seg; ++j) {
                B.in[k][j] = ins[k] ? ins[k][s0 + j] : nullptr;
                if (ins[k]) {
                    if (!B.in[k][j] || reinterpret_cast<uintptr_t>(B.in[k][j]) % sizeof(T))
                        return set_error(EK_ERR_ARG, "%s: input %d of segment %d is NULL or not aligned to its element size", what, k, s0 + j);
                    if (!aligned16(B.in[k][j])) vec_ok = 0;
                }
            }
        }
        for (int o = 0; o < Op::NOUT; ++o)
            for (int j = 0; j < B.n_seg; ++j) {
                B.out[o][j] = outs[o] ? outs[o][s0 + j] : nullptr;
                if (outs[o]) {
                    if (!B.out[o][j] || reinterpret_cast<uintptr_t>(B.out[o][j]) % sizeof(T))
                        return set_error(EK_ERR_ARG, "%s: output %d of segment %d is NULL or not aligned to its element size", what, o, s0 + j);
                    if (!aligned16(B.out[o][j])) vec_ok = 0;
                }
            }
        const int64_t ntiles = (n_per_seg / tile) * B.n_seg;
        const int64_t tail_blocks = ((n_per_seg % tile) * B.n_seg + kThreads - 1) / kThreads;
        int64_t cap = (int64_t)sms * g_ctas_per_sm.load(std::memory_order_relaxed);
        const int64_t wave = (int64_t)sms * MinCtasOf<Op>::value;
        if (ntiles <= 8 * wave && wave < cap) cap = wave;
        int64_t blocks = ntiles > tail_blocks ? ntiles : tail_blocks;
        if (blocks > cap) blocks = cap;
        if (blocks < 1) blocks = 1;
        if (int rc = launch_streaming<&ew_batch_kernel<Op, OpE, T, unroll>>((unsigned)blocks, smem_for<T>(), static_cast<cudaStream_t>(stream), B, n_per_seg, P,
                                                                            vec_ok))
            return rc;
        g_launches.fetch_add(1, std::memory_order_relaxed);
        cudaError_t err = cudaGetLastError();
        if (err != cudaSuccess) return set_error((int)err, "%s: kernel launch failed: %s", what, cudaGetErrorString(err));
    }
    return EK_OK;
}

inline bool valid_phase(int v) { return v >= 0 && v <= 2; }

// defines ek_thermo_<NAME>_f64 / _f32 forwarding to the template function impl_<NAME><T>
#define EK_API(NAME, PARAMS, ARGS)                                                    \
    extern "C" EK_EXPORT int ek_thermo_##NAME##_f64 PARAMS { return impl_##NAME<double> ARGS; } \
    extern "C" EK_EXPORT int ek_thermo_##NAME##_f32 PARAMS { return impl_##NAME<float> ARGS; }

}  // namespace ek
