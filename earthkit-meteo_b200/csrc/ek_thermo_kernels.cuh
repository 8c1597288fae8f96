// ek_thermo_kernels.cuh -- the one streaming kernel template behind every entry point.
//
// The path is elementwise with no reuse, so the design is the HBM-streaming one (SURVEY.md §8(d)):
//   * 128-bit coalesced loads/stores (double2 / float4) with streaming cache hints (ld.global.cs /
//     st.global.cs: the data is touched once, keep it out of the way in L1/L2);
//   * each thread front-loads kUnroll vectors per input before any math so that enough bytes are in
//     flight per SM to cover HBM latency (needs ~35 KB/SM in flight at 6.5 TB/s);
//   * all intermediates of a point live in registers; outputs are stored as soon as a vector is done;
//   * tiles are handed to CTAs round-robin (grid-stride), grid sized as SMs x CTAs-per-SM;
//   * no shared-memory staging, no TMA, no tensor cores: there is nothing to stage or contract (shared memory only
//     holds the log/exp tables of the lean math, ek_thermo_lean.cuh);
//   * every point goes through the fast (lean-math) functor; a point whose result contains a NaN is recomputed by
//     the exact functor in an out-of-line cold path, so special values behave exactly as the reference.
// Broadcast scalars arrive by value (never materialised); unaligned views use scalar ld/st inside the
// same kernel (uniform branch), and the sub-tile tail is a scalar grid-stride loop.
#pragma once
#include <cuda_runtime.h>

#include "ek_thermo_math.cuh"

namespace ek {

template <int N> struct InArgs {
    const void* p[N];
    double s[N];
};
template <int N> struct OutArgs {
    void* p[N];
};

template <typename T> struct Vec16;
template <> struct Vec16<double> {
    using type = double2;
    static constexpr int N = 2;
    static __device__ __forceinline__ void load(const double* src, double* dst) {
        double2 v = __ldcs(reinterpret_cast<const double2*>(src));
        dst[0] = v.x;
        dst[1] = v.y;
    }
    static __device__ __forceinline__ void store(double* dst, const double* src) {
        __stcs(reinterpret_cast<double2*>(dst), make_double2(src[0], src[1]));
    }
};
template <> struct Vec16<float> {
    using type = float4;
    static constexpr int N = 4;
    static __device__ __forceinline__ void load(const float* src, float* dst) {
        float4 v = __ldcs(reinterpret_cast<const float4*>(src));
        dst[0] = v.x;
        dst[1] = v.y;
        dst[2] = v.z;
        dst[3] = v.w;
    }
    static __device__ __forceinline__ void store(float* dst, const float* src) {
        __stcs(reinterpret_cast<float4*>(dst), make_float4(src[0], src[1], src[2], src[3]));
    }
};

// dynamic shared memory a launch must provide (the lean fp64 log/exp tables)
#if EK_LEAN_MATH
constexpr unsigned kSmemBytes = 2 * 8 * EK_LOG_TAB_N + 8 * EK_EXP_TAB_N;  // lean::Tables (checked against sizeof in the kernel)
#else
constexpr unsigned kSmemBytes = 0;
#endif

constexpr int kThreads = 256;  // CTA size is a compile-time constant: tile offsets become immediates
constexpr int kUnroll = 2;     // 16-byte vectors per input per thread per tile (1 vector: suite +1 %, theta -13 %)
constexpr int kPfDist = 2;     // tiles ahead of the current one that prefetch_tile_l2 asks L2 for (functors with PREFETCH_NEXT);
                               // 1 or 3 tiles ahead: suite 0.92 -> 0.89
constexpr int kMinCtas = 4;    // <= 64 registers per thread: 4 CTAs = 32 warps per SM hide the fp64 dependency chains
// Resident CTAs per SM for the functors that declare HEAVY (the fused suites, ept / ept + wet bulb): 80 registers instead of 64 --
// no spills in their ~200-instruction bodies -- and, with the L2 prefetch two tiles ahead covering what the fourth CTA's loads
// covered, 3-6 % more of the roofline (profiles/r02_ab_ew.log: suite 0.886 -> 0.923, ept + wet bulb 0.80 -> 0.86, single pass
// 0.76 -> 0.84); the short single-output kernels lose 7-10 % with it (theta 0.974 -> 0.871) and keep kMinCtas.
constexpr int kHeavyMinCtas = 3;

template <typename T> __device__ __forceinline__ bool is_nan_val(T v) { return v != v; }

// Cold path of a lean build: a result of the fast functor contains a NaN.  Out of line on purpose (its registers and
// code stay out of the hot loop).  Missing-value points -- every ARRAY input NaN (`array_mask` bit k = input k is an
// array, not a broadcast scalar) -- keep the fast result: every output depends on an array input, so IEEE propagation
// makes the exact result NaN as well (masked fields, e.g. below-ground points, therefore stay on the fast path).
// Any other point is recomputed with the exact functor (libdevice math, IEEE division).
template <class OpE, typename T> __device__ __noinline__ void cold_point(const T* a, T* r, const Params P, const uint32_t array_mask) {
    bool missing = array_mask != 0;
#pragma unroll
    for (int k = 0; k < OpE::NIN; ++k)
        if ((array_mask >> k) & 1u) missing = missing && is_nan_val(a[k]);
    if (missing) return;
#pragma unroll
    for (int o = 0; o < OpE::NOUT; ++o) r[o] = T(0);
    OpE::template apply<T>(a, r, P);
}

// True when a result of the fast functor may come from outside the lean primitives' domain (they answer NaN
// there): the high word of a double NaN is >= 0x7ff80000 once the sign is cleared.
template <int NOUT> __device__ __forceinline__ bool any_nan(const double* r) {
    int m = 0;
#pragma unroll
    for (int o = 0; o < NOUT; ++o) m = max(m, __double2hiint(r[o]) & 0x7fffffff);
    return m >= 0x7ff80000;
}
template <int NOUT> __device__ __forceinline__ bool any_nan(const float* r) {
    int m = 0;
#pragma unroll
    for (int o = 0; o < NOUT; ++o) m = max(m, __float_as_int(r[o]) & 0x7fffffff);
    return m > 0x7f800000;
}

// float32 lean math is self-contained (its primitives follow IEEE special values), so float32 points skip the cold
// path -- except for functors that declare `COLD_F32 = true`: the tabulated bisection poisons ties, underflow and
// non-positive inputs with NaN in float32 as well.
template <class Op, class = void> struct ColdF32 {
    static constexpr bool value = false;
};
template <class Op> struct ColdF32<Op, decltype((void)Op::COLD_F32)> {
    static constexpr bool value = Op::COLD_F32;
};

// One grid point: fast functor, then (lean build; float64, or float32 where the functor asks) the cold path if the
// result has a NaN in it.
template <class Op, class OpE, typename T>
__device__ __forceinline__ void point(const T* a, T* r, const Params& P, const uint32_t array_mask) {
#pragma unroll
    for (int o = 0; o < Op::NOUT; ++o) r[o] = T(0);
    Op::template apply<T>(a, r, P);
#if EK_LEAN_DEVICE
    if ((sizeof(T) == 8 || ColdF32<Op>::value) && __builtin_expect(any_nan<Op::NOUT>(r), 0)) {
        T a2[Op::NIN], r2[Op::NOUT];
#pragma unroll
        for (int k = 0; k < Op::NIN; ++k) a2[k] = a[k];
#pragma unroll
        for (int o = 0; o < Op::NOUT; ++o) r2[o] = r[o];
        cold_point<OpE, T>(a2, r2, P, array_mask);
#pragma unroll
        for (int o = 0; o < Op::NOUT; ++o) r[o] = r2[o];
    }
#else
    (void)array_mask;
#endif
}

// Functors that declare `BATCH = true` provide apply_n(): the N points of one 16-byte vector evaluated together (the
// bisection advances them side by side).  Same per-point results and the same NaN -> cold-path rule as point().
template <class Op, class = void> struct IsBatch {
    static constexpr bool value = false;
};
template <class Op> struct IsBatch<Op, decltype((void)Op::BATCH)> {
    static constexpr bool value = Op::BATCH;
};

template <class Op, class OpE, typename T, int N>
__device__ __forceinline__ void points_n(const T (&a)[N][Op::NIN], T (&r)[N][Op::NOUT], const Params& P, const uint32_t array_mask) {
#pragma unroll
    for (int j = 0; j < N; ++j)
#pragma unroll
        for (int o = 0; o < Op::NOUT; ++o) r[j][o] = T(0);
    Op::template apply_n<T, N>(a, r, P);
#if EK_LEAN_DEVICE
    if (sizeof(T) == 8 || ColdF32<Op>::value) {
#pragma unroll
        for (int j = 0; j < N; ++j) {
            if (__builtin_expect(any_nan<Op::NOUT>(r[j]), 0)) {
                T a2[Op::NIN], r2[Op::NOUT];
#pragma unroll
                for (int k = 0; k < Op::NIN; ++k) a2[k] = a[j][k];
#pragma unroll
                for (int o = 0; o < Op::NOUT; ++o) r2[o] = r[j][o];
                cold_point<OpE, T>(a2, r2, P, array_mask);
#pragma unroll
                for (int o = 0; o < Op::NOUT; ++o) r[j][o] = r2[o];
            }
        }
    }
#else
    (void)array_mask;
#endif
}

// 16-byte vectors per input per thread per tile: kUnroll unless the functor declares `UNROLL` (the one-step Newton solve keeps
// one vector in flight: its ~550-instruction body needs the registers, and without spills it runs 8-12 % faster).
template <class Op, class = void> struct UnrollOf {
    static constexpr int value = kUnroll;
};
template <class Op> struct UnrollOf<Op, decltype((void)Op::UNROLL)> {
    static constexpr int value = Op::UNROLL > 0 ? Op::UNROLL : kUnroll;
};

// The "last input is a scalar" tile loop (load_tile ALLARR == 2) unless the functor opts out with LAST_SCALAR_LOOP = false
template <class Op, class = void> struct LastScalarLoopOf {
    static constexpr bool value = true;
};
template <class Op> struct LastScalarLoopOf<Op, decltype((void)Op::LAST_SCALAR_LOOP)> {
    static constexpr bool value = Op::LAST_SCALAR_LOOP;
};

template <class Op, class = void> struct DeferColdOf {
    static constexpr bool value = false;
};
template <class Op> struct DeferColdOf<Op, decltype((void)Op::DEFER_COLD)> {
    static constexpr bool value = Op::DEFER_COLD;
};

// Resident CTAs per SM a functor's register budget is sized for: kMinCtas, or kHeavyMinCtas where the functor says HEAVY.
template <class Op, class = void> struct MinCtasOf {
    static constexpr int value = kMinCtas;
};
template <class Op> struct MinCtasOf<Op, decltype((void)Op::HEAVY)> {
    static constexpr int value = Op::HEAVY ? kHeavyMinCtas : kMinCtas;
};

// The inputs of one tile, per thread: UNROLL 16-byte vectors of every input array, in registers.
template <class Op, typename T, int UNROLL> struct TileRegs {
    T x[Op::NIN][UNROLL][Vec16<T>::N];
};

// ALLARR (the shape of the call, fixed at compile time so the loop carries no predicated loads and no broadcast moves):
//   1  every input is an array (the whole-field call; measured in the SASS of the ept kernel: 6 of 160 instructions per
//      point were those moves);
//   2  every input but the LAST is an array and the last is a broadcast scalar -- pressure-level data (t, q arrays; p one
//      number): the scalar is a loop invariant the compiler can see, so everything that depends on p alone (ln(p0/p), the Exner
//      factor) is computed once per thread instead of once per point;
//   0  anything else (run-time mask).
template <class Op, typename T, int UNROLL, bool VECOK, int ALLARR>
__device__ __forceinline__ void load_tile(TileRegs<Op, T, UNROLL>& r, const InArgs<Op::NIN>& in, const int64_t base) {
    constexpr int VEC = Vec16<T>::N;
    constexpr int VSTRIDE = kThreads * VEC;  // elements between a thread's successive vectors
#pragma unroll
    for (int k = 0; k < Op::NIN; ++k) {
        const bool is_array = ALLARR == 1 ? true : (ALLARR == 2 ? k < Op::NIN - 1 : in.p[k] != nullptr);
        if (is_array) {
            const T* src = static_cast<const T*>(in.p[k]) + base;
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) {
                if (VECOK) {
                    Vec16<T>::load(src + u * VSTRIDE, r.x[k][u]);
                } else {
#pragma unroll
                    for (int v = 0; v < VEC; ++v) r.x[k][u][v] = __ldcs(src + u * VSTRIDE + v);
                }
            }
        } else {
            const T s = static_cast<T>(in.s[k]);
#pragma unroll
            for (int u = 0; u < UNROLL; ++u)
#pragma unroll
                for (int v = 0; v < VEC; ++v) r.x[k][u][v] = s;
        }
    }
}

// Ask L2 to fetch the lines a thread will load for the CTA's NEXT tile (no registers involved): keeps HBM requests in
// flight while the warp is in the math / store phase of the current tile.  Per-functor switch (Op::PREFETCH_NEXT):
// measured on B200, it lifts the multi-output suites, whose math phase per tile is long (O1280 x 137 fp64 suite
// 0.845 -> 0.886 of the HBM roofline, ENS conversions 0.876 -> 0.885), and costs the short single-output kernels
// 1.5-5 % (theta 0.963 -> 0.930, ept+wbpt 0.770 -> 0.727), so only the (t, q, p) suite turns it on.  ncu, one launch of
// the contract workload: 10.28 -> 9.69 ms, long-scoreboard stalls per issue 8.3 -> 4.6, DRAM traffic +0.3 %.
template <class Op, typename T, int UNROLL>
__device__ __forceinline__ void prefetch_tile_l2(const InArgs<Op::NIN>& in, const int64_t base) {
    constexpr int VSTRIDE = kThreads * Vec16<T>::N;
#pragma unroll
    for (int k = 0; k < Op::NIN; ++k) {
        if (in.p[k] != nullptr) {
            const T* src = static_cast<const T*>(in.p[k]) + base;
#pragma unroll
            for (int u = 0; u < UNROLL; ++u) asm volatile("prefetch.global.L2 [%0];" ::"l"(src + u * VSTRIDE));
        }
    }
}

template <class Op, class OpE, typename T, int UNROLL, bool VECOK>
__device__ __forceinline__ void compute_store_tile(const TileRegs<Op, T, UNROLL>& r, const OutArgs<Op::NOUT>& out, const int64_t base,
                                                   const Params& P, const uint32_t array_mask) {
    constexpr int NIN = Op::NIN;
    constexpr int NOUT = Op::NOUT;
    constexpr int VEC = Vec16<T>::N;
    constexpr int VSTRIDE = kThreads * VEC;
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
        T y[NOUT][VEC];
        if constexpr (IsBatch<Op>::value) {
            T a[VEC][NIN], res[VEC][NOUT];
#pragma unroll
            for (int v = 0; v < VEC; ++v)
#pragma unroll
                for (int k = 0; k < NIN; ++k) a[v][k] = r.x[k][u][v];
            points_n<Op, OpE, T, VEC>(a, res, P, array_mask);
#pragma unroll
            for (int v = 0; v < VEC; ++v)
#pragma unroll
                for (int o = 0; o < NOUT; ++o) y[o][v] = res[v][o];
        } else if constexpr (DeferColdOf<Op>::value && EK_LEAN_DEVICE) {
            // Functors that declare DEFER_COLD: the VEC points of a vector go through the fast functor back to back and are
            // checked for NaN afterwards -- one basic block, so the scheduler interleaves their dependency chains (these fp64
            // kernels wait on fixed-latency results: ept 0.83 -> 0.93, ept + wet bulb 0.87 -> 0.89, es 0.63 -> 0.66 of the
            // roofline, profiles/r02_ab_ew3.log).  The multi-output suites lose 2-5 % with it (registers) and keep point().
            T res[VEC][NOUT];
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                T a[NIN];
#pragma unroll
                for (int k = 0; k < NIN; ++k) a[k] = r.x[k][u][v];
#pragma unroll
                for (int o = 0; o < NOUT; ++o) res[v][o] = T(0);
                Op::template apply<T>(a, res[v], P);
            }
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                if ((sizeof(T) == 8 || ColdF32<Op>::value) && __builtin_expect(any_nan<NOUT>(res[v]), 0)) {
                    T a2[NIN], r2[NOUT];
#pragma unroll
                    for (int k = 0; k < NIN; ++k) a2[k] = r.x[k][u][v];
#pragma unroll
                    for (int o = 0; o < NOUT; ++o) r2[o] = res[v][o];
                    cold_point<OpE, T>(a2, r2, P, array_mask);
#pragma unroll
                    for (int o = 0; o < NOUT; ++o) res[v][o] = r2[o];
                }
#pragma unroll
                for (int o = 0; o < NOUT; ++o) y[o][v] = res[v][o];
            }
        } else {
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                T a[NIN], res[NOUT];
#pragma unroll
                for (int k = 0; k < NIN; ++k) a[k] = r.x[k][u][v];
                point<Op, OpE, T>(a, res, P, array_mask);
#pragma unroll
                for (int o = 0; o < NOUT; ++o) y[o][v] = res[o];
            }
        }
#pragma unroll
        for (int o = 0; o < NOUT; ++o) {
            const bool w = Op::STATIC_MASK ? (((Op::STATIC_MASK >> o) & 1u) != 0) : (out.p[o] != nullptr);
            if (w) {
                T* dst = static_cast<T*>(out.p[o]) + base + u * VSTRIDE;
                if (VECOK) {
                    Vec16<T>::store(dst, y[o]);
                } else {
#pragma unroll
                    for (int v = 0; v < VEC; ++v) __stcs(dst + v, y[o][v]);
                }
            }
        }
    }
}

// Tiles are handed to CTAs round-robin; a tile's loads are all issued before its math.  Loading the NEXT tile into a second
// register set before computing the current one measured no gain on B200 (profiles/r01_kbench_pipeline_unroll_variants.log):
// 32 resident warps/SM with 2 front-loaded vectors per input already cover the HBM latency.
template <class Op, class OpE, typename T, int UNROLL, bool VECOK, int ALLARR>
__device__ __forceinline__ void tile_loop(const InArgs<Op::NIN>& in, const OutArgs<Op::NOUT>& out, const int64_t ntiles, const Params& P,
                                          const uint32_t array_mask) {
    constexpr int TILE = kThreads * Vec16<T>::N * UNROLL;
    const int64_t G = gridDim.x;
    const int64_t toff = (int64_t)threadIdx.x * Vec16<T>::N;
    int64_t ta = blockIdx.x;
    if (ta >= ntiles) return;
    for (; ta < ntiles; ta += G) {
        TileRegs<Op, T, UNROLL> A;
        load_tile<Op, T, UNROLL, VECOK, ALLARR>(A, in, ta * TILE + toff);
        if (Op::PREFETCH_NEXT && ta + kPfDist * G < ntiles) prefetch_tile_l2<Op, T, UNROLL>(in, (ta + kPfDist * G) * TILE + toff);
        compute_store_tile<Op, OpE, T, UNROLL, VECOK>(A, out, ta * TILE + toff, P, array_mask);
    }
}

// Programmatic dependent launch (sm_90+): a streaming kernel lets its successor in the stream start (launch latency, CTA
// scheduling, the copy of the lean tables) while its own last CTAs drain.  One launch per 1 M-point level, theta + rh: eager
// 13.3 -> 11.3 us, graph replay 11.8 -> 11.0 us (profiles/r02f_kbench_levels.log).
// pdl_release: the next kernel of the stream may be scheduled as soon as every CTA of this grid has started; pdl_acquire: wait
// until the previous kernel of the stream has completed and its writes are visible.  Everything that reads or writes a field
// comes after pdl_acquire; only the table copy (immutable data) runs before it.  Both are no-ops for a kernel launched without
// the programmatic-serialization attribute.
__device__ __forceinline__ void pdl_release() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void pdl_acquire() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <class Op, class OpE, typename T, int UNROLL>
__global__ void __launch_bounds__(kThreads, MinCtasOf<Op>::value)
    ew_kernel(const InArgs<Op::NIN> in, const OutArgs<Op::NOUT> out, const int64_t n, const Params P, const int vec_ok) {
    constexpr int NIN = Op::NIN;
    constexpr int NOUT = Op::NOUT;
    constexpr int TILE = kThreads * Vec16<T>::N * UNROLL;
    pdl_release();
#if EK_LEAN_DEVICE
    static_assert(sizeof(lean::Tables) == kSmemBytes, "kSmemBytes must match lean::Tables");
    if (sizeof(T) == 8) lean::init_tables();
#endif
    pdl_acquire();
    const int64_t ntiles = n / TILE;
    uint32_t array_mask = 0;
#pragma unroll
    for (int k = 0; k < NIN; ++k) array_mask |= (in.p[k] != nullptr) ? (1u << k) : 0u;
    if (vec_ok && array_mask == (1u << NIN) - 1u)
        tile_loop<Op, OpE, T, UNROLL, true, 1>(in, out, ntiles, P, array_mask);
    else if (LastScalarLoopOf<Op>::value && NIN >= 2 && vec_ok && array_mask == (1u << (NIN - 1)) - 1u)
        tile_loop<Op, OpE, T, UNROLL, true, 2>(in, out, ntiles, P, array_mask);
    else if (vec_ok)
        tile_loop<Op, OpE, T, UNROLL, true, 0>(in, out, ntiles, P, array_mask);
    else
        tile_loop<Op, OpE, T, UNROLL, false, 0>(in, out, ntiles, P, array_mask);

    // tail: fewer than one tile of points, one point per thread, grid-stride
    for (int64_t i = ntiles * TILE + (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kThreads) {
        T a[NIN], r[NOUT];
#pragma unroll
        for (int k = 0; k < NIN; ++k) a[k] = (in.p[k] != nullptr) ? __ldcs(static_cast<const T*>(in.p[k]) + i) : static_cast<T>(in.s[k]);
        point<Op, OpE, T>(a, r, P, array_mask);
#pragma unroll
        for (int o = 0; o < NOUT; ++o) {
            const bool w = Op::STATIC_MASK ? (((Op::STATIC_MASK >> o) & 1u) != 0) : (out.p[o] != nullptr);
            if (w) __stcs(static_cast<T*>(out.p[o]) + i, r[o]);
        }
    }
}

// ---- batched launch: the same functor over n_seg separate fields of n_per_seg points each, ONE launch ------------------
// For callers that hold a model field level by level (one allocation per level, e.g. the fields of a GRIB message list):
// a launch per 1 M-point level is bound by launch + table-copy + pipeline-fill latency (12-16 us for 6 us of HBM time), a
// single launch over all levels is not.  The per-segment pointers travel in the kernel parameters (constant bank, indexed
// with the warp-uniform segment number).  Every point goes through point(): results are the bits of the per-field launch.
constexpr int kBatchMaxSeg = 128;
template <int NIN, int NOUT> struct BatchArgs {
    const void* in[NIN][kBatchMaxSeg];
    void* out[NOUT][kBatchMaxSeg];
    double s[NIN];       // broadcast scalar of input k when in[k][0] == NULL (the same for every segment)
    double s_last[kBatchMaxSeg];  // last_per_seg: the LAST input as one number per segment (pressure-level data: t, q fields; p per level)
    int last_per_seg;
    uint32_t in_mask;    // bit k: input k is an array
    uint32_t out_mask;   // bit o: output o is written
    int n_seg;
};

template <class Op, class OpE, typename T, int UNROLL>
__global__ void __launch_bounds__(kThreads, MinCtasOf<Op>::value)
    ew_batch_kernel(const __grid_constant__ BatchArgs<Op::NIN, Op::NOUT> B, const int64_t n_per_seg, const Params P, const int vec_ok) {
    constexpr int NIN = Op::NIN;
    constexpr int NOUT = Op::NOUT;
    constexpr int TILE = kThreads * Vec16<T>::N * UNROLL;
    pdl_release();
#if EK_LEAN_DEVICE
    if (sizeof(T) == 8) lean::init_tables();
#endif
    pdl_acquire();
    const int64_t tiles_per_seg = n_per_seg / TILE;
    const int64_t ntiles = tiles_per_seg * B.n_seg;
    const int64_t toff = (int64_t)threadIdx.x * Vec16<T>::N;
    const bool all_arrays = B.in_mask == (1u << NIN) - 1u;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int seg = (int)(tile / tiles_per_seg);
        const int64_t base = (tile - (int64_t)seg * tiles_per_seg) * TILE + toff;
        InArgs<NIN> in;
        OutArgs<NOUT> out;
#pragma unroll
        for (int k = 0; k < NIN; ++k) {
            in.p[k] = ((B.in_mask >> k) & 1u) ? B.in[k][seg] : nullptr;
            in.s[k] = (k == NIN - 1 && B.last_per_seg) ? B.s_last[seg] : B.s[k];
        }
#pragma unroll
        for (int o = 0; o < NOUT; ++o) out.p[o] = ((B.out_mask >> o) & 1u) ? B.out[o][seg] : nullptr;
        auto prefetch_next = [&]() {
            if (Op::PREFETCH_NEXT) {  // the CTA's tile kPfDist rounds ahead, possibly in a later segment
                const int64_t nt = tile + kPfDist * (int64_t)gridDim.x;
                if (nt < ntiles) {
                    const int nseg = (int)(nt / tiles_per_seg);
                    InArgs<NIN> nin;
    #pragma unroll
                    for (int k = 0; k < NIN; ++k) nin.p[k] = ((B.in_mask >> k) & 1u) ? B.in[k][nseg] : nullptr;
                    prefetch_tile_l2<Op, T, UNROLL>(nin, (nt - (int64_t)nseg * tiles_per_seg) * TILE + toff);
                }
            }
        };
        TileRegs<Op, T, UNROLL> A;
        if constexpr (LastScalarLoopOf<Op>::value && NIN >= 2) {
            // pressure-level data (every input a field, the last one a number per segment): its own copy of the tile body, in which the
            // compiler sees that the points of a tile share the scalar and computes what depends on it alone once per tile
            if (vec_ok && B.in_mask == (1u << (NIN - 1)) - 1u) {
                load_tile<Op, T, UNROLL, true, 2>(A, in, base);
                prefetch_next();
                compute_store_tile<Op, OpE, T, UNROLL, true>(A, out, base, P, B.in_mask);
                continue;
            }
        }
        if (vec_ok && all_arrays)
            load_tile<Op, T, UNROLL, true, 1>(A, in, base);
        else if (vec_ok)
            load_tile<Op, T, UNROLL, true, 0>(A, in, base);
        else
            load_tile<Op, T, UNROLL, false, 0>(A, in, base);
        prefetch_next();
        if (vec_ok)
            compute_store_tile<Op, OpE, T, UNROLL, true>(A, out, base, P, B.in_mask);
        else
            compute_store_tile<Op, OpE, T, UNROLL, false>(A, out, base, P, B.in_mask);
    }
    // tails: fewer than one tile of points per segment, one point per thread
    const int64_t tail = n_per_seg - tiles_per_seg * TILE;
    const int64_t tail_total = tail * B.n_seg;
    for (int64_t j = (int64_t)blockIdx.x * kThreads + threadIdx.x; j < tail_total; j += (int64_t)gridDim.x * kThreads) {
        const int seg = (int)(j / tail);
        const int64_t i = tiles_per_seg * TILE + (j - (int64_t)seg * tail);
        T a[NIN], r[NOUT];
#pragma unroll
        for (int k = 0; k < NIN; ++k)
            a[k] = ((B.in_mask >> k) & 1u) ? __ldcs(static_cast<const T*>(B.in[k][seg]) + i)
                                           : static_cast<T>((k == NIN - 1 && B.last_per_seg) ? B.s_last[seg] : B.s[k]);
        point<Op, OpE, T>(a, r, P, B.in_mask);
#pragma unroll
        for (int o = 0; o < NOUT; ++o)
            if ((B.out_mask >> o) & 1u) __stcs(static_cast<T*>(B.out[o][seg]) + i, r[o]);
    }
}

}  // namespace ek
