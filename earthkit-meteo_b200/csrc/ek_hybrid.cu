// ek_hybrid.cu -- hybrid (IFS model) level pressure, stand-alone and fused into the (t, q) thermo suite.
//
// SURVEY.md 8(f)-1: `pressure_on_hybrid_levels` (reference vertical/array/vertical.py:505-737, "V") is the step
// right before the thermo path on model levels: it expands surface pressure sp[point] and the A/B half-level
// coefficients into the [level, point] pressure field the thermo kernels read.  Two kernels:
//
//   hybrid_pressure_kernel   any of {full, half, delta, alpha} for a list of levels: sp is read once per point
//                            tile and every requested row is written from registers (write-bound streaming).
//   suite_hybrid_kernel      the fused (t, q, p) suite with p computed in registers from sp and A/B: the
//                            [level, point] pressure array is never materialised or read (64 -> 56 B/pt).
//
// Work item = (tile of 256 x VEC points, chunk of levels); items are handed to CTAs round-robin.  A/B are read
// through the read-only path with a warp-uniform address (broadcast).  Same lean-math + exact-recompute scheme
// as ek_thermo_kernels.cuh.
#include "ek_launch.cuh"

using namespace ek;

#if EK_LEAN_MATH
#define EK_FAST_NS fastm
#else
#define EK_FAST_NS exactm
#endif

// The level loops of the hybrid suite and the column (geopotential) kernel issue the loads of several levels before any math
// and ask L2 for a later group of levels while the current one is computed.  ncu on the round-1 hybrid suite, without the L2
// prefetch: 7.4 warps per issue slot waiting on global loads, DRAM at 79 % -- the level loop kept too few bytes in flight.
// Measured on B200, O1280 x 137 fp64 (profiles/r02_ab_hybrid.log, r02_ab_hybrid2.log, r02_ab_hybrid3.log):
//   hybrid suite: 3 levels in flight at 2 CTAs per SM (128 registers) 0.87 of the roofline, stable; 3 levels at 3 CTAs spill
//     (0.72), 4 levels at 2 CTAs 0.84, 2 levels at 3 CTAs 0.80-0.88;
//   column kernel: 2 levels in flight 4.46 ms, 4 -> 5.40 ms, 6 -> 7.68 ms (at the 64-register cap: beyond 2 it spills); 3 CTAs (80
//     registers, no spills of the column state) beat 4 (64) for the thickness / geopotential forms (0.885 -> 0.926), the
//     geometric-height forms keep 4 (0.877 vs 0.825 with 3);
//   prefetch distance: 2 groups of levels ahead 0.86 vs 0.83 (hybrid suite), geometric height 0.91 vs 0.88.
constexpr int kHybLevels = 3;       // hybrid suite: levels whose t/q loads are in flight per thread
constexpr int kHybMinCtas = 2;      // hybrid suite: resident CTAs per SM its register budget is sized for
constexpr int kHybPfDist = 2;       // hybrid suite: groups of kHybLevels levels the L2 prefetch runs ahead
constexpr int kColLevels = 2;       // column kernel, computed alpha/delta: levels in flight per thread (see CLU)
constexpr int kColMinCtas = 3;      // column kernel: resident CTAs per SM
constexpr int kColMinCtasGeom = 4;  // column kernel, geometric-height forms: resident CTAs per SM
constexpr int kColPfDist = 2;       // column kernel: groups of levels the L2 prefetch runs ahead
// suite + geopotential walk, measured on B200 at 1000 W, O1280 x 137 fp64, 5 outputs + z, fused time / the two launches it replaces
// in the same process (profiles/r03_kbench_geo_sweep_f64.log): 2 levels in flight 0.95 (other runs 0.92-0.94), 1 level 0.92, 3 levels
// 1.01; 3 CTAs per SM (80 registers) 1.09; prefetch 1 or 3 groups ahead 0.93 / 0.95.  1 and 2 levels and the prefetch distances are
// inside the run-to-run spread; 2 levels at 2 CTAs (128 registers) and 2 groups ahead, the column kernel's values, are kept.  With
// them (profiles/r03_kbench_geo_f64.log, r03_kbench_geo_f32.log): fp64 11.60 ms = 0.75 of the 64 B/pt roofline, fp32 4.96 ms = 0.88.
constexpr int kGeoLevels = 2;       // suite + geopotential walk: levels whose t/q loads are in flight per thread
constexpr int kGeoMinCtas = 2;      // suite + geopotential walk: resident CTAs per SM
constexpr int kGeoPfDist = 2;       // suite + geopotential walk: groups of levels the L2 prefetch runs ahead

namespace {

template <typename T> __device__ __forceinline__ bool is_nan_bits(T v);
template <> __device__ __forceinline__ bool is_nan_bits<double>(double v) { return (__double2hiint(v) & 0x7fffffff) >= 0x7ff80000; }
template <> __device__ __forceinline__ bool is_nan_bits<float>(float) { return false; }

template <typename T> __device__ __noinline__ void exact_delta_alpha(T ph0, T ph1, bool top, T at, T* d, T* a) {
    exactm::hyb_delta_alpha<T>(ph0, ph1, top, at, *d, *a);
}

// cold path of the column kernel's output form: out of line, so the six-way switch with IEEE divisions stays out of the
// level loop (inlined it was most of the loop's 1680 instructions and pushed the kernel into spills)
template <typename T> __device__ __noinline__ T exact_height_output(T dphi, T zs, int mode) {
    return exactm::height_output(dphi, zs, exactm::geom_from_z(zs), mode);
}

template <typename T> __device__ __forceinline__ void delta_alpha(T ph0, T ph1, bool top, T at, T& d, T& a) {
#if EK_LEAN_DEVICE
    fastm::hyb_delta_alpha<T>(ph0, ph1, top, at, d, a);
    if (sizeof(T) == 8 && __builtin_expect(is_nan_bits(d) || is_nan_bits(a), 0)) {
        T d2, a2;
        exact_delta_alpha<T>(ph0, ph1, top, at, &d2, &a2);
        d = d2;
        a = a2;
    }
#else
    exactm::hyb_delta_alpha<T>(ph0, ph1, top, at, d, a);
#endif
}

// loads / stores of one thread's VEC consecutive points of a row; vector path when aligned and in range
template <typename T, bool VECOK> __device__ __forceinline__ void ld_row(const T* row, int64_t i0, int64_t npl, T* v, bool streaming) {
    constexpr int VEC = Vec16<T>::N;
    if (VECOK) {  // the vector instantiation is only launched when npl is a multiple of VEC: i0 < npl implies the whole vector is in range
        if (streaming) {
            Vec16<T>::load(row + i0, v);
        } else {
#pragma unroll
            for (int j = 0; j < VEC; ++j) v[j] = __ldg(row + i0 + j);
        }
    } else {
#pragma unroll
        for (int j = 0; j < VEC; ++j) v[j] = (i0 + j < npl) ? __ldg(row + i0 + j) : T(1);
    }
}
template <typename T, bool VECOK> __device__ __forceinline__ void st_row(T* row, int64_t i0, int64_t npl, const T* v) {
    constexpr int VEC = Vec16<T>::N;
    if (VECOK) {
        Vec16<T>::store(row + i0, v);
    } else {
#pragma unroll
        for (int j = 0; j < VEC; ++j)
            if (i0 + j < npl) __stcs(row + i0 + j, v[j]);
    }
}

// delta / alpha rows of a float32 launch stored as float64 (what the reference returns: it allocates them with xp.zeros(...),
// V:672,686): the float32 values, widened in the store
template <bool VECOK> __device__ __forceinline__ void st_row_f64(double* row, int64_t i0, int64_t npl, const float* v) {
    if (VECOK) {
        __stcs(reinterpret_cast<double2*>(row + i0), make_double2((double)v[0], (double)v[1]));
        __stcs(reinterpret_cast<double2*>(row + i0 + 2), make_double2((double)v[2], (double)v[3]));
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (i0 + j < npl) __stcs(row + i0 + j, (double)v[j]);
    }
}
template <bool VECOK> __device__ __forceinline__ void st_row_f64(double* row, int64_t i0, int64_t npl, const double* v) {
    st_row<double, VECOK>(row, i0, npl, v);
}

struct HybridArgs {
    const void* sp;
    const void* A;         // nhalf half-level coefficients (device)
    const void* B;
    const int* full_rows;  // full-level index k (0-based) of every full/delta/alpha output row
    const int* half_rows;  // half-level index of every half output row
    int n_full, n_half;
    int top_k;     // the full level treated as the column top (first level of the computed band, V:645-647)
    int top_toa;   // any(p_half[top] <= 0.1) over the field (V:678)
    double alpha_top;
    void *full, *half, *delta, *alpha;
    int64_t npl;
    int rows_per_item;
    int ad_f64;  // delta / alpha are float64 arrays whatever T is
};

template <typename T, bool VECOK>
__global__ void __launch_bounds__(kThreads, kMinCtas) hybrid_pressure_kernel(const HybridArgs g) {
    constexpr int VEC = Vec16<T>::N;
    constexpr int TILE = kThreads * VEC;
    const bool want_da = g.delta != nullptr || g.alpha != nullptr;
#if EK_LEAN_DEVICE
    if (sizeof(T) == 8 && want_da) lean::init_tables();  // only delta / alpha take a logarithm (the launch passes no shared memory otherwise)
#endif
    const T* A = static_cast<const T*>(g.A);
    const T* B = static_cast<const T*>(g.B);
    const int64_t ptiles = (g.npl + TILE - 1) / TILE;
    const int n_rows = g.n_full > g.n_half ? g.n_full : g.n_half;
    const int chunks = (n_rows + g.rows_per_item - 1) / g.rows_per_item;
    const int64_t items = ptiles * chunks;
    for (int64_t it = blockIdx.x; it < items; it += gridDim.x) {
        const int64_t pt = it / chunks;
        const int r0 = (int)(it - pt * chunks) * g.rows_per_item;
        const int64_t i0 = pt * TILE + (int64_t)threadIdx.x * VEC;
        if (i0 >= g.npl) continue;
        T sp[VEC];
        ld_row<T, VECOK>(static_cast<const T*>(g.sp), i0, g.npl, sp, false);
        for (int r = r0; r < r0 + g.rows_per_item; ++r) {
            if (r < g.n_full && (g.full != nullptr || want_da)) {
                const int k = g.full_rows[r];
                const T a0 = __ldg(A + k), b0 = __ldg(B + k), a1 = __ldg(A + k + 1), b1 = __ldg(B + k + 1);
                const bool top = g.top_toa && k == g.top_k;
                T f[VEC], d[VEC], al[VEC];
#pragma unroll
                for (int j = 0; j < VEC; ++j) {
                    const T ph0 = exactm::hyb_half(a0, b0, sp[j]), ph1 = exactm::hyb_half(a1, b1, sp[j]);
                    f[j] = exactm::hyb_full(ph0, ph1);
                    if (want_da) delta_alpha<T>(ph0, ph1, top, static_cast<T>(g.alpha_top), d[j], al[j]);
                }
                const int64_t off = (int64_t)r * g.npl;
                if (g.full) st_row<T, VECOK>(static_cast<T*>(g.full) + off, i0, g.npl, f);
                if (g.ad_f64) {
                    if (g.delta) st_row_f64<VECOK>(static_cast<double*>(g.delta) + off, i0, g.npl, d);
                    if (g.alpha) st_row_f64<VECOK>(static_cast<double*>(g.alpha) + off, i0, g.npl, al);
                } else {
                    if (g.delta) st_row<T, VECOK>(static_cast<T*>(g.delta) + off, i0, g.npl, d);
                    if (g.alpha) st_row<T, VECOK>(static_cast<T*>(g.alpha) + off, i0, g.npl, al);
                }
            }
            if (r < g.n_half && g.half != nullptr) {
                const int h = g.half_rows[r];
                const T a0 = __ldg(A + h), b0 = __ldg(B + h);
                T ph[VEC];
#pragma unroll
                for (int j = 0; j < VEC; ++j) ph[j] = exactm::hyb_half(a0, b0, sp[j]);
                st_row<T, VECOK>(static_cast<T*>(g.half) + (int64_t)r * g.npl, i0, g.npl, ph);
            }
        }
    }
}

// any(A0 + B0 * sp <= thr) over the field (V:678): one flag for the whole launch
template <typename T> __global__ void any_le_kernel(const T* sp, int64_t n, T a0, T b0, T thr, int* flag) {
    int hit = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        hit |= (exactm::hyb_half(a0, b0, __ldg(sp + i)) <= thr) ? 1 : 0;
    if (__syncthreads_or(hit) && threadIdx.x == 0) atomicOr(flag, 1);
}

struct SuiteHybridArgs {
    const void *t, *q, *sp, *A, *B;  // t, q: [nlev, npl]; sp: [npl]; A, B: nlev + 1 half-level coefficients
    void* outs[S_NSLOTS];
    void* p_out;  // optional: the full-level pressure itself
    int nlev;
    int64_t npl;
    int rows_per_item;
};

// Half-level coefficients in shared memory, behind the lean tables: A[0..nhalf), then B[0..nhalf), as T.  One copy per CTA;
// reads in the level loop are warp-uniform (broadcast).  (Through the read-only global path the compiler hoisted the four
// loads of a level far above their use and spilled them: 8 local-memory round trips per level at the 64-register cap.)
template <typename T> __device__ __forceinline__ T* coef_smem() {
    extern __shared__ __align__(16) unsigned char ek_smem_raw[];
    return reinterpret_cast<T*>(ek_smem_raw + (sizeof(T) == 8 ? kSmemBytes : 0u));
}
template <typename T> __device__ __forceinline__ void coef_smem_fill(const T* A, const T* B, int first, int n) {
    T* c = coef_smem<T>();
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        c[i] = __ldg(A + first + i);
        c[n + i] = __ldg(B + first + i);
    }
    __syncthreads();
}
template <typename T> constexpr unsigned coef_smem_bytes(int nhalf) { return 2u * (unsigned)nhalf * (unsigned)sizeof(T); }

template <class Op, class OpE, typename T, bool VECOK>
__global__ void __launch_bounds__(kThreads, kHybMinCtas) suite_hybrid_kernel(const SuiteHybridArgs g, const Params P) {
    constexpr int VEC = Vec16<T>::N;
    constexpr int TILE = kThreads * VEC;
    constexpr int LU = kHybLevels;  // levels in flight per thread (their loads are issued before any math)
#if EK_LEAN_DEVICE
    if (sizeof(T) == 8) lean::init_tables();
#endif
    const int nhalf = g.nlev + 1;
    coef_smem_fill<T>(static_cast<const T*>(g.A), static_cast<const T*>(g.B), 0, nhalf);
    const T* sA = coef_smem<T>();
    const T* sB = sA + nhalf;
    const T* tq[2] = {static_cast<const T*>(g.t), static_cast<const T*>(g.q)};
    const int64_t ptiles = (g.npl + TILE - 1) / TILE;
    const int chunks = (g.nlev + g.rows_per_item - 1) / g.rows_per_item;
    const int64_t items = ptiles * chunks;
    for (int64_t it = blockIdx.x; it < items; it += gridDim.x) {
        const int64_t pt = it / chunks;
        const int k0 = (int)(it - pt * chunks) * g.rows_per_item;
        const int k1 = min(k0 + g.rows_per_item, g.nlev);
        const int64_t i0 = pt * TILE + (int64_t)threadIdx.x * VEC;
        if (i0 >= g.npl) continue;
        T sp[VEC], ph[VEC];  // ph: pressure of the half level on top of the current level, carried down the column
        ld_row<T, VECOK>(static_cast<const T*>(g.sp), i0, g.npl, sp, false);
        {
            const T a0 = sA[k0], b0 = sB[k0];
#pragma unroll
            for (int j = 0; j < VEC; ++j) ph[j] = exactm::hyb_half(a0, b0, sp[j]);  // V:663
        }
        for (int k = k0; k < k1; k += LU) {
            T x[LU][2][VEC];
#pragma unroll
            for (int u = 0; u < LU; ++u)
                if (k + u < k1) {
#pragma unroll
                    for (int c = 0; c < 2; ++c) ld_row<T, VECOK>(tq[c] + (int64_t)(k + u) * g.npl, i0, g.npl, x[u][c], true);
                }
#pragma unroll
            for (int u = 0; u < LU; ++u)  // ask L2 for a later group of levels while this group is being computed
                if (k + LU * kHybPfDist + u < k1) {
#pragma unroll
                    for (int c = 0; c < 2; ++c) asm volatile("prefetch.global.L2 [%0];" ::"l"(tq[c] + (int64_t)(k + LU * kHybPfDist + u) * g.npl + i0));
                }
#pragma unroll
            for (int u = 0; u < LU; ++u) {
                if (k + u >= k1) break;
                const int kk = k + u;
                const T a1 = sA[kk + 1], b1 = sB[kk + 1];
                T y[S_NSLOTS][VEC], pf[VEC];
#pragma unroll
                for (int j = 0; j < VEC; ++j) {
                    const T ph1 = exactm::hyb_half(a1, b1, sp[j]);
                    pf[j] = exactm::hyb_full(ph[j], ph1);  // V:708; the same two half-level values the reference forms
                    ph[j] = ph1;
                    T a[3] = {x[u][0][j], x[u][1][j], pf[j]}, r[S_NSLOTS];
                    point<Op, OpE, T>(a, r, P, 3u);  // t and q are the array inputs; p is derived
#pragma unroll
                    for (int o = 0; o < S_NSLOTS; ++o) y[o][j] = r[o];
                }
                const int64_t off = (int64_t)kk * g.npl;
#pragma unroll
                for (int o = 0; o < S_NSLOTS; ++o) {
                    const bool w = Op::STATIC_MASK ? (((Op::STATIC_MASK >> o) & 1u) != 0) : (g.outs[o] != nullptr);
                    if (w) st_row<T, VECOK>(static_cast<T*>(g.outs[o]) + off, i0, g.npl, y[o]);
                }
                if (g.p_out) st_row<T, VECOK>(static_cast<T*>(g.p_out) + off, i0, g.npl, pf);
            }
        }
    }
}

struct GeoArgs {
    const void *t, *q;           // [nlev, npl], level 0 = top of the band
    const void *sp, *A, *B;      // computed alpha/delta: surface pressure + half-level coefficients of the WHOLE model
    const void *alpha, *delta;   // given alpha/delta: [nlev, npl]
    const void* zs;              // surface geopotential [npl] (modes that need it)
    void* out;                   // [nlev, npl]
    int nlev;
    int64_t npl;
    int band0;     // half-level index of the band's top (model levels - nlev)
    int top_toa;   // field-wide any(p_half[band0] <= 0.1) (V:678)
    double alpha_top;
    int mode;      // HeightMode
};

// One thread walks VEC columns from the bottom level to the top one: d = R(q) t, dphi_k = sum_{j>k} d_j delta_j + d_k alpha_k
// (V:799-810, same accumulation order as the reference's flipped cumulative sum).  alpha/delta come from registers
// (sp and the half-level coefficients in shared memory; the pressure of the half level under the current level is carried
// up the column, so a level forms one new half-level pressure) or from memory (GIVEN_AD).  Loads of two levels are in
// flight before the math of the lower one.
// MODE >= 0: the output form is a compile-time constant (the registers of zs / geom(zs) and the form choices drop out of
// the level loop where they are not needed); MODE = -1: taken from g.mode at run time (the rarer launch shapes).
template <typename T, bool GIVEN_AD, bool VECOK, int MODE>
__global__ void __launch_bounds__(kThreads, (MODE >= EK_HM_GEOM_SEA ? kColMinCtasGeom : kColMinCtas)) column_geopotential_kernel(const GeoArgs g) {
    const int mode = MODE >= 0 ? MODE : g.mode;
    constexpr int VEC = Vec16<T>::N;
    constexpr int TILE = kThreads * VEC;
    constexpr int NARR = GIVEN_AD ? 4 : 2;
    // levels in flight per thread: the geometric-height forms (a reciprocal more per level) fit their registers only with one
    // (measured: geometric height 0.58 -> 0.61 with 1, thickness 0.77 -> 0.75)
    constexpr int CLU = GIVEN_AD ? 2 : (MODE >= EK_HM_GEOM_SEA ? 1 : kColLevels);
#if EK_LEAN_DEVICE
    if (sizeof(T) == 8) lean::init_tables();
#endif
    const T* sA = nullptr;
    const T* sB = nullptr;
    if (!GIVEN_AD) {  // the band's nlev + 1 half-level coefficients
        coef_smem_fill<T>(static_cast<const T*>(g.A), static_cast<const T*>(g.B), g.band0, g.nlev + 1);
        sA = coef_smem<T>();
        sB = sA + (g.nlev + 1);
    }
    const T* arr[4] = {static_cast<const T*>(g.t), static_cast<const T*>(g.q), static_cast<const T*>(g.alpha), static_cast<const T*>(g.delta)};
    const int64_t ptiles = (g.npl + TILE - 1) / TILE;
    for (int64_t pt = blockIdx.x; pt < ptiles; pt += gridDim.x) {
        const int64_t i0 = pt * TILE + (int64_t)threadIdx.x * VEC;
        if (i0 >= g.npl) continue;
        T sp[VEC], zs[VEC], hsub[VEC], sum[VEC], phb[VEC];  // phb: pressure of the half level under the current level
#pragma unroll
        for (int j = 0; j < VEC; ++j) sp[j] = zs[j] = hsub[j] = sum[j] = phb[j] = T(0);
        if (!GIVEN_AD) {
            ld_row<T, VECOK>(static_cast<const T*>(g.sp), i0, g.npl, sp, false);
            const T ab = sA[g.nlev], bb = sB[g.nlev];
#pragma unroll
            for (int j = 0; j < VEC; ++j) phb[j] = exactm::hyb_half(ab, bb, sp[j]);  // V:663
        }
        const bool add_zs = mode != EK_HM_THICKNESS && mode != EK_HM_GH_GROUND;
        if (add_zs) ld_row<T, VECOK>(static_cast<const T*>(g.zs), i0, g.npl, zs, false);
        // The six output forms (V:1064-1069, V:1163-1188) as one expression: z = dphi (+ zs), then nothing / z/g / the
        // geometric height of z minus hsub (geom(zs) or 0: subtracting 0 changes no bit), so the level loop carries
        // warp-uniform two- and three-way choices instead of a six-way switch.
        const int form = mode >> 1;  // 0: geopotential units, 1: geopotential height, 2: geometric height
        if (mode == EK_HM_GEOM_GROUND) {
#pragma unroll
            for (int j = 0; j < VEC; ++j) hsub[j] = EK_FAST_NS::geom_from_z(zs[j]);
        }
        for (int k = g.nlev - 1; k >= 0; k -= CLU) {
            T x[CLU][NARR][VEC];
#pragma unroll
            for (int u = 0; u < CLU; ++u)
                if (k - u >= 0) {
#pragma unroll
                    for (int c = 0; c < NARR; ++c) ld_row<T, VECOK>(arr[c] + (int64_t)(k - u) * g.npl, i0, g.npl, x[u][c], true);
                }
#pragma unroll
            for (int u = 0; u < CLU; ++u)
                if (k - CLU * kColPfDist - u >= 0) {
#pragma unroll
                    for (int c = 0; c < NARR; ++c) asm volatile("prefetch.global.L2 [%0];" ::"l"(arr[c] + (int64_t)(k - CLU * kColPfDist - u) * g.npl + i0));
                }
#pragma unroll
            for (int u = 0; u < CLU; ++u) {
                const int kk = k - u;
                if (kk < 0) break;
                T a0 = T(0), b0 = T(0);
                if (!GIVEN_AD) a0 = sA[kk], b0 = sB[kk];
                const bool top = g.top_toa && kk == 0;
                T y[VEC];
#pragma unroll
                for (int j = 0; j < VEC; ++j) {
                    T al, de;
                    if (GIVEN_AD) {
                        al = x[u][2][j];
                        de = x[u][3][j];
                    } else {
                        const T pht = exactm::hyb_half(a0, b0, sp[j]);  // the half level on top of this level (V:663)
                        delta_alpha<T>(pht, phb[j], top, static_cast<T>(g.alpha_top), de, al);
                        phb[j] = pht;
                    }
                    const T d = exactm::gas_constant(x[u][1][j]) * x[u][0][j];
                    // the running sum starts at 0: 0 + x is x, so the bottom level needs no special case
                    const T dphi = sum[j] + d * al;  // V:808-809
                    sum[j] = sum[j] + d * de;        // V:804 (running sum of d * delta below this layer)
                    const T z = add_zs ? dphi + zs[j] : dphi;
                    T h = form == 0 ? z : (form == 1 ? EK_FAST_NS::gh_from_z(z) : EK_FAST_NS::geom_from_z(z) - hsub[j]);
#if EK_LEAN_DEVICE
                    if (sizeof(T) == 8 && __builtin_expect(is_nan_bits(h), 0)) h = exact_height_output<T>(dphi, zs[j], mode);
#endif
                    y[j] = h;
                }
                st_row<T, VECOK>(static_cast<T*>(g.out) + (int64_t)kk * g.npl, i0, g.npl, y);
            }
        }
    }
}

struct SuiteGeoArgs {
    const void *t, *q, *sp, *zs, *A, *B;  // t, q: [nlev, npl]; sp, zs: [npl] (zs may be NULL when no output adds it); A, B: nlev + 1
    void* outs[S_NSLOTS];
    void* p_out;                          // optional: the full-level pressure
    void *thickness, *z, *height;         // optional column outputs [nlev, npl]
    int nlev;
    int64_t npl;
    int top_toa;   // field-wide any(p_half[0] <= 0.1) (V:678)
    double alpha_top;
    int mode;      // HeightMode of `height`
};

// The (t, q, p) suite and the geopotential of the same levels in one walk: one thread per VEC columns from the bottom level to the
// top one, as column_geopotential_kernel (computed alpha/delta).  A level forms its top half-level pressure once; the full-level
// pressure (the same two operands as suite_hybrid_kernel: bit-identical to pressure_on_hybrid_levels), delta and alpha all come
// from it and the half level below.  The three column outputs are forms of the same dphi; the height form is a warp-uniform
// run-time value (column_geopotential_kernel's MODE = -1 expression).
template <class Op, class OpE, typename T, bool VECOK>
__global__ void __launch_bounds__(kThreads, kGeoMinCtas) suite_geo_kernel(const SuiteGeoArgs g, const Params P) {
    constexpr int VEC = Vec16<T>::N;
    constexpr int TILE = kThreads * VEC;
    constexpr int LU = kGeoLevels;
#if EK_LEAN_DEVICE
    if (sizeof(T) == 8) lean::init_tables();
#endif
    const int nhalf = g.nlev + 1;
    coef_smem_fill<T>(static_cast<const T*>(g.A), static_cast<const T*>(g.B), 0, nhalf);
    const T* sA = coef_smem<T>();
    const T* sB = sA + nhalf;
    const T* tq[2] = {static_cast<const T*>(g.t), static_cast<const T*>(g.q)};
    const int mode = g.mode;
    const bool want_h = g.height != nullptr;
    const bool h_zs = want_h && mode != EK_HM_THICKNESS && mode != EK_HM_GH_GROUND;
    const int form = mode >> 1;  // 0: geopotential units, 1: geopotential height, 2: geometric height
    const T at = static_cast<T>(g.alpha_top);
    const int64_t ptiles = (g.npl + TILE - 1) / TILE;
    for (int64_t pt = blockIdx.x; pt < ptiles; pt += gridDim.x) {
        const int64_t i0 = pt * TILE + (int64_t)threadIdx.x * VEC;
        if (i0 >= g.npl) continue;
        T sp[VEC], zs[VEC], hsub[VEC], sum[VEC], phb[VEC];  // phb: pressure of the half level under the current level
#pragma unroll
        for (int j = 0; j < VEC; ++j) zs[j] = hsub[j] = sum[j] = T(0);
        ld_row<T, VECOK>(static_cast<const T*>(g.sp), i0, g.npl, sp, false);
        {
            const T ab = sA[g.nlev], bb = sB[g.nlev];
#pragma unroll
            for (int j = 0; j < VEC; ++j) phb[j] = exactm::hyb_half(ab, bb, sp[j]);  // V:663
        }
        if (g.z || h_zs) ld_row<T, VECOK>(static_cast<const T*>(g.zs), i0, g.npl, zs, false);
        if (want_h && mode == EK_HM_GEOM_GROUND) {
#pragma unroll
            for (int j = 0; j < VEC; ++j) hsub[j] = EK_FAST_NS::geom_from_z(zs[j]);
        }
        for (int k = g.nlev - 1; k >= 0; k -= LU) {
            T x[LU][2][VEC];
#pragma unroll
            for (int u = 0; u < LU; ++u)
                if (k - u >= 0) {
#pragma unroll
                    for (int c = 0; c < 2; ++c) ld_row<T, VECOK>(tq[c] + (int64_t)(k - u) * g.npl, i0, g.npl, x[u][c], true);
                }
#pragma unroll
            for (int u = 0; u < LU; ++u)  // ask L2 for a later group of levels while this group is being computed
                if (k - LU * kGeoPfDist - u >= 0) {
#pragma unroll
                    for (int c = 0; c < 2; ++c) asm volatile("prefetch.global.L2 [%0];" ::"l"(tq[c] + (int64_t)(k - LU * kGeoPfDist - u) * g.npl + i0));
                }
#pragma unroll
            for (int u = 0; u < LU; ++u) {
                const int kk = k - u;
                if (kk < 0) break;
                const T a0 = sA[kk], b0 = sB[kk];
                const bool top = g.top_toa && kk == 0;
                T y[S_NSLOTS][VEC], pf[VEC], th[VEC], zz[VEC], hh[VEC];
#pragma unroll
                for (int j = 0; j < VEC; ++j) {
                    const T pht = exactm::hyb_half(a0, b0, sp[j]);  // the half level on top of this level (V:663)
                    pf[j] = exactm::hyb_full(pht, phb[j]);          // V:708
                    T de, al;
                    delta_alpha<T>(pht, phb[j], top, at, de, al);
                    phb[j] = pht;
                    T a[3] = {x[u][0][j], x[u][1][j], pf[j]}, r[S_NSLOTS];
                    point<Op, OpE, T>(a, r, P, 3u);  // t and q are the array inputs; p is derived
#pragma unroll
                    for (int o = 0; o < S_NSLOTS; ++o) y[o][j] = r[o];
                    const T d = exactm::gas_constant(x[u][1][j]) * x[u][0][j];
                    const T dphi = sum[j] + d * al;  // V:808-809
                    sum[j] = sum[j] + d * de;        // V:804
                    th[j] = dphi;
                    zz[j] = dphi + zs[j];
                    if (want_h) {
                        const T z = h_zs ? zz[j] : dphi;
                        T h = form == 0 ? z : (form == 1 ? EK_FAST_NS::gh_from_z(z) : EK_FAST_NS::geom_from_z(z) - hsub[j]);
#if EK_LEAN_DEVICE
                        if (sizeof(T) == 8 && __builtin_expect(is_nan_bits(h), 0)) h = exact_height_output<T>(dphi, zs[j], mode);
#endif
                        hh[j] = h;
                    }
                }
                const int64_t off = (int64_t)kk * g.npl;
#pragma unroll
                for (int o = 0; o < S_NSLOTS; ++o) {
                    const bool w = Op::STATIC_MASK ? (((Op::STATIC_MASK >> o) & 1u) != 0) : (g.outs[o] != nullptr);
                    if (w) st_row<T, VECOK>(static_cast<T*>(g.outs[o]) + off, i0, g.npl, y[o]);
                }
                if (g.p_out) st_row<T, VECOK>(static_cast<T*>(g.p_out) + off, i0, g.npl, pf);
                if (g.thickness) st_row<T, VECOK>(static_cast<T*>(g.thickness) + off, i0, g.npl, th);
                if (g.z) st_row<T, VECOK>(static_cast<T*>(g.z) + off, i0, g.npl, zz);
                if (want_h) st_row<T, VECOK>(static_cast<T*>(g.height) + off, i0, g.npl, hh);
            }
        }
    }
}

int grid_for(int64_t items) {
    const int sms = sm_count_current_device();
    if (sms <= 0) return -1;
    const int64_t cap = (int64_t)sms * g_ctas_per_sm.load(std::memory_order_relaxed);
    return (int)(items < cap ? (items > 0 ? items : 1) : cap);
}

// levels per work item: enough items to balance the grid, at least 2 levels each
int rows_per_item_for(int64_t ptiles, int n_rows) {
    const int sms = sm_count_current_device();
    const int64_t want_items = (int64_t)(sms > 0 ? sms : 148) * 64;
    int64_t chunks = (want_items + ptiles - 1) / ptiles;
    if (chunks < 1) chunks = 1;
    int rpi = (int)((n_rows + chunks - 1) / chunks);
    if (rpi < 2) rpi = 2;
    if (rpi & 1) ++rpi;
    return rpi;
}

bool ok16(const void* p) { return p == nullptr || aligned16(p); }

}  // namespace

template <typename T>
static int impl_pressure_on_hybrid_levels(const void* A, const void* B, int nhalf, const void* sp, int64_t npl, const int* full_rows, int n_full,
                                          const int* half_rows, int n_half, int top_k, int top_toa, double alpha_top, void* full, void* half,
                                          void* delta, void* alpha, int alpha_delta_f64, void* stream) {
    const char* what = "pressure_on_hybrid_levels";
    if (!A || !B || !sp || nhalf < 2 || npl < 0 || n_full < 0 || n_half < 0) return set_error(EK_ERR_ARG, "%s: bad arguments", what);
    if (!full && !half && !delta && !alpha) return set_error(EK_ERR_ARG, "%s: no output buffer given", what);
    if ((full || delta || alpha) && (n_full < 1 || !full_rows)) return set_error(EK_ERR_ARG, "%s: full/delta/alpha need full_rows", what);
    if (half && (n_half < 1 || !half_rows)) return set_error(EK_ERR_ARG, "%s: half needs half_rows", what);
    if (npl == 0) return EK_OK;
    HybridArgs g{sp, A, B, full_rows, half_rows, (full || delta || alpha) ? n_full : 0, half ? n_half : 0, top_k, top_toa, alpha_top,
                 full, half, delta, alpha, npl, 2, (alpha_delta_f64 || sizeof(T) == 8) ? 1 : 0};
    constexpr int TILE = kThreads * Vec16<T>::N;
    const int64_t ptiles = (npl + TILE - 1) / TILE;
    const int n_rows = g.n_full > g.n_half ? g.n_full : g.n_half;
    g.rows_per_item = rows_per_item_for(ptiles, n_rows);
    const int64_t items = ptiles * ((n_rows + g.rows_per_item - 1) / g.rows_per_item);
    const int blocks = grid_for(items);
    if (blocks < 0) return set_error(EK_ERR_ARG, "%s: no CUDA device is current", what);
    const bool vec = npl % Vec16<T>::N == 0 && ok16(sp) && ok16(full) && ok16(half) && ok16(delta) && ok16(alpha);
    const unsigned smem = (delta || alpha) ? smem_for<T>() : 0u;  // the log table, for delta / alpha only
    const int rc = vec ? launch_kernel_smem<&hybrid_pressure_kernel<T, true>>(blocks, static_cast<cudaStream_t>(stream), smem, g)
                       : launch_kernel_smem<&hybrid_pressure_kernel<T, false>>(blocks, static_cast<cudaStream_t>(stream), smem, g);
    if (rc) return rc;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return set_error((int)err, "%s: kernel launch failed: %s", what, cudaGetErrorString(err));
    return EK_OK;
}
EK_API(pressure_on_hybrid_levels,
       (const void* A, const void* B, int nhalf, const void* sp, int64_t npl, const int* full_rows, int n_full, const int* half_rows, int n_half,
        int top_k, int top_toa, double alpha_top, void* full, void* half, void* delta, void* alpha, int alpha_delta_f64, void* stream),
       (A, B, nhalf, sp, npl, full_rows, n_full, half_rows, n_half, top_k, top_toa, alpha_top, full, half, delta, alpha, alpha_delta_f64, stream))

template <typename T>
static int impl_hybrid_top_is_toa(const void* sp, int64_t npl, double a_top, double b_top, int* flag, void* stream) {
    if (!sp || !flag || npl < 0) return set_error(EK_ERR_ARG, "hybrid_top_is_toa: bad arguments");
    if (npl == 0) return EK_OK;
    const int blocks = grid_for((npl + 255) / 256);
    if (blocks < 0) return set_error(EK_ERR_ARG, "hybrid_top_is_toa: no CUDA device is current");
    any_le_kernel<T><<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(static_cast<const T*>(sp), npl, (T)a_top, (T)b_top, (T)0.1, flag);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return set_error((int)err, "hybrid_top_is_toa: kernel launch failed: %s", cudaGetErrorString(err));
    return EK_OK;
}
EK_API(hybrid_top_is_toa, (const void* sp, int64_t npl, double a_top, double b_top, int* flag, void* stream), (sp, npl, a_top, b_top, flag, stream))

template <typename T>
static int impl_geopotential_on_hybrid_levels(const void* t, const void* q, int nlev, int64_t npl, const void* sp, const void* A, const void* B,
                                              int nhalf, int top_toa, double alpha_top, const void* alpha, const void* delta, const void* zs,
                                              int mode, void* out, void* stream) {
    const char* what = "geopotential_on_hybrid_levels";
    const bool given = alpha != nullptr || delta != nullptr;
    if (!t || !q || !out || nlev < 1 || npl < 0 || mode < 0 || mode > 5) return set_error(EK_ERR_ARG, "%s: bad arguments", what);
    if (given && (!alpha || !delta)) return set_error(EK_ERR_ARG, "%s: alpha and delta must be given together", what);
    if (!given && (!sp || !A || !B || nhalf < nlev + 1)) return set_error(EK_ERR_ARG, "%s: sp, A, B (>= nlev + 1 half-levels) are required", what);
    if ((mode == 1 || mode == 2 || mode == 4 || mode == 5) && !zs) return set_error(EK_ERR_ARG, "%s: this output needs the surface geopotential zs", what);
    if (npl == 0) return EK_OK;
    GeoArgs g{t, q, sp, A, B, alpha, delta, zs, out, nlev, npl, given ? 0 : nhalf - 1 - nlev, top_toa, alpha_top, mode};
    constexpr int TILE = kThreads * Vec16<T>::N;
    const int blocks = grid_for((npl + TILE - 1) / TILE);
    if (blocks < 0) return set_error(EK_ERR_ARG, "%s: no CUDA device is current", what);
    const bool vec = npl % Vec16<T>::N == 0 && ok16(t) && ok16(q) && ok16(sp) && ok16(alpha) && ok16(delta) && ok16(zs) && ok16(out);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const unsigned smem = smem_for<T>() + (given ? 0u : coef_smem_bytes<T>(nlev + 1));  // lean tables + the band's half-level coefficients
    if (smem > 200u * 1024u) return set_error(EK_ERR_ARG, "%s: nlev=%d is too large for the shared-memory coefficient copy", what, nlev);
    int rc;
    if (given) {
        if (vec) rc = launch_kernel_smem<&column_geopotential_kernel<T, true, true, -1>>(blocks, st, smem, g);
        else rc = launch_kernel_smem<&column_geopotential_kernel<T, true, false, -1>>(blocks, st, smem, g);
    } else if (!vec) {
        rc = launch_kernel_smem<&column_geopotential_kernel<T, false, false, -1>>(blocks, st, smem, g);
    } else {  // the whole-field case: one instantiation per output form
        switch (mode) {
            case EK_HM_THICKNESS: rc = launch_kernel_smem<&column_geopotential_kernel<T, false, true, EK_HM_THICKNESS>>(blocks, st, smem, g); break;
            case EK_HM_GEOPOTENTIAL: rc = launch_kernel_smem<&column_geopotential_kernel<T, false, true, EK_HM_GEOPOTENTIAL>>(blocks, st, smem, g); break;
            case EK_HM_GH_SEA: rc = launch_kernel_smem<&column_geopotential_kernel<T, false, true, EK_HM_GH_SEA>>(blocks, st, smem, g); break;
            case EK_HM_GH_GROUND: rc = launch_kernel_smem<&column_geopotential_kernel<T, false, true, EK_HM_GH_GROUND>>(blocks, st, smem, g); break;
            case EK_HM_GEOM_SEA: rc = launch_kernel_smem<&column_geopotential_kernel<T, false, true, EK_HM_GEOM_SEA>>(blocks, st, smem, g); break;
            default: rc = launch_kernel_smem<&column_geopotential_kernel<T, false, true, EK_HM_GEOM_GROUND>>(blocks, st, smem, g); break;
        }
    }
    if (rc) return rc;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return set_error((int)err, "%s: kernel launch failed: %s", what, cudaGetErrorString(err));
    return EK_OK;
}
EK_API(geopotential_on_hybrid_levels,
       (const void* t, const void* q, int nlev, int64_t npl, const void* sp, const void* A, const void* B, int nhalf, int top_toa,
        double alpha_top, const void* alpha, const void* delta, const void* zs, int mode, void* out, void* stream),
       (t, q, nlev, npl, sp, A, B, nhalf, top_toa, alpha_top, alpha, delta, zs, mode, out, stream))

// The suite arguments shared by the hybrid launchers: the ept method (reset to IFS when no slot uses it) and the output table
// of the requested slots; `vec` is cleared when a buffer is not 16-byte aligned.
static int suite_outputs(const char* what, void* const* outs, uint32_t out_mask, bool any_other, int& ept_method, void** dst, bool& vec) {
    if (out_mask >= (1u << S_NSLOTS) || (out_mask == 0 && !any_other)) return set_error(EK_ERR_ARG, "%s: out_mask=0x%x selects no output", what, out_mask);
    constexpr uint32_t EPT = (1u << S_EPT) | (1u << S_WBPT);
    if (!(out_mask & EPT)) ept_method = EK_EPT_IFS;
    if (ept_method < EK_EPT_IFS || ept_method > EK_EPT_BOLTON39) return set_error(EK_ERR_ENUM, "%s: invalid ept method id %d", what, ept_method);
    for (int k = 0; k < S_NSLOTS; ++k) {
        dst[k] = ((out_mask >> k) & 1u) ? (outs ? outs[k] : nullptr) : nullptr;
        if (((out_mask >> k) & 1u) && !dst[k]) return set_error(EK_ERR_ARG, "%s: output %d requested but its buffer is NULL", what, k);
        vec = vec && ok16(dst[k]);
    }
    return EK_OK;
}

// The suite instantiations of the hybrid kernels: a run-time mask for each non-IFS ept method, and for IFS the two common static
// masks (the default five outputs, and those with ept + wbpt) or a run-time mask.  LAUNCH(MASK, EPT_METHOD) launches one.
#define EK_SUITE_DISPATCH(LAUNCH)         \
    do {                                  \
        if (ept_method == EK_EPT_BOLTON35) \
            LAUNCH(0, EPT_BOLTON35);       \
        else if (ept_method == EK_EPT_BOLTON39) \
            LAUNCH(0, EPT_BOLTON39);       \
        else if (out_mask == 0x1F)         \
            LAUNCH(0x1F, EPT_IFS);         \
        else if (out_mask == 0x31F)        \
            LAUNCH(0x31F, EPT_IFS);        \
        else                               \
            LAUNCH(0, EPT_IFS);            \
    } while (0)

template <template <uint32_t, int> class OpM, template <uint32_t, int> class OpME, typename T>
static int suite_hybrid(const void* t, const void* q, const void* sp, const void* A, const void* B, int nlev, int64_t npl, void* const* outs,
                        uint32_t out_mask, int ept_method, void* p_out, void* stream) {
    const char* what = "suite_tq_hybrid";
    if (!t || !q || !sp || !A || !B || nlev < 1 || npl < 0) return set_error(EK_ERR_ARG, "%s: bad arguments", what);
    SuiteHybridArgs g{t, q, sp, A, B, {}, p_out, nlev, npl, 2};
    bool vec = npl % Vec16<T>::N == 0 && ok16(t) && ok16(q) && ok16(sp) && ok16(p_out);
    if (int rc = suite_outputs(what, outs, out_mask, p_out != nullptr, ept_method, g.outs, vec)) return rc;
    if (npl == 0) return EK_OK;
    constexpr int TILE = kThreads * Vec16<T>::N;
    const int64_t ptiles = (npl + TILE - 1) / TILE;
    g.rows_per_item = rows_per_item_for(ptiles, nlev);
    const int64_t items = ptiles * ((nlev + g.rows_per_item - 1) / g.rows_per_item);
    const int blocks = grid_for(items);
    if (blocks < 0) return set_error(EK_ERR_ARG, "%s: no CUDA device is current", what);
    Params P;
    P.out_mask = out_mask;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const unsigned smem = smem_for<T>() + coef_smem_bytes<T>(nlev + 1);  // lean tables (float64) + the half-level coefficients
    if (smem > 200u * 1024u) return set_error(EK_ERR_ARG, "%s: nlev=%d is too large for the shared-memory coefficient copy", what, nlev);
#define EK_LAUNCH_SH(M, EM)                                                                                      \
    do {                                                                                                         \
        if (vec)                                                                                                 \
            rc = launch_kernel_smem<&suite_hybrid_kernel<OpM<M, EM>, OpME<M, EM>, T, true>>(blocks, st, smem, g, P); \
        else                                                                                                     \
            rc = launch_kernel_smem<&suite_hybrid_kernel<OpM<M, EM>, OpME<M, EM>, T, false>>(blocks, st, smem, g, P); \
    } while (0)
    int rc;
    EK_SUITE_DISPATCH(EK_LAUNCH_SH);
    if (rc) return rc;
#undef EK_LAUNCH_SH
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return set_error((int)err, "%s: kernel launch failed: %s", what, cudaGetErrorString(err));
    return EK_OK;
}

template <template <uint32_t, int> class OpM, template <uint32_t, int> class OpME, typename T>
static int suite_hybrid_geo(const void* t, const void* q, const void* sp, const void* zs, const void* A, const void* B, int nlev, int64_t npl,
                            void* const* outs, uint32_t out_mask, int ept_method, void* p_out, int top_toa, double alpha_top, void* thickness_out,
                            void* z_out, void* height_out, int height_mode, void* stream) {
    const char* what = "suite_tq_hybrid_geo";
    if (!t || !q || !sp || !A || !B || nlev < 1 || npl < 0) return set_error(EK_ERR_ARG, "%s: bad arguments", what);
    if (height_out && (height_mode < EK_HM_THICKNESS || height_mode > EK_HM_GEOM_GROUND))
        return set_error(EK_ERR_ENUM, "%s: invalid height mode %d", what, height_mode);
    const bool need_zs = z_out || (height_out && height_mode != EK_HM_THICKNESS && height_mode != EK_HM_GH_GROUND);
    if (need_zs && !zs) return set_error(EK_ERR_ARG, "%s: this output needs the surface geopotential zs", what);
    SuiteGeoArgs g{t, q, sp, need_zs ? zs : nullptr, A, B, {}, p_out, thickness_out, z_out, height_out, nlev, npl, top_toa, alpha_top,
                   height_out ? height_mode : EK_HM_THICKNESS};
    bool vec = npl % Vec16<T>::N == 0 && ok16(t) && ok16(q) && ok16(sp) && ok16(g.zs) && ok16(p_out) && ok16(thickness_out) && ok16(z_out) &&
               ok16(height_out);
    const bool other = p_out || thickness_out || z_out || height_out;
    if (int rc = suite_outputs(what, outs, out_mask, other, ept_method, g.outs, vec)) return rc;
    if (npl == 0) return EK_OK;
    constexpr int TILE = kThreads * Vec16<T>::N;
    const int blocks = grid_for((npl + TILE - 1) / TILE);  // one work item per column tile: the level walk is sequential
    if (blocks < 0) return set_error(EK_ERR_ARG, "%s: no CUDA device is current", what);
    Params P;
    P.out_mask = out_mask;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const unsigned smem = smem_for<T>() + coef_smem_bytes<T>(nlev + 1);  // lean tables (float64) + the half-level coefficients
    if (smem > 200u * 1024u) return set_error(EK_ERR_ARG, "%s: nlev=%d is too large for the shared-memory coefficient copy", what, nlev);
#define EK_LAUNCH_SG(M, EM)                                                                                      \
    do {                                                                                                         \
        if (vec)                                                                                                 \
            rc = launch_kernel_smem<&suite_geo_kernel<OpM<M, EM>, OpME<M, EM>, T, true>>(blocks, st, smem, g, P); \
        else                                                                                                     \
            rc = launch_kernel_smem<&suite_geo_kernel<OpM<M, EM>, OpME<M, EM>, T, false>>(blocks, st, smem, g, P); \
    } while (0)
    int rc;
    EK_SUITE_DISPATCH(EK_LAUNCH_SG);
    if (rc) return rc;
#undef EK_LAUNCH_SG
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t err = cudaGetLastError();
    if (err != cudaSuccess) return set_error((int)err, "%s: kernel launch failed: %s", what, cudaGetErrorString(err));
    return EK_OK;
}

template <typename T>
static int impl_suite_tq_hybrid(const void* t, const void* q, const void* sp, const void* A, const void* B, int nlev, int64_t npl,
                                void* const* outs, uint32_t out_mask, int ept_method, void* p_out, void* stream) {
    return suite_hybrid<EK_OPS(OpSuiteTQPm), T>(t, q, sp, A, B, nlev, npl, outs, out_mask, ept_method, p_out, stream);
}
EK_API(suite_tq_hybrid,
       (const void* t, const void* q, const void* sp, const void* A, const void* B, int nlev, int64_t npl, void* const* outs, uint32_t out_mask,
        int ept_method, void* p_out, void* stream),
       (t, q, sp, A, B, nlev, npl, outs, out_mask, ept_method, p_out, stream))

template <typename T>
static int impl_suite_tq_hybrid_geo(const void* t, const void* q, const void* sp, const void* zs, const void* A, const void* B, int nlev, int64_t npl,
                                    void* const* outs, uint32_t out_mask, int ept_method, void* p_out, int top_toa, double alpha_top,
                                    void* thickness_out, void* z_out, void* height_out, int height_mode, void* stream) {
    return suite_hybrid_geo<EK_OPS(OpSuiteTQPm), T>(t, q, sp, zs, A, B, nlev, npl, outs, out_mask, ept_method, p_out, top_toa, alpha_top, thickness_out,
                                                    z_out, height_out, height_mode, stream);
}
EK_API(suite_tq_hybrid_geo,
       (const void* t, const void* q, const void* sp, const void* zs, const void* A, const void* B, int nlev, int64_t npl, void* const* outs,
        uint32_t out_mask, int ept_method, void* p_out, int top_toa, double alpha_top, void* thickness_out, void* z_out, void* height_out,
        int height_mode, void* stream),
       (t, q, sp, zs, A, B, nlev, npl, outs, out_mask, ept_method, p_out, top_toa, alpha_top, thickness_out, z_out, height_out, height_mode, stream))

// used by the host-buffer pipeline in ek_api.cu
template <typename T>
int ek_suite_launch_hybrid(const void* t, const void* q, const void* sp, const void* A, const void* B, int nlev, int64_t npl, void* const* outs,
                           uint32_t out_mask, int ept_method, void* stream) {
    return suite_hybrid<EK_OPS(OpSuiteTQPm), T>(t, q, sp, A, B, nlev, npl, outs, out_mask, ept_method, nullptr, stream);
}
template int ek_suite_launch_hybrid<double>(const void*, const void*, const void*, const void*, const void*, int, int64_t, void* const*, uint32_t, int, void*);
template int ek_suite_launch_hybrid<float>(const void*, const void*, const void*, const void*, const void*, int, int64_t, void* const*, uint32_t, int, void*);
template <typename T>
int ek_suite_launch_hybrid_geo(const void* t, const void* q, const void* sp, const void* zs, const void* A, const void* B, int nlev, int64_t npl,
                               void* const* outs, uint32_t out_mask, int ept_method, int top_toa, double alpha_top, void* const* cols,
                               int height_mode, void* stream) {
    return suite_hybrid_geo<EK_OPS(OpSuiteTQPm), T>(t, q, sp, zs, A, B, nlev, npl, outs, out_mask, ept_method, nullptr, top_toa, alpha_top, cols[0],
                                                    cols[1], cols[2], height_mode, stream);
}
template int ek_suite_launch_hybrid_geo<double>(const void*, const void*, const void*, const void*, const void*, const void*, int, int64_t,
                                                void* const*, uint32_t, int, int, double, void* const*, int, void*);
template int ek_suite_launch_hybrid_geo<float>(const void*, const void*, const void*, const void*, const void*, const void*, int, int64_t,
                                               void* const*, uint32_t, int, int, double, void* const*, int, void*);
