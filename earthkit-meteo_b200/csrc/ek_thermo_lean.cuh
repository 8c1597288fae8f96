// ek_thermo_lean.cuh -- device-only math primitives sized for the instruction-issue budget of sm_100a.
//
// Why: with libdevice exp/log/pow and IEEE division the fused fp64 suite issues ~900 SASS instructions per
// grid point -- two thirds of them UMOV/IMAD.MOV pairs that materialise 64-bit polynomial coefficients as
// immediates -- and runs at 35 % of the HBM roofline, bound by instruction issue (profiles/r01_*).  These
// replacements keep every constant in constant memory / uniform registers (one DFMA per Horner step, no
// moves), use small shared-memory tables to shorten the polynomials, and drop work the path does not
// need (correct rounding of the quotient, denormal results):
//
//   rcp_/div_  MUFU.RCP64H seed (2^-19.9, measured: tools/probe_mufu.cu) + one cubic Newton step: <= 2 ulp
//   log_       2^10-entry {1/c, ln c} table, r = z/c - 1 (|r| < 2^-11), log1p polynomial of degree 4, k*ln2 added as a
//              hi/lo pair: ~1 ulp (abs 2e-16)
//   exp_       2^11-entry 2^(j/2^11) table, polynomial of degree 3 on |r| <= ln2/2^12: ~1 ulp
//   (the tables come from tools/gen_lean_tables.py: their 32 KB of shared memory per CTA buy two FP64 instructions per log_
//   and per exp_)
//   pow_       exp_(y * log_(x)): relative error ~ |y ln x| * 2e-16
//
// The constants whose low 32 bits are zero (+-0.5, -0.25, the 1.5*2^52 rounding constant) are written as literals: they
// become 32-bit immediates of DFMA / DADD instead of occupying uniform registers, and a polynomial step fma(r, c1, c0) no
// longer needs two constant operands (only one fits an instruction).
//
// The fp64 primitives are branch-free.  Outside their fast domain (x <= 0, denormal, inf, NaN for log_; |x| >= 708
// or NaN for exp_; b = 0, denormal, inf, NaN for rcp_) they answer NaN; the kernel recomputes any point whose
// result contains a NaN with the exact functor (cold path), so special values behave exactly as in the exact
// build.  float32 uses hardware-approximate division and logarithm (MUFU) and libdevice expf, which are short and
// handle special values themselves.
//
// The tables live in shared memory (filled once per CTA by lean::init_tables from ek_thermo_kernels.cuh):
// per-lane indexed reads from constant memory would serialise.
#pragma once
#include "ek_thermo_lean_tables.inc"

// the polynomial degrees of log_ and exp_ are chosen for these table sizes
static_assert(EK_LOG_TAB_BITS == 10 && EK_LOG_TAB_N == 1024 && EK_EXP_TAB_BITS == 11 && EK_EXP_TAB_N == 2048,
              "log_ / exp_ need 2^10-entry log and 2^11-entry exp tables");

namespace ek {
namespace lean {

struct Tables {
    double2 log_tab[EK_LOG_TAB_N];  // {invc, logc}
    double exp_tab[EK_EXP_TAB_N];   // 2^(j/N)
};

// polynomial coefficients: constant bank -> uniform registers, never immediates
__constant__ double kLog[5] = {-0.5, 0x1.5555555555555p-2 /*1/3*/, -0.25, 0x1.999999999999ap-3 /*1/5*/, -0x1.5555555555555p-3 /*-1/6*/};
__constant__ double kExp[4] = {0.5, 0x1.5555555555555p-3 /*1/6*/, 0x1.5555555555555p-5 /*1/24*/, 0x1.1111111111111p-7 /*1/120*/};
__constant__ double kRed[10] = {EK_INVLN2_N, EK_LN2N_HI, EK_LN2N_LO, EK_LN2_HI,   EK_LN2_LO, 0x1.8p52 /*magic*/,
                                EK_LOG_P0,   EK_LOG_T0DJ, 0x1.62e42fefa39efp-1 /*ln 2*/, 0.285691 * EK_LOG_P0 /*kappa ln p0*/};

__device__ __forceinline__ Tables* tables() {
    extern __shared__ __align__(16) unsigned char ek_smem_raw[];
    return reinterpret_cast<Tables*>(ek_smem_raw);
}
// Table reads go through explicit shared-state-space loads on a 32-bit address: with generic pointers the
// compiler re-derives the shared window base (S2UR CgaCtaId + ULEA) at every access.
__device__ __forceinline__ uint32_t tab_base() { return static_cast<uint32_t>(__cvta_generic_to_shared(tables())); }
__device__ __forceinline__ double2 lds_log(int i) {
    double2 v;
    asm("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(tab_base() + 16u * (uint32_t)i));
    return v;
}
__device__ __forceinline__ double lds_exp(int j) {
    double v;
    asm("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(tab_base() + (uint32_t)(16 * EK_LOG_TAB_N) + 8u * (uint32_t)j));
    return v;
}

__device__ __forceinline__ void init_tables() {
    // 16-byte copies global (L2-resident after the first CTA) -> shared
    double2* dst = reinterpret_cast<double2*>(tables());
    const double2* lg = reinterpret_cast<const double2*>(ek_log_tab_g);
    const double2* ex = reinterpret_cast<const double2*>(ek_exp_tab_g);
    for (int i = threadIdx.x; i < EK_LOG_TAB_N; i += blockDim.x) dst[i] = __ldg(lg + i);
    for (int i = threadIdx.x; i < EK_EXP_TAB_N / 2; i += blockDim.x) dst[EK_LOG_TAB_N + i] = __ldg(ex + i);
    __syncthreads();
}

// ---- float64 ------------------------------------------------------------------------------------------
__device__ __forceinline__ double rcp_(double b) {
    double r0;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r0) : "d"(b));
    const double e = fma(-b, r0, 1.0);
    return fma(fma(e, e, e), r0, r0);  // b = 0, denormal, inf, NaN: e is NaN -> NaN (the point is recomputed exactly)
}
__device__ __forceinline__ double div_(double a, double b) { return a * rcp_(b); }
// Loop-invariant values the compiler would rather recompute inside a loop than keep live (it rematerialises cheap
// expressions under register pressure): an empty asm makes the value opaque, so it is computed once.
__device__ __forceinline__ double keep_in_register(double x) {
    asm volatile("" : "+d"(x));
    return x;
}
__device__ __forceinline__ float keep_in_register(float x) {
    asm volatile("" : "+f"(x));
    return x;
}
// 1/b to 2^-39 (seed + one quadratic step): for callers that only need the sign of a difference and treat a
// near-tie as "recompute exactly" (the tabulated bisection)
__device__ __forceinline__ double rcp_sign_(double b) {
    double r0;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r0) : "d"(b));
    return fma(r0, fma(-b, r0, 1.0), r0);
}

__device__ __forceinline__ double log_(double x) {
    const int hi = __double2hiint(x);
    const bool bad = (unsigned)(hi - 0x00100000) >= 0x7fe00000u;  // <= 0, denormal, inf, NaN: answer NaN
    const int tmp = hi - 0x3fe60000;
    const int i = (tmp >> (20 - EK_LOG_TAB_BITS)) & (EK_LOG_TAB_N - 1);
    const int k = tmp >> 20;
    const double z = __hiloint2double(hi - (tmp & 0xfff00000), __double2loint(x));
    const double2 tc = lds_log(i);
    const double r = fma(z, tc.x, -1.0);
    const double kd = (double)k;
    const double r2 = r * r;
    // log1p(r) = r + r^2 s(r), s = -1/2 + r/3 - r^2/4 (Estrin: short dependency chains)
    const double s = fma(r2, -0.25, fma(r, kLog[1], -0.5));
    // k*ln2 as a hi/lo pair (abs error ~2e-16); one FMA with ln2 is ~1.5 ulp of the result and measured within noise on B200
    // (ept + wet bulb +3 %, suites -1.5 %)
    const double t1 = fma(kd, kRed[3], tc.y);
    const double t2 = fma(kd, kRed[4], r);
    const double y = fma(r2, s, t2) + t1;
    return __hiloint2double(bad ? 0x7ff80000 : __double2hiint(y), __double2loint(y));
}

__device__ __forceinline__ double exp_(double x) {
    const bool bad = (unsigned)(__double2hiint(x) & 0x7fffffff) >= 0x40862000u;  // |x| >= 708, inf, NaN: answer NaN
    const double t = fma(x, kRed[0], 0x1.8p52);
    const int ki = __double2loint(t);
    const double kd = t - 0x1.8p52;
    double r = fma(kd, -kRed[1], x);
    r = fma(kd, -kRed[2], r);
    const double T = lds_exp(ki & (EK_EXP_TAB_N - 1));
    const double r2 = r * r;
    // e^r - 1 = r + r^2 s(r), s = 1/2 + r/6
    const double s = fma(r, kExp[1], 0.5);
    const double p = fma(r2, s, r);
    const double y = fma(T, p, T);
    return __hiloint2double(bad ? 0x7ff80000 : __double2hiint(y) + ((ki >> EK_EXP_TAB_BITS) << 20), __double2loint(y));
}

__device__ __forceinline__ double pow_(double x, double y) { return exp_(y * log_(x)); }
// pow(p0/x, y), pow(x/p0, y), pow(273.16/x, y): the logarithm of the constant is tabulated, no division
__device__ __forceinline__ double pow_p0_over_(double x, double y) { return exp_(y * (kRed[6] - log_(x))); }
__device__ __forceinline__ double pow_over_p0_(double x, double y) { return exp_(y * (log_(x) - kRed[6])); }
__device__ __forceinline__ double pow_t0_over_(double x, double y) { return exp_(y * (kRed[7] - log_(x))); }

// ln(p0 / x) without the division
__device__ __forceinline__ double log_p0_over(double x);
__device__ __forceinline__ float log_p0_over(float x) { return (float)EK_LOG_P0 - __logf(x); }

// kappa * ln(p0 / x): the exponent of the Exner factor, for callers that fold it into a larger exponential
__device__ __forceinline__ double kappa_log_p0_over(double x) { return fma(-::ek::kCdev.kappa, log_(x), kRed[9]); }  // kRed[9] = kappa ln p0
__device__ __forceinline__ float kappa_log_p0_over(float x) { return (float)::ek::kC.kappa * ((float)EK_LOG_P0 - __logf(x)); }

__device__ __forceinline__ double log_p0_over(double x) { return kRed[6] - log_(x); }

// ---- sin / cos / atan2 for the wind functions (SURVEY.md 8(f)-3) ---------------------------------------------------------
// Same contract as the primitives above: branch-free, ~1 ulp inside a fast domain, NaN outside it (the kernel then recomputes the
// point with libdevice).  sincos_: |x| < 2^19, three-part Cody-Waite reduction by pi/2 (33 + 33 + 33 bits: exact products for
// |k| < 2^20) and the fdlibm kernel polynomials.  atan2_: both arguments finite, normal and non-zero; atan on [0, 1] by fdlibm's
// two break points (7/16, 11/16) and its degree-11 polynomial in w^2: two reciprocals and 11 FMAs instead of libdevice's ~100
// instructions (the 24 B/pt direction kernel was issue-bound at 0.75 of the roofline).
__constant__ double kTrig[22] = {
    6.36619772367581382433e-01 /*2/pi*/, 1.57079632673412561417e+00 /*pio2_1*/, 6.07710050630396597660e-11 /*pio2_2*/, 2.02226624871116645580e-21 /*pio2_3*/,
    -1.66666666666666324348e-01, 8.33333333332248946124e-03, -1.98412698298579493134e-04, 2.75573137070700676789e-06, -2.50507602534068634195e-08,
    1.58969099521155010221e-10,  // S1..S6 (indices 4..9)
    4.16666666666666019037e-02, -1.38888888888741095749e-03, 2.48015872894767294178e-05, -2.75573143513906633035e-07, 2.08757232129817482790e-09,
    -1.13596475577881948265e-11,  // C1..C6 (10..15)
    4.63647609000806093515e-01 /*atan(1/2) hi*/, 2.26987774529616870924e-17 /*lo*/, 7.85398163397448278999e-01 /*pi/4 hi*/, 3.06161699786838301793e-17 /*lo*/,
    1.57079632679489655800e+00 /*pi/2 hi*/, 6.12323399573676603587e-17 /*lo*/};
__constant__ double kAtan[11] = {3.33333333333329318027e-01,  -1.99999999998764832476e-01, 1.42857142725034663711e-01,  -1.11111104054623557880e-01,
                                 9.09088713343650656196e-02,  -7.69187620504482999495e-02, 6.66107313738753120669e-02,  -5.83357013379057348645e-02,
                                 4.97687799461593236017e-02,  -3.65315727442169155270e-02, 1.62858201153657823623e-02};

__device__ __forceinline__ void sincos_(double x, double& s, double& c) {
    const bool bad = (unsigned)(__double2hiint(x) & 0x7fffffff) >= 0x41200000u;  // |x| >= 2^19, inf, NaN: answer NaN
    const double t = fma(x, kTrig[0], 0x1.8p52);
    const int q = __double2loint(t);
    const double kd = t - 0x1.8p52;
    double r = fma(kd, -kTrig[1], x);
    r = fma(kd, -kTrig[2], r);
    r = fma(kd, -kTrig[3], r);
    const double r2 = r * r;
    double ps = fma(r2, kTrig[9], kTrig[8]);
    ps = fma(r2, ps, kTrig[7]);
    ps = fma(r2, ps, kTrig[6]);
    ps = fma(r2, ps, kTrig[5]);
    ps = fma(r2, ps, kTrig[4]);
    const double sn = fma(r * r2, ps, r);
    double pc = fma(r2, kTrig[15], kTrig[14]);
    pc = fma(r2, pc, kTrig[13]);
    pc = fma(r2, pc, kTrig[12]);
    pc = fma(r2, pc, kTrig[11]);
    pc = fma(r2, pc, kTrig[10]);
    const double cs = fma(r2 * r2, pc, fma(r2, -0.5, 1.0));
    const double a = (q & 1) ? cs : sn, b = (q & 1) ? sn : cs;
    const double nan = __hiloint2double(0x7ff80000, 0);
    s = bad ? nan : ((q & 2) ? -a : a);
    c = bad ? nan : (((q + 1) & 2) ? -b : b);
}
__device__ __forceinline__ double sin_(double x) {
    double s, c;
    sincos_(x, s, c);
    return s;
}

__device__ __forceinline__ double atan2_(double y, double x) {
    const int hx = __double2hiint(x) & 0x7fffffff, hy = __double2hiint(y) & 0x7fffffff;
    // zero, denormal, tiny, huge, inf, NaN in either argument: answer NaN (2^-1007 <= |.| < 2^1009 is the fast domain)
    const bool bad = (unsigned)(hx - 0x01000000) >= 0x7e000000u || (unsigned)(hy - 0x01000000) >= 0x7e000000u;
    const double ax = fabs(x), ay = fabs(y);
    const bool swap = ay > ax;
    const double mx = swap ? ay : ax, mn = swap ? ax : ay;
    const double z = mn * rcp_(mx);  // in [0, 1]
    // z >= 7/16: atan(z) = pi/4 + atan((z - 1) / (z + 1)), |w| <= 0.392 on [7/16, 1]: inside the range of fdlibm's polynomial
    // (|w| < 7/16), so its second break point (11/16, with atan(1/2)) is not needed on [0, 1]
    const bool m = z >= 0.4375;
    const double num = m ? z - 1.0 : z;
    const double den = m ? z + 1.0 : 1.0;
    const double w = num * rcp_(den);
    const double hi = m ? kTrig[18] : 0.0, lo = m ? kTrig[19] : 0.0;
    const double w2 = w * w, w4 = w2 * w2;
    double s1 = fma(w4, kAtan[10], kAtan[8]);
    s1 = fma(w4, s1, kAtan[6]);
    s1 = fma(w4, s1, kAtan[4]);
    s1 = fma(w4, s1, kAtan[2]);
    s1 = fma(w4, s1, kAtan[0]);
    double s2 = fma(w4, kAtan[9], kAtan[7]);
    s2 = fma(w4, s2, kAtan[5]);
    s2 = fma(w4, s2, kAtan[3]);
    s2 = fma(w4, s2, kAtan[1]);
    const double p = fma(w2, s1, w4 * s2);           // w^2 s1 + w^4 s2
    double r = hi - ((fma(w, p, -lo)) - w);          // atan(z) in [0, pi/4]
    if (swap) r = (kTrig[20] - r) + kTrig[21];       // |y| > |x|: pi/2 - atan(|x|/|y|)
    if (__double2hiint(x) < 0) r = (2.0 * kTrig[20] - r) + 2.0 * kTrig[21];  // x < 0: pi - r
    r = __hiloint2double(__double2hiint(r) | (__double2hiint(y) & 0x80000000), __double2loint(r));  // the sign of y
    return bad ? __hiloint2double(0x7ff80000, 0) : r;
}

// ---- bisection tree table (see t_on_ma_bisect_tab in ek_thermo_formulas.inc) -----------------------------------
// The reference's moist-adiabat bisection (T:1055-1079) starts every point at T0 - 20 and moves by +-60, +-30, ... K:
// after i steps the iterate is one of 2^i values that do not depend on the data.  {es_mixed(t), ln t} of the 4095
// nodes visited by the 12 steps are tabulated once per launch (bisect_tab_init_kernel), which removes the exponential,
// the phase blend and two reciprocals from every iteration.  Heap numbering: root = 1, children 2n (down), 2n + 1 (up).
#define EK_BISECT_NODES 4096
static __device__ double2 ek_bisect_tab[EK_BISECT_NODES];
static __device__ float2 ek_bisect_tab_f[EK_BISECT_NODES];  // float32 twin: nodes, es and ln t in float32 arithmetic

// ---- float32 ------------------------------------------------------------------------------------------
__device__ __forceinline__ float div_(float a, float b) { return __fdividef(a, b); }
__device__ __forceinline__ float rcp_sign_(float b) { return __fdividef(1.0f, b); }
// 1/b in the dtype's lean flavour, for formulas that fold the quotient into an FMA
__device__ __forceinline__ double rcp_any(double b) { return rcp_(b); }
__device__ __forceinline__ float rcp_any(float b) { return __fdividef(1.0f, b); }
// MUFU.LG2-based: absolute error ~1e-6 on |ln x| <= 12 -- after the factors it meets on this path (kappa = 0.29 in the
// Exner exponent, d(td)/d(ln e) ~ 14 K) that is <= 7e-7 relative, inside the float32 bar of 1e-5; 3 instructions vs 24
__device__ __forceinline__ float log_(float x) { return __logf(x); }
__device__ __forceinline__ float exp_(float x) { return ::expf(x); }
__device__ __forceinline__ float pow_(float x, float y) { return ::expf(y * __logf(x)); }
__device__ __forceinline__ float pow_p0_over_(float x, float y) { return ::expf(y * ((float)EK_LOG_P0 - __logf(x))); }
__device__ __forceinline__ float pow_over_p0_(float x, float y) { return ::expf(y * (__logf(x) - (float)EK_LOG_P0)); }
__device__ __forceinline__ float pow_t0_over_(float x, float y) { return ::expf(y * ((float)EK_LOG_T0DJ - __logf(x))); }

}  // namespace lean
}  // namespace ek
