// ek_thermo_math.cuh -- per-point thermodynamic formulas of the earthkit-meteo thermo hot path,
// written as templated __host__ __device__ functions over T in {double, float}.
//
// Reference citations: T = src/earthkit/meteo/thermo/array/thermo.py, E = .../array/es_comp.py,
// C = src/earthkit/meteo/constants/constants.py (all in the reference tree).  The formulas keep the
// reference's operation order; constants are the reference's literals (C:22-50, E:14-20) and the
// derived ones are evaluated in double exactly as Python evaluates them, then rounded to T once
// (which is what NumPy-2 weak-scalar promotion does for float32 arrays).
//
// Everything a thread needs lives in registers: the reference's _ThermoState scratch object
// (T:1003-1017) becomes local variables here.
//
// Two build modes (same formulas, same operation order):
//   EK_LEAN_MATH=0  libdevice exp/log/pow, IEEE division, constants as immediates ("exact" build; also
//                   what the host check harness tests/_hostmath compiles with std:: math);
//   EK_LEAN_MATH=1  device code takes its 64-bit constants from constant memory (CK(), one uniform-register
//                   operand instead of two move instructions per use), and exp/log/pow/division from
//                   ek_thermo_lean.cuh.  Division by a constant becomes multiplication by its reciprocal.
//                   The lean primitives are branch-free and answer NaN outside their fast domain; a point
//                   whose result contains a NaN is recomputed by the exact functor (kernel, cold path), so
//                   special values behave exactly as in the exact build.  In-domain results move by a few
//                   ulp; every parity bound of tests/ holds in both modes.
#pragma once
#include <cmath>
#include <cstdint>
#include <limits>

#if defined(__CUDACC__)
#define EK_HD __host__ __device__ __forceinline__
#else
#define EK_HD inline
#endif

#ifndef EK_LEAN_MATH
#define EK_LEAN_MATH 0
#endif

#if EK_LEAN_MATH && defined(__CUDA_ARCH__)
#define EK_LEAN_DEVICE 1
#else
#define EK_LEAN_DEVICE 0
#endif

namespace ek {

// ------------------------------------------------------------------------------------------
// constants: the reference's literals and the double expressions Python evaluates from them
// ------------------------------------------------------------------------------------------
struct Consts {
    double Rd, Rv_m_Rd, kappa, lambda, p0, inv_p0, eps, c_vp, c1_tv, eps_m1, T0, TI;
    double C1, inv_C1, C3W, C4W, C3I, C4I, slope_w, slope_i, band, inv_band, d_alpha_c, C3W_T0;
    double K0_ifs, neg_K0_ifs, neg_lam_K0_ifs;
    double dj_a, dj_b, dj_c, dj_a0;               // Davies-Jones lcl fit (T:961); dj_a0 = dj_a - (dj_b - dj_c) T0
    double b35_K3, neg_lam_b35_K0;               // T:1202-1203
    double b39_K1, b39_K2, b39_K4, b39_2K2, neg_b39_K1, neg_lam_b39_K0, neg_lam_b39_K1;  // T:1263-1266
    double wa0, wa1, wa2, wa3, wa4, wb1, wb2, wb3, wb4, inv_t0;  // wbpt "direct" rational fit (T:1051-1052)
    double wsa1, wsa2, wsa3, wsa4, wsb1, wsb2, wsb3, wsb4;       // the same coefficients divided by 273.16^k (lean build: Horner in ept itself)
    double td_K;                                                 // C3W (C4W - T0): t_from_es as C4W + td_K / (v - C3W) (lean build)
    double k10, k11, k12, k20, k21, k22, dD1, dD0, c121, c266, c058, c04;  // Davies-Jones first guess (T:1090-1128)
    double t_start, eps_default, neg_lambda, hundred, hundredth, c800, inv_800;
    double bis_c_ifs, bis_tie, bis_plim_scale;  // lean bisection (ek_thermo_formulas.inc: t_on_ma_bisect_tab_n)
    double g, inv_g, R_earth;  // constants.py:53,57 (height conversions, vertical.py:330-502)
    double degree, radian, two_omega, neg_Rd_g, minus_pi2, pi15;  // wind (constants.py:60-78, wind/array/wind.py)
};

namespace cdef {
constexpr double Rd = 287.0597, Rv = 461.51, c_pd = 1004.79, Lv = 2.5008e6;  // C:22,26,30,38
constexpr double kappa = 0.285691, p0 = 1e5, eps = 0.621981, T0 = 273.16;    // C:41,44,47,50
constexpr double C1 = 611.21, C3W = 17.502, C4W = 32.19, C3I = 22.587, C4I = -0.7;  // E:14-18
constexpr double TI = T0 - 23;                                              // E:20
constexpr double lambda = 1.0 / kappa;                                      // T:1022
constexpr double K0_ifs = Lv / c_pd;                                        // T:1164
constexpr double band = T0 - TI;                                            // E:164
}  // namespace cdef

constexpr Consts make_consts() {
    Consts k{};
    k.Rd = cdef::Rd;
    k.Rv_m_Rd = cdef::Rv - cdef::Rd;  // T:1706
    k.kappa = cdef::kappa;
    k.lambda = cdef::lambda;
    k.p0 = cdef::p0;
    k.inv_p0 = 1.0 / cdef::p0;
    k.eps = cdef::eps;
    k.c_vp = cdef::eps * (1.0 / cdef::eps - 1.0);  // T:130
    k.c1_tv = (1.0 - cdef::eps) / cdef::eps;       // T:763
    k.eps_m1 = cdef::eps - 1;                      // T:193, T:465
    k.T0 = cdef::T0;
    k.TI = cdef::TI;
    k.C1 = cdef::C1;
    k.inv_C1 = 1.0 / cdef::C1;
    k.C3W = cdef::C3W;
    k.C4W = cdef::C4W;
    k.C3I = cdef::C3I;
    k.C4I = cdef::C4I;
    k.slope_w = cdef::C3W * (cdef::T0 - cdef::C4W);  // E:170
    k.slope_i = cdef::C3I * (cdef::T0 - cdef::C4I);  // E:174
    k.band = cdef::band;                             // E:164
    k.inv_band = 1.0 / cdef::band;
    k.d_alpha_c = 2.0 / (cdef::band * cdef::band);   // E:192
    k.C3W_T0 = cdef::C3W * cdef::T0;                 // E:130
    k.K0_ifs = cdef::K0_ifs;
    k.neg_K0_ifs = -1.0 * cdef::K0_ifs;              // scale = -1.0 (T:1075, T:1182)
    k.neg_lam_K0_ifs = -cdef::lambda * cdef::K0_ifs;  // scale = -c_lambda (T:1194)
    k.dj_a = 0.212;
    k.dj_b = 1.571e-3;
    k.dj_c = 4.36e-4;
    k.dj_a0 = 0.212 - (1.571e-3 - 4.36e-4) * cdef::T0;
    k.b35_K3 = 0.28;
    k.neg_lam_b35_K0 = -cdef::lambda * 2675.0;
    k.b39_K1 = 1.78;
    k.b39_K2 = 0.448;
    k.b39_K4 = 0.28;
    k.b39_2K2 = 2 * 0.448;
    k.neg_b39_K1 = -1.0 * 1.78;
    k.neg_lam_b39_K0 = -cdef::lambda * 3036.0;
    k.neg_lam_b39_K1 = -cdef::lambda * 1.78;
    k.wa0 = 7.101574;
    k.wa1 = -20.68208;
    k.wa2 = 16.11182;
    k.wa3 = 2.574631;
    k.wa4 = -5.205688;
    k.wb1 = -3.552497;
    k.wb2 = 3.781782;
    k.wb3 = -0.6899655;
    k.wb4 = -0.5929340;
    k.inv_t0 = 1.0 / 273.16;
    {
        constexpr double t1 = 273.16, t2 = t1 * t1, t3 = t2 * t1, t4 = t2 * t2;
        k.wsa1 = -20.68208 / t1;
        k.wsa2 = 16.11182 / t2;
        k.wsa3 = 2.574631 / t3;
        k.wsa4 = -5.205688 / t4;
        k.wsb1 = -3.552497 / t1;
        k.wsb2 = 3.781782 / t2;
        k.wsb3 = -0.6899655 / t3;
        k.wsb4 = -0.5929340 / t4;
    }
    k.td_K = cdef::C3W * (cdef::C4W - cdef::T0);
    k.k10 = -53.737;
    k.k11 = 137.81;
    k.k12 = -38.5;
    k.k20 = -0.384;
    k.k21 = 56.831;
    k.k22 = -4.392;
    k.dD1 = 0.1859e-5;
    k.dD0 = 0.6512;
    k.c121 = 1.21;
    k.c266 = 2.66;
    k.c058 = 0.58;
    k.c04 = 0.4;
    k.t_start = cdef::T0 - 20;  // T:1061
    k.eps_default = 1e-4;
    k.bis_c_ifs = (-1.0 * cdef::K0_ifs) * cdef::eps;  // G = bis_c_ifs * es / (v t)
    k.bis_tie = 1e-10;
    k.bis_plim_scale = 1.0 - 1e-9;
    k.neg_lambda = -cdef::lambda;
    k.hundred = 100.0;
    k.hundredth = 0.01;
    k.c800 = 800.0;
    k.inv_800 = 1.0 / 800.0;
    k.g = 9.80665;
    k.inv_g = 1.0 / 9.80665;
    k.R_earth = 6371229.0;
    // constants.py:60-78, evaluated in the order Python evaluates them
    constexpr double pi = 3.141592653589793;  // numpy.pi
    constexpr double solar_day = 86400;
    constexpr double sideral_year = 365.25 * solar_day * 2 * pi / 6.283076;
    constexpr double sideral_day = solar_day / (1.0 + solar_day / sideral_year);
    constexpr double omega = 2.0 * pi / sideral_day;
    k.degree = 180.0 / pi;
    k.radian = 1.0 / (180.0 / pi);
    k.two_omega = 2 * omega;                      // wind.py:251
    k.neg_Rd_g = -cdef::Rd / 9.80665;             // wind.py:222
    k.minus_pi2 = -pi / 2.0;                      // wind.py:42
    k.pi15 = 1.5 * pi;                            // wind.py:48
    return k;
}

constexpr Consts kC = make_consts();
#if defined(__CUDACC__)
__constant__ Consts kCdev = make_consts();
#endif

enum Phase : int { PHASE_MIXED = 0, PHASE_WATER = 1, PHASE_ICE = 2 };
enum LclMethod : int { LCL_DAVIES = 0, LCL_BOLTON = 1 };
enum EptMethod : int { EPT_IFS = 0, EPT_BOLTON35 = 1, EPT_BOLTON39 = 2 };
enum TMethod : int { TM_NONE = 0, TM_DIRECT = 1, TM_BISECT = 2, TM_NEWTON = 3 };

// ------------------------------------------------------------------------------------------
// math primitives: libdevice / libm ("exact")
// ------------------------------------------------------------------------------------------
EK_HD double m_exp_exact(double x) { return ::exp(x); }
EK_HD float m_exp_exact(float x) { return ::expf(x); }
EK_HD double m_log_exact(double x) { return ::log(x); }
EK_HD float m_log_exact(float x) { return ::logf(x); }
EK_HD double m_pow_exact(double x, double y) { return ::pow(x, y); }
EK_HD float m_pow_exact(float x, float y) { return ::powf(x, y); }

EK_HD double m_hypot(double x, double y) { return ::hypot(x, y); }
EK_HD float m_hypot(float x, float y) { return ::hypotf(x, y); }
EK_HD double m_atan2(double y, double x) { return ::atan2(y, x); }
EK_HD float m_atan2(float y, float x) { return ::atan2f(y, x); }
EK_HD double m_sin(double x) { return ::sin(x); }
EK_HD float m_sin(float x) { return ::sinf(x); }
EK_HD double m_cos(double x) { return ::cos(x); }
EK_HD float m_cos(float x) { return ::cosf(x); }

template <typename T> EK_HD T m_nan() { return static_cast<T>(NAN); }
template <typename T> EK_HD T sq(T x) { return x * x; }
// numpy.sign: -1, 0, +1, NaN for NaN (T:1075 relies on the NaN case to poison the iterate)
template <typename T> EK_HD T m_sign(T x) { return (x > T(0)) ? T(1) : ((x < T(0)) ? T(-1) : ((x == T(0)) ? T(0) : x)); }

// Per-launch options, passed by value to the kernel (uniform across the grid).
struct Params {
    int opt0 = 0;           // phase | lcl method | humidity kind (0 = dewpoint, 1 = specific humidity)
    int opt1 = 0;           // flags: bit0 "es given", bit1 "es_slope given" | wet-bulb level (0 = at p, 1 = at p0)
    double eps = 1e-4;      // the eps argument of the NaN rule (T:162,199,367,418)
    uint32_t out_mask = 1;  // which outputs are wanted (bit k = output k)
};

// output slots of the fused suites (see ek_thermo_ops.inc)
enum SuiteSlot : int { S_THETA = 0, S_ES = 1, S_RH = 2, S_TDQ = 3, S_TV = 4, S_W = 5, S_E = 6, S_THETAV = 7, S_EPT = 8, S_WBPT = 9, S_NSLOTS = 10 };

}  // namespace ek

#if EK_LEAN_MATH && defined(__CUDACC__)
#include "ek_thermo_lean.cuh"  // both compilation passes must see its __constant__ / __device__ tables
#endif

// ------------------------------------------------------------------------------------------
// The formulas (ek_thermo_formulas.inc) and the kernel functors (ek_thermo_ops.inc) are compiled once per
// math mode, each in its own namespace:
//   ek::exactm  libdevice exp/log/pow, IEEE division, constants as immediates.  The whole product in an
//               EK_LEAN_MATH=0 build, the host check harness, and the cold "recompute this point" path of a
//               lean build.
//   ek::fastm   (device code of an EK_LEAN_MATH=1 build only) lean primitives, constants from the constant bank.
// ------------------------------------------------------------------------------------------
#define EK_INC_LEAN 0
#define EK_MODE_NS exactm
#include "ek_thermo_formulas.inc"
#include "ek_thermo_ops.inc"
#undef EK_INC_LEAN
#undef EK_MODE_NS

#if EK_LEAN_MATH && defined(__CUDACC__)
#define EK_INC_LEAN 1
#define EK_MODE_NS fastm
#include "ek_thermo_formulas.inc"
#include "ek_thermo_ops.inc"
#undef EK_INC_LEAN
#undef EK_MODE_NS
#define EK_OPS(...) ::ek::fastm::__VA_ARGS__, ::ek::exactm::__VA_ARGS__
#else
#define EK_OPS(...) ::ek::exactm::__VA_ARGS__, ::ek::exactm::__VA_ARGS__
#endif
