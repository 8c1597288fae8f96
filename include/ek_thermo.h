/* ek_thermo.h -- C ABI of libek_thermo.so: B200 (sm_100a) kernels for the earthkit-meteo thermo hot path.
 *
 * The reference (ecmwf/earthkit-meteo) has no FFI: its boundary for this path is the Python function
 * namespace earthkit.meteo.thermo.array.* (src/earthkit/meteo/thermo/array/thermo.py = "T" below,
 * es_comp.py = "E").  Each entry point here replaces the body of one of those functions for device
 * arrays; the Python drop-in (earthkit-meteo_b200/ek_thermo/thermo.py) binds them with ctypes and keeps
 * the reference's names, argument order, defaults and exceptions.  INTEGRATION.md shows the stub a
 * maintainer of the reference would add.
 *
 * Conventions (all entry points):
 *  - every array argument is a DEVICE pointer to n contiguous elements of the function's dtype
 *    (suffix _f64 = double, _f32 = float); only natural alignment is required (16-byte aligned
 *    pointers take the 128-bit load/store path, others a scalar path inside the same kernel);
 *  - an input may instead be a broadcast scalar: ek_operand{NULL, value};
 *  - the caller allocates and owns every buffer; the library never allocates, frees or synchronises;
 *  - the launch is asynchronous on `stream` (a cudaStream_t / CUstream, NULL = default stream) of the
 *    CURRENT device; the caller selects the device;
 *  - return 0 on success, a positive cudaError_t if the launch failed, or a negative EK_ERR_* code for
 *    argument errors (ek_thermo_last_error() gives the text, thread-local);
 *  - numerical failures are in-band NaN, exactly where the reference produces NaN;
 *  - thread-safe and re-entrant; no CPU fallback exists anywhere in the library.
 */
#ifndef EK_THERMO_H
#define EK_THERMO_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EK_THERMO_VERSION 112 /* 0.1.2: the hybrid-level suite with geopotential / height of the same levels in one pass
                                  (suite_tq_hybrid_geo, host_suite_tq_hybrid_geo).  0.1.1: suite slots 8 (ept) / 9 (wbpt) and their
                                  ept_method argument; host pipelines for every suite; batched suites with one pressure per level */

typedef struct ek_operand {
    const void* ptr; /* device pointer, or NULL for a broadcast scalar */
    double value;    /* the scalar when ptr == NULL (rounded to the dtype once, as numpy does) */
} ek_operand;

enum { EK_OK = 0, EK_ERR_ARG = -1, EK_ERR_ENUM = -2, EK_ERR_EPS = -3, EK_ERR_PIPE = -4 };

/* option enums (strings of the reference API -> ints) */
enum { EK_PHASE_MIXED = 0, EK_PHASE_WATER = 1, EK_PHASE_ICE = 2 };            /* E:22 */
enum { EK_LCL_DAVIES = 0, EK_LCL_BOLTON = 1 };                                /* T:960-968 */
enum { EK_EPT_IFS = 0, EK_EPT_BOLTON35 = 1, EK_EPT_BOLTON39 = 2 };            /* T:1319-1323 */
enum { EK_TM_NONE = 0, EK_TM_DIRECT = 1, EK_TM_BISECT = 2, EK_TM_NEWTON = 3 }; /* T:1504-1509, T:1631 */
enum { EK_HUM_DEWPOINT = 0, EK_HUM_SPECIFIC = 1 };

/* output slots of the fused suites (bit k of out_mask <-> outs[k]) */
enum {
    EK_S_THETA = 0, EK_S_ES = 1, EK_S_RH = 2, EK_S_TD_OR_Q = 3, EK_S_TV = 4, EK_S_W = 5, EK_S_E = 6, EK_S_THETAV = 7,
    EK_S_EPT = 8,  /* ept_from_specific_humidity / ept_from_dewpoint, T:1390-1415 / T:1326-1387 */
    EK_S_WBPT = 9, /* wet_bulb_potential_temperature_from_*, t_method="direct" (the reference's default), T:1637-1675 / T:1593-1634 */
    EK_S_NSLOTS = 10
};

/* declares ek_thermo_<name>_f64 and ek_thermo_<name>_f32 with the same parameter list */
#define EK_THERMO_FN(name, ...)              \
    int ek_thermo_##name##_f64(__VA_ARGS__); \
    int ek_thermo_##name##_f32(__VA_ARGS__);

/* ---- library ------------------------------------------------------------------------------- */
int ek_thermo_version(void);
const char* ek_thermo_last_error(void);
/* threads per CTA (multiple of 32, <= 1024) and CTAs per SM used to size grids; 0 keeps the default */
int ek_thermo_set_launch_config(int threads, int ctas_per_sm);
/* number of kernels this library has launched since load (all threads) */
uint64_t ek_thermo_launch_count(void);
/* field partitioner: contiguous shard [begin,end) of rank `rank` of `world` over n points, edges
 * aligned to `align` points (SURVEY.md §8(e)); returns EK_ERR_ARG on bad arguments */
int ek_thermo_shard_range(int64_t n, int world, int rank, int64_t align, int64_t* begin, int64_t* end);

/* ---- simple conversions ---------------------------------------------------------------------- */
EK_THERMO_FN(celsius_to_kelvin, ek_operand t, void* out, int64_t n, void* stream)                    /* T:21-35 */
EK_THERMO_FN(kelvin_to_celsius, ek_operand t, void* out, int64_t n, void* stream)                    /* T:38-52 */
EK_THERMO_FN(specific_humidity_from_mixing_ratio, ek_operand w, void* out, int64_t n, void* stream)  /* T:55-77 */
EK_THERMO_FN(mixing_ratio_from_specific_humidity, ek_operand q, void* out, int64_t n, void* stream)  /* T:80-102 */
EK_THERMO_FN(vapour_pressure_from_specific_humidity, ek_operand q, ek_operand p, void* out, int64_t n, void* stream) /* T:105-131 */
EK_THERMO_FN(vapour_pressure_from_mixing_ratio, ek_operand w, ek_operand p, void* out, int64_t n, void* stream)      /* T:134-159 */
/* eps <= 0 -> EK_ERR_EPS (reference: ValueError, T:189-190 / T:226-227) */
EK_THERMO_FN(specific_humidity_from_vapour_pressure, ek_operand e, ek_operand p, double eps, void* out, int64_t n, void* stream) /* T:162-196 */
EK_THERMO_FN(mixing_ratio_from_vapour_pressure, ek_operand e, ek_operand p, double eps, void* out, int64_t n, void* stream)      /* T:199-232 */

/* ---- saturation vapour pressure and friends -------------------------------------------------- */
EK_THERMO_FN(saturation_vapour_pressure, ek_operand t, int phase, void* out, int64_t n, void* stream)                 /* T:235-279, E:31-79 */
EK_THERMO_FN(saturation_vapour_pressure_slope, ek_operand t, int phase, void* out, int64_t n, void* stream)           /* T:344-364, E:82-106 */
EK_THERMO_FN(saturation_mixing_ratio, ek_operand t, ek_operand p, int phase, void* out, int64_t n, void* stream)      /* T:282-310 */
EK_THERMO_FN(saturation_specific_humidity, ek_operand t, ek_operand p, int phase, void* out, int64_t n, void* stream) /* T:313-341 */
/* es / es_slope are optional precomputed inputs: pass has_es / has_es_slope = 0 to have them computed (T:407-410) */
EK_THERMO_FN(saturation_mixing_ratio_slope, ek_operand t, ek_operand p, ek_operand es, ek_operand es_slope, int has_es,
             int has_es_slope, int phase, double eps, void* out, int64_t n, void* stream)                             /* T:367-415 */
EK_THERMO_FN(saturation_specific_humidity_slope, ek_operand t, ek_operand p, ek_operand es, ek_operand es_slope, int has_es,
             int has_es_slope, int phase, double eps, void* out, int64_t n, void* stream)                             /* T:418-467 */
EK_THERMO_FN(temperature_from_saturation_vapour_pressure, ek_operand es, void* out, int64_t n, void* stream)          /* T:470-491, E:109-130 */

/* ---- humidity / dewpoint conversions ---------------------------------------------------------- */
EK_THERMO_FN(relative_humidity_from_dewpoint, ek_operand t, ek_operand td, void* out, int64_t n, void* stream)                     /* T:494-521 */
EK_THERMO_FN(relative_humidity_from_specific_humidity, ek_operand t, ek_operand q, ek_operand p, void* out, int64_t n, void* stream) /* T:524-556 */
EK_THERMO_FN(specific_humidity_from_dewpoint, ek_operand td, ek_operand p, void* out, int64_t n, void* stream)                     /* T:559-591 */
EK_THERMO_FN(mixing_ratio_from_dewpoint, ek_operand td, ek_operand p, void* out, int64_t n, void* stream)                          /* T:594-626 */
EK_THERMO_FN(specific_humidity_from_relative_humidity, ek_operand t, ek_operand r, ek_operand p, void* out, int64_t n, void* stream) /* T:629-663 */
EK_THERMO_FN(dewpoint_from_relative_humidity, ek_operand t, ek_operand r, void* out, int64_t n, void* stream)                      /* T:666-699 */
EK_THERMO_FN(dewpoint_from_specific_humidity, ek_operand q, ek_operand p, void* out, int64_t n, void* stream)                      /* T:702-735 */

/* ---- virtual / potential temperature, dry adiabats, lcl ----------------------------------------- */
EK_THERMO_FN(virtual_temperature, ek_operand t, ek_operand q, void* out, int64_t n, void* stream)                          /* T:738-764 */
EK_THERMO_FN(virtual_potential_temperature, ek_operand t, ek_operand q, ek_operand p, void* out, int64_t n, void* stream)  /* T:767-798 */
EK_THERMO_FN(potential_temperature, ek_operand t, ek_operand p, void* out, int64_t n, void* stream)                        /* T:801-829 */
EK_THERMO_FN(temperature_from_potential_temperature, ek_operand th, ek_operand p, void* out, int64_t n, void* stream)      /* T:832-858 */
EK_THERMO_FN(pressure_on_dry_adiabat, ek_operand t, ek_operand t_def, ek_operand p_def, void* out, int64_t n, void* stream) /* T:861-889 */
EK_THERMO_FN(temperature_on_dry_adiabat, ek_operand p, ek_operand t_def, ek_operand p_def, void* out, int64_t n, void* stream) /* T:892-920 */
EK_THERMO_FN(lcl_temperature, ek_operand t, ek_operand td, int method, void* out, int64_t n, void* stream)                 /* T:923-968 */
EK_THERMO_FN(lcl, ek_operand t, ek_operand td, ek_operand p, int method, void* t_lcl_out, void* p_lcl_out, int64_t n, void* stream) /* T:971-1000 */
EK_THERMO_FN(specific_gas_constant, ek_operand q, void* out, int64_t n, void* stream)                                      /* T:1678-1707 */

/* ---- equivalent potential temperature, moist adiabats, wet bulb -------------------------------- */
EK_THERMO_FN(ept_from_dewpoint, ek_operand t, ek_operand td, ek_operand p, int method, void* out, int64_t n, void* stream)          /* T:1326-1387 */
EK_THERMO_FN(ept_from_specific_humidity, ek_operand t, ek_operand q, ek_operand p, int method, void* out, int64_t n, void* stream)  /* T:1390-1415 */
EK_THERMO_FN(saturation_ept, ek_operand t, ek_operand p, int method, void* out, int64_t n, void* stream)                            /* T:1418-1469 */
/* t_method: EK_TM_BISECT or EK_TM_NEWTON */
EK_THERMO_FN(temperature_on_moist_adiabat, ek_operand ept, ek_operand p, int ept_method, int t_method, void* out, int64_t n, void* stream) /* T:1472-1509 */
EK_THERMO_FN(wet_bulb_temperature_from_dewpoint, ek_operand t, ek_operand td, ek_operand p, int ept_method, int t_method, void* out,
             int64_t n, void* stream)                                                                                                /* T:1512-1549 */
EK_THERMO_FN(wet_bulb_temperature_from_specific_humidity, ek_operand t, ek_operand q, ek_operand p, int ept_method, int t_method,
             void* out, int64_t n, void* stream)                                                                                     /* T:1552-1590 */
/* t_method: EK_TM_DIRECT, EK_TM_BISECT or EK_TM_NEWTON */
EK_THERMO_FN(wet_bulb_potential_temperature_from_dewpoint, ek_operand t, ek_operand td, ek_operand p, int ept_method, int t_method,
             void* out, int64_t n, void* stream)                                                                                     /* T:1593-1634 */
EK_THERMO_FN(wet_bulb_potential_temperature_from_specific_humidity, ek_operand t, ek_operand q, ek_operand p, int ept_method,
             int t_method, void* out, int64_t n, void* stream)                                                                       /* T:1637-1675 */

/* ---- fused multi-output kernels (new in this build; each output equals the reference function named
 *      at its slot, see EK_S_*) ------------------------------------------------------------------- */
/* (t, q, p) -> any subset of {theta, es, rh, td, tv, w, e, thetav, ept, wbpt}; outs has EK_S_NSLOTS entries, outs[k] may be
 * NULL when bit k is clear.  ept_method (EK_EPT_*) is the formulation of slots 8 / 9 and is ignored when neither is asked
 * for.  One launch with mask 0x30D is the single pass "read t/q/p once, write theta, rh, td, theta_e, theta_w"; the chain it
 * replaces in the reference is T:1637-1675 -> T:1390-1415 -> T:1031-1040 -> T:702-735 + T:801-829. */
EK_THERMO_FN(suite_tqp, ek_operand t, ek_operand q, ek_operand p, void* const* outs, uint32_t out_mask, int ept_method, int64_t n,
             void* stream)
/* (t, td, p) -> any subset of {theta, es, rh, q, tv, w, e, thetav, ept, wbpt} */
EK_THERMO_FN(suite_ttdp, ek_operand t, ek_operand td, ek_operand p, void* const* outs, uint32_t out_mask, int ept_method, int64_t n,
             void* stream)
/* The suites over n_seg SEPARATE fields of n_per_seg points each (one allocation per level / member, as a per-level caller
 * holds them) in ONE launch: a launch per 1 M-point level is latency-bound (12-16 us for 6 us of HBM time).  t / h / p: HOST
 * arrays of n_seg DEVICE pointers, or NULL for the broadcast scalar scalars[k] (k = 0, 1, 2); outs[k]: HOST array of n_seg
 * DEVICE pointers for slot k, or NULL when bit k of out_mask is clear.  level_scalars: NULL, or a HOST array of n_seg numbers --
 * the pressure as ONE number per field (pressure-level data: the loop `for lev: theta(t[lev], p_lev)` of a reference user in one
 * launch); p must then be NULL.  The pointer tables and level scalars are copied into the kernel parameters at launch; results
 * are bit-identical to n_seg separate suite launches. */
EK_THERMO_FN(suite_tqp_batch, int n_seg, const void* const* t, const void* const* q, const void* const* p, const double* scalars,
             const double* level_scalars, void* const* const* outs, uint32_t out_mask, int ept_method, int64_t n_per_seg, void* stream)
EK_THERMO_FN(suite_ttdp_batch, int n_seg, const void* const* t, const void* const* td, const void* const* p, const double* scalars,
             const double* level_scalars, void* const* const* outs, uint32_t out_mask, int ept_method, int64_t n_per_seg, void* stream)
/* (t, h, p) -> ept and/or the wet-bulb (potential) temperature in one pass.  h is td or q (humidity_kind),
 * at_p0 = 1 gives the wet-bulb POTENTIAL temperature; either output pointer may be NULL (but not both);
 * t_method EK_TM_NONE computes ept only */
EK_THERMO_FN(ept_wet_bulb, ek_operand t, ek_operand h, ek_operand p, int humidity_kind, int ept_method, int t_method, int at_p0,
             void* ept_out, void* wb_out, int64_t n, void* stream)

/* ---- wind: the elementwise functions of earthkit.meteo.wind (SURVEY.md 8(f)-3; src/earthkit/meteo/wind/array/wind.py "W") ----
 * convention: 0 = "meteo", 1 = "polar" (W:99-104, W:184-189) */
enum { EK_WIND_METEO = 0, EK_WIND_POLAR = 1 };
EK_THERMO_FN(wind_speed, ek_operand u, ek_operand v, void* out, int64_t n, void* stream)                                       /* W:15-34 */
EK_THERMO_FN(wind_direction, ek_operand u, ek_operand v, int convention, int to_positive, void* out, int64_t n, void* stream)  /* W:64-104 */
EK_THERMO_FN(wind_xy_to_polar, ek_operand x, ek_operand y, int convention, void* speed_out, void* direction_out, int64_t n, void* stream) /* W:107-135 */
EK_THERMO_FN(wind_polar_to_xy, ek_operand magnitude, ek_operand direction, int convention, void* x_out, void* y_out, int64_t n, void* stream) /* W:156-189 */
EK_THERMO_FN(w_from_omega, ek_operand omega, ek_operand t, ek_operand p, void* out, int64_t n, void* stream)                   /* W:192-222 */
EK_THERMO_FN(coriolis, ek_operand lat, void* out, int64_t n, void* stream)                                                     /* W:225-251 */

/* ---- hybrid (IFS model) levels: the step before the thermo path on model levels (SURVEY.md 8(f)-1) -----------
 * Reference: earthkit.meteo.vertical.pressure_on_hybrid_levels, src/earthkit/meteo/vertical/array/vertical.py:505-737 ("V").
 * A, B: DEVICE arrays of nhalf half-level coefficients of the dtype; sp: npl surface pressures.
 * Outputs are [rows, npl], any may be NULL: `full`, `delta`, `alpha` have one row per entry of full_rows (0-based
 * full-level index k = level number - 1), `half` one row per entry of half_rows (half-level index).  top_k is the
 * full level treated as the column top (the first level of the computed band, V:645-647), top_toa the field-wide
 * decision any(p_half[top] <= 0.1 Pa) (V:678; ek_thermo_hybrid_top_is_toa computes it), alpha_top = ln 2 ("ifs")
 * or 1.0 ("arpege") (V:669).  alpha_delta_f64 = 1: `delta` and `alpha` are float64 arrays also in the _f32 entry point -- the
 * reference allocates them with xp.zeros(...), i.e. float64, whatever the dtype of sp (V:672,686). */
EK_THERMO_FN(pressure_on_hybrid_levels, const void* A, const void* B, int nhalf, const void* sp, int64_t npl, const int* full_rows,
             int n_full, const int* half_rows, int n_half, int top_k, int top_toa, double alpha_top, void* full, void* half, void* delta,
             void* alpha, int alpha_delta_f64, void* stream)
/* ORs 1 into *flag (a zero-initialised DEVICE int) when any(a_top + b_top * sp <= 0.1) (V:678) */
EK_THERMO_FN(hybrid_top_is_toa, const void* sp, int64_t npl, double a_top, double b_top, int* flag, void* stream)
/* geopotential thickness / geopotential / height of hybrid full levels (SURVEY.md 8(f)-2; V:741-1188): d = R(q) t per
 * layer and a bottom-up running sum along the level axis, one thread per column.  t, q, out: [nlev, npl] with level 0 the
 * top of the band; the band is the nlev BOTTOM-most model levels (V:1191-1203).  alpha/delta are computed in registers
 * from sp and the nhalf half-level coefficients A, B -- or read from memory when `alpha` and `delta` are non-NULL
 * (then sp/A/B may be NULL).  mode: 0 thickness, 1 geopotential (+ zs), 2 geopotential height above sea ((dphi+zs)/g),
 * 3 geopotential height above ground (dphi/g), 4 geometric height above sea, 5 geometric height above ground. */
enum { EK_HM_THICKNESS = 0, EK_HM_GEOPOTENTIAL = 1, EK_HM_GH_SEA = 2, EK_HM_GH_GROUND = 3, EK_HM_GEOM_SEA = 4, EK_HM_GEOM_GROUND = 5 };
EK_THERMO_FN(geopotential_on_hybrid_levels, const void* t, const void* q, int nlev, int64_t npl, const void* sp, const void* A,
             const void* B, int nhalf, int top_toa, double alpha_top, const void* alpha, const void* delta, const void* zs, int mode,
             void* out, void* stream)
/* the output forms of the function above, elementwise, for a thickness / geopotential that is already in memory: mode 0-5 as
 * EK_HM_* (dphi = thickness, zs = surface geopotential), 6 = geometric_height_from_geopotential(dphi) (V:472-502); mode 3 with
 * dphi = z is geopotential_height_from_geopotential(z) (V:330-353).  Used by the replicated vertical_axis != 0 path. */
EK_THERMO_FN(height_from_thickness, ek_operand dphi, ek_operand zs, int mode, void* out, int64_t n, void* stream)
/* the (t, q, p) suite with p = full-level pressure computed in registers from sp and A/B (nlev + 1 coefficients each);
 * t, q and every output are [nlev, npl]; p_out (optional) receives the pressure itself */
EK_THERMO_FN(suite_tq_hybrid, const void* t, const void* q, const void* sp, const void* A, const void* B, int nlev, int64_t npl,
             void* const* outs, uint32_t out_mask, int ept_method, void* p_out, void* stream)
/* suite_tq_hybrid and the geopotential of the same levels in one walk of the columns (bottom to top): t and q are read once
 * for both.  t, q, outs, out_mask, ept_method, p_out as for suite_tq_hybrid (the suite: T:801-829 ... T:1637-1675 at the
 * slots of EK_S_*; p: V:663,708); out_mask may be 0 when a column output is given.  The column outputs are
 * geopotential_on_hybrid_levels over all nlev levels (A, B: nlev + 1 half-level coefficients), any may be NULL:
 *   thickness_out  dphi, relative_geopotential_thickness_on_hybrid_levels (V:894-994; d = R(q) t, V:799-810);
 *   z_out          dphi + zs, geopotential_on_hybrid_levels (V:997-1069);
 *   height_out     form height_mode (EK_HM_*) of dphi, height_on_hybrid_levels (V:1072-1188).
 * zs: surface geopotential [npl], needed by z_out and by the height modes that add it (all but EK_HM_THICKNESS and
 * EK_HM_GH_GROUND), else may be NULL.  top_toa: any(A[0] + B[0] * sp <= 0.1) over the field (V:678; ek_thermo_hybrid_top_is_toa
 * computes it); alpha_top = ln 2 ("ifs") or 1.0 ("arpege") (V:669).  Every output is bit-identical to the separate
 * suite_tq_hybrid and geopotential_on_hybrid_levels launches on the same arrays. */
EK_THERMO_FN(suite_tq_hybrid_geo, const void* t, const void* q, const void* sp, const void* zs, const void* A, const void* B, int nlev,
             int64_t npl, void* const* outs, uint32_t out_mask, int ept_method, void* p_out, int top_toa, double alpha_top,
             void* thickness_out, void* z_out, void* height_out, int height_mode, void* stream)

/* ---- host-buffer pipelines: the same suite kernels fed from HOST arrays ------------------------------
 * Stream n points through the GPU in chunks: H2D copy, kernel and D2H copy of successive chunks overlap on
 * `n_slots` internal streams.  Host buffers should be page-locked for full PCIe speed.  `workspace` is a
 * caller-owned DEVICE buffer of workspace_bytes with no work pending on it; chunk size = workspace_bytes /
 * (n_slots * (3 + popcount(mask)) * sizeof(T)).  Block until every output byte is in host memory (also on error:
 * the pipeline's streams are drained before the call returns).  kind: 0 = suite_tqp, 1 = suite_ttdp; out_mask,
 * ept_method as for the suites (slots 8 / 9 included, so the ept / wet-bulb workload has a host path too). */
EK_THERMO_FN(host_suite, int kind, const void* h_a, const void* h_b, const void* h_c, void* const* h_outs, uint32_t out_mask,
             int ept_method, int64_t n, void* workspace, size_t workspace_bytes, int n_slots)
/* suite_tq_hybrid from HOST arrays: h_t, h_q and every output [nlev, npl], h_sp [npl], h_A / h_B nlev + 1 half-level
 * coefficients.  The pressure field exists on neither side of PCIe (16 + 8/nlev instead of 24 bytes per point travel
 * to the device).  Chunks are column ranges of all levels, moved as 2-D copies. */
EK_THERMO_FN(host_suite_tq_hybrid, const void* h_t, const void* h_q, const void* h_sp, const void* h_A, const void* h_B, int nlev,
             int64_t npl, void* const* h_outs, uint32_t out_mask, int ept_method, void* workspace, size_t workspace_bytes, int n_slots)
/* suite_tq_hybrid_geo from HOST arrays: h_t, h_q, every suite output and h_thickness / h_z / h_height [nlev, npl], h_sp and h_zs
 * [npl], h_A / h_B nlev + 1 half-level coefficients; zs, top_toa, alpha_top, height_mode and the NULL rules as for
 * suite_tq_hybrid_geo (no pressure output).  h_zs travels with each chunk only when an output needs it. */
EK_THERMO_FN(host_suite_tq_hybrid_geo, const void* h_t, const void* h_q, const void* h_sp, const void* h_zs, const void* h_A, const void* h_B,
             int nlev, int64_t npl, void* const* h_outs, uint32_t out_mask, int ept_method, int top_toa, double alpha_top, void* h_thickness,
             void* h_z, void* h_height, int height_mode, void* workspace, size_t workspace_bytes, int n_slots)

#ifdef __cplusplus
}
#endif
#endif /* EK_THERMO_H */
