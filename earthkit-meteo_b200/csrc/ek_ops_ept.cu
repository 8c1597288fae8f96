// ek_ops_ept.cu -- equivalent potential temperature, moist adiabats and wet-bulb temperatures
// (SURVEY.md §8(a) A31-A44).  One kernel instantiation per (ept formulation, solver) pair so that the
// iterate and every intermediate of the chosen formulation stay in registers.
#include "ek_launch.cuh"

using namespace ek;

#if EK_LEAN_MATH
// Fills lean::ek_bisect_tab: {es_mixed(t), ln t} for the 4095 nodes of the bisection tree (see ek_thermo_lean.cuh).
// Launched on the caller's stream right before every bisection kernel: ~3 us, stateless, safe under graph capture.
__global__ void bisect_tab_init_kernel() {
#if EK_LEAN_DEVICE
    lean::init_tables();
    for (int node = 1 + blockIdx.x * blockDim.x + threadIdx.x; node < EK_BISECT_NODES; node += gridDim.x * blockDim.x) {
        const double t = fastm::bisect_node_t<double>(node);
        lean::ek_bisect_tab[node] = make_double2(fastm::es_mixed(t), lean::log_(t));
        const float tf = fastm::bisect_node_t<float>(node);
        lean::ek_bisect_tab_f[node] = make_float2(fastm::es_mixed(tf), lean::log_(tf));
    }
#endif
}
static int bisect_prepare(const char* what, void* stream) {
    bisect_tab_init_kernel<<<16, 256, kSmemBytes, static_cast<cudaStream_t>(stream)>>>();
    return launched(what);
}
#else
static int bisect_prepare(const char*, void*) { return EK_OK; }
#endif

template <typename T, int M, int TM, int HUM = -1>
static int ept_wb_mt(ek_operand t, ek_operand h, ek_operand p, int hum, int at_p0, void* ept_out, void* wb_out, int64_t n, void* stream) {
    ek_operand ins[3] = {t, h, p};
    void* outs[2] = {ept_out, TM == TM_NONE ? nullptr : wb_out};
    Params P;
    P.opt0 = hum;
    P.opt1 = at_p0;
    if (TM == TM_BISECT && n > 0) {
        const int rc = bisect_prepare("ept_wet_bulb", stream);
        if (rc != EK_OK) return rc;
    }
    return launch<EK_OPS(OpEptWb<M, TM, HUM>), T>("ept_wet_bulb", ins, outs, n, P, stream);
}

template <typename T, int M>
static int ept_wb_m(int tm, ek_operand t, ek_operand h, ek_operand p, int hum, int at_p0, void* e, void* w, int64_t n, void* s) {
    switch (tm) {
        // the two HBM-bound forms get one instantiation per humidity kind (see OpEptWb)
        case EK_TM_NONE:
            return hum ? ept_wb_mt<T, M, TM_NONE, 1>(t, h, p, hum, at_p0, e, w, n, s) : ept_wb_mt<T, M, TM_NONE, 0>(t, h, p, hum, at_p0, e, w, n, s);
        case EK_TM_DIRECT:
            return hum ? ept_wb_mt<T, M, TM_DIRECT, 1>(t, h, p, hum, at_p0, e, w, n, s) : ept_wb_mt<T, M, TM_DIRECT, 0>(t, h, p, hum, at_p0, e, w, n, s);
        case EK_TM_BISECT: return ept_wb_mt<T, M, TM_BISECT>(t, h, p, hum, at_p0, e, w, n, s);
        case EK_TM_NEWTON: return ept_wb_mt<T, M, TM_NEWTON>(t, h, p, hum, at_p0, e, w, n, s);
    }
    return set_error(EK_ERR_ENUM, "ept_wet_bulb: invalid t_method id %d", tm);
}

template <typename T>
static int impl_ept_wet_bulb(ek_operand t, ek_operand h, ek_operand p, int hum, int m, int tm, int at_p0, void* ept_out, void* wb_out,
                             int64_t n, void* stream) {
    if (hum != EK_HUM_DEWPOINT && hum != EK_HUM_SPECIFIC) return set_error(EK_ERR_ENUM, "ept_wet_bulb: invalid humidity kind %d", hum);
    if (tm == EK_TM_NONE && !ept_out) return set_error(EK_ERR_ARG, "ept_wet_bulb: t_method NONE needs ept_out");
    if (tm != EK_TM_NONE && !ept_out && !wb_out) return set_error(EK_ERR_ARG, "ept_wet_bulb: no output buffer given");
    if (tm == EK_TM_DIRECT && !at_p0) return set_error(EK_ERR_ENUM, "ept_wet_bulb: t_method DIRECT only exists for the potential (at_p0) variant");
    switch (m) {
        case EK_EPT_IFS: return ept_wb_m<T, EPT_IFS>(tm, t, h, p, hum, at_p0, ept_out, wb_out, n, stream);
        case EK_EPT_BOLTON35: return ept_wb_m<T, EPT_BOLTON35>(tm, t, h, p, hum, at_p0, ept_out, wb_out, n, stream);
        case EK_EPT_BOLTON39: return ept_wb_m<T, EPT_BOLTON39>(tm, t, h, p, hum, at_p0, ept_out, wb_out, n, stream);
    }
    return set_error(EK_ERR_ENUM, "ept_wet_bulb: invalid ept method id %d", m);
}
EK_API(ept_wet_bulb,
       (ek_operand t, ek_operand h, ek_operand p, int hum, int m, int tm, int at_p0, void* ept_out, void* wb_out, int64_t n, void* stream),
       (t, h, p, hum, m, tm, at_p0, ept_out, wb_out, n, stream))

// ---- the reference's public names, as thin views of the fused entry point -------------------------
template <typename T> static int impl_ept_from_dewpoint(ek_operand t, ek_operand td, ek_operand p, int m, void* out, int64_t n, void* s) {
    return impl_ept_wet_bulb<T>(t, td, p, EK_HUM_DEWPOINT, m, EK_TM_NONE, 0, out, nullptr, n, s);
}
EK_API(ept_from_dewpoint, (ek_operand t, ek_operand td, ek_operand p, int m, void* out, int64_t n, void* s), (t, td, p, m, out, n, s))

template <typename T> static int impl_ept_from_specific_humidity(ek_operand t, ek_operand q, ek_operand p, int m, void* out, int64_t n, void* s) {
    return impl_ept_wet_bulb<T>(t, q, p, EK_HUM_SPECIFIC, m, EK_TM_NONE, 0, out, nullptr, n, s);
}
EK_API(ept_from_specific_humidity, (ek_operand t, ek_operand q, ek_operand p, int m, void* out, int64_t n, void* s), (t, q, p, m, out, n, s))

#define EK_WB(NAME, HUM, AT_P0, ALLOW_DIRECT)                                                                                    \
    template <typename T> static int impl_##NAME(ek_operand t, ek_operand h, ek_operand p, int m, int tm, void* out, int64_t n, void* s) { \
        if (!(tm == EK_TM_BISECT || tm == EK_TM_NEWTON || (ALLOW_DIRECT && tm == EK_TM_DIRECT)))                                 \
            return set_error(EK_ERR_ENUM, #NAME ": invalid t_method id %d", tm);                                                 \
        if (!out) return set_error(EK_ERR_ARG, #NAME ": out is NULL");                                                           \
        return impl_ept_wet_bulb<T>(t, h, p, HUM, m, tm, AT_P0, nullptr, out, n, s);                                             \
    }                                                                                                                            \
    EK_API(NAME, (ek_operand t, ek_operand h, ek_operand p, int m, int tm, void* out, int64_t n, void* s), (t, h, p, m, tm, out, n, s))

EK_WB(wet_bulb_temperature_from_dewpoint, EK_HUM_DEWPOINT, 0, 0)
EK_WB(wet_bulb_temperature_from_specific_humidity, EK_HUM_SPECIFIC, 0, 0)
EK_WB(wet_bulb_potential_temperature_from_dewpoint, EK_HUM_DEWPOINT, 1, 1)
EK_WB(wet_bulb_potential_temperature_from_specific_humidity, EK_HUM_SPECIFIC, 1, 1)

// ---- saturation ept (T:1418-1469) ------------------------------------------------------------------
template <typename T> static int impl_saturation_ept(ek_operand t, ek_operand p, int m, void* out, int64_t n, void* stream) {
    ek_operand ins[2] = {t, p};
    void* outs[1] = {out};
    switch (m) {
        case EK_EPT_IFS: return launch<EK_OPS(OpSatEpt<EPT_IFS>), T>("saturation_ept", ins, outs, n, Params{}, stream);
        case EK_EPT_BOLTON35: return launch<EK_OPS(OpSatEpt<EPT_BOLTON35>), T>("saturation_ept", ins, outs, n, Params{}, stream);
        case EK_EPT_BOLTON39: return launch<EK_OPS(OpSatEpt<EPT_BOLTON39>), T>("saturation_ept", ins, outs, n, Params{}, stream);
    }
    return set_error(EK_ERR_ENUM, "saturation_ept: invalid ept method id %d", m);
}
EK_API(saturation_ept, (ek_operand t, ek_operand p, int m, void* out, int64_t n, void* stream), (t, p, m, out, n, stream))

// ---- temperature on a moist adiabat (T:1472-1509) ---------------------------------------------------
template <typename T, int M> static int t_on_ma_m(int tm, const ek_operand* ins, void* const* outs, int64_t n, void* stream) {
    if (tm == EK_TM_BISECT) {
        if (n > 0) {
            const int rc = bisect_prepare("temperature_on_moist_adiabat", stream);
            if (rc != EK_OK) return rc;
        }
        return launch<EK_OPS(OpTOnMa<M, TM_BISECT>), T>("temperature_on_moist_adiabat", ins, outs, n, Params{}, stream);
    }
    if (tm == EK_TM_NEWTON) return launch<EK_OPS(OpTOnMa<M, TM_NEWTON>), T>("temperature_on_moist_adiabat", ins, outs, n, Params{}, stream);
    return set_error(EK_ERR_ENUM, "temperature_on_moist_adiabat: invalid t_method id %d", tm);
}
template <typename T>
static int impl_temperature_on_moist_adiabat(ek_operand ept, ek_operand p, int m, int tm, void* out, int64_t n, void* stream) {
    ek_operand ins[2] = {ept, p};
    void* outs[1] = {out};
    switch (m) {
        case EK_EPT_IFS: return t_on_ma_m<T, EPT_IFS>(tm, ins, outs, n, stream);
        case EK_EPT_BOLTON35: return t_on_ma_m<T, EPT_BOLTON35>(tm, ins, outs, n, stream);
        case EK_EPT_BOLTON39: return t_on_ma_m<T, EPT_BOLTON39>(tm, ins, outs, n, stream);
    }
    return set_error(EK_ERR_ENUM, "temperature_on_moist_adiabat: invalid ept method id %d", m);
}
EK_API(temperature_on_moist_adiabat, (ek_operand ept, ek_operand p, int m, int tm, void* out, int64_t n, void* stream),
       (ept, p, m, tm, out, n, stream))
