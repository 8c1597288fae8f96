// ek_ops_fused_impl.cuh -- fused multi-output suites: read (t,q,p), (t,td,p) or (t,r,p) once, write every requested field.
// Included by ek_ops_fused_tqp.cu / ek_ops_fused_ttdp.cu / ek_ops_fused_trp.cu (one translation unit per suite, compiled in parallel).
#pragma once
#include "ek_launch.cuh"

using namespace ek;

template <template <uint32_t, int> class OpM, template <uint32_t, int> class OpME, typename T>
static int suite(const char* what, ek_operand a, ek_operand b, ek_operand c, void* const* outs, uint32_t out_mask, int ept_method, int64_t n,
                 void* stream) {
    void* o[S_NSLOTS];
    if (int rc = suite_outputs(what, outs, out_mask, false, o)) return rc;
    if (int rc = suite_ept_method(what, out_mask, ept_method)) return rc;
    ek_operand ins[3] = {a, b, c};
    // output sets with a dedicated compile-time instantiation (the bench / config workloads); any other set
    // runs the generic kernel that tests the mask at run time
    switch (ept_method) {
        case EK_EPT_IFS:
            switch (out_mask) {
                case 0x1F: return launch<OpM<0x1F, EPT_IFS>, OpME<0x1F, EPT_IFS>, T>(what, ins, o, n, Params{}, stream);  // theta, es, rh, td|q, tv
                case 0x05: return launch<OpM<0x05, EPT_IFS>, OpME<0x05, EPT_IFS>, T>(what, ins, o, n, Params{}, stream);  // theta, rh
                case 0x2C: return launch<OpM<0x2C, EPT_IFS>, OpME<0x2C, EPT_IFS>, T>(what, ins, o, n, Params{}, stream);  // rh, td|q, w
                case 0x31F: return launch<OpM<0x31F, EPT_IFS>, OpME<0x31F, EPT_IFS>, T>(what, ins, o, n, Params{}, stream);  // + ept, wbpt: the single pass
                case 0x30D: return launch<OpM<0x30D, EPT_IFS>, OpME<0x30D, EPT_IFS>, T>(what, ins, o, n, Params{}, stream);  // theta, rh, td|q, ept, wbpt
                case 0x300: return launch<OpM<0x300, EPT_IFS>, OpME<0x300, EPT_IFS>, T>(what, ins, o, n, Params{}, stream);  // ept, wbpt
                default: return launch<OpM<0, EPT_IFS>, OpME<0, EPT_IFS>, T>(what, ins, o, n, Params{}, stream);
            }
        case EK_EPT_BOLTON35: return launch<OpM<0, EPT_BOLTON35>, OpME<0, EPT_BOLTON35>, T>(what, ins, o, n, Params{}, stream);
        default: return launch<OpM<0, EPT_BOLTON39>, OpME<0, EPT_BOLTON39>, T>(what, ins, o, n, Params{}, stream);  // EK_EPT_BOLTON39
    }
}

// The same suites over n_seg separate fields (one allocation per level / member) in one launch.  Run-time mask kernel per ept
// formulation, plus the compile-time sets a per-level caller is most likely to ask for.
template <template <uint32_t, int> class OpM, template <uint32_t, int> class OpME, typename T>
static int suite_batch(const char* what, int n_seg, const void* const* a, const void* const* b, const void* const* c, const double* scalars,
                       const double* level_scalars, void* const* const* outs, uint32_t out_mask, int ept_method, int64_t n_per_seg, void* stream) {
    void* const* o[S_NSLOTS];
    if (int rc = suite_outputs(what, outs, out_mask, false, o)) return rc;
    if (int rc = suite_ept_method(what, out_mask, ept_method)) return rc;
    const void* const* ins[3] = {a, b, c};
    switch (ept_method) {
        case EK_EPT_IFS:
            switch (out_mask) {
                case 0x1F: return launch_batch<OpM<0x1F, EPT_IFS>, OpME<0x1F, EPT_IFS>, T>(what, n_seg, ins, scalars, level_scalars, o, n_per_seg, Params{}, stream);
                case 0x05: return launch_batch<OpM<0x05, EPT_IFS>, OpME<0x05, EPT_IFS>, T>(what, n_seg, ins, scalars, level_scalars, o, n_per_seg, Params{}, stream);
                case 0x31F: return launch_batch<OpM<0x31F, EPT_IFS>, OpME<0x31F, EPT_IFS>, T>(what, n_seg, ins, scalars, level_scalars, o, n_per_seg, Params{}, stream);
                default: return launch_batch<OpM<0, EPT_IFS>, OpME<0, EPT_IFS>, T>(what, n_seg, ins, scalars, level_scalars, o, n_per_seg, Params{}, stream);
            }
        case EK_EPT_BOLTON35: return launch_batch<OpM<0, EPT_BOLTON35>, OpME<0, EPT_BOLTON35>, T>(what, n_seg, ins, scalars, level_scalars, o, n_per_seg, Params{}, stream);
        default: return launch_batch<OpM<0, EPT_BOLTON39>, OpME<0, EPT_BOLTON39>, T>(what, n_seg, ins, scalars, level_scalars, o, n_per_seg, Params{}, stream);  // EK_EPT_BOLTON39
    }
}
