// ek_ops_fused_trp.cu -- entry points of the (t, r, p) suite.
#include "ek_ops_fused_impl.cuh"

template <typename T>
static int impl_suite_trp(ek_operand t, ek_operand r, ek_operand p, void* const* outs, uint32_t m, int ept_method, int64_t n, void* stream) {
    return suite<EK_OPS(OpSuiteTRPm), T>("suite_trp", t, r, p, outs, m, ept_method, n, stream);
}
EK_API(suite_trp, (ek_operand t, ek_operand r, ek_operand p, void* const* outs, uint32_t m, int ept_method, int64_t n, void* stream),
       (t, r, p, outs, m, ept_method, n, stream))

template <typename T>
static int impl_suite_trp_batch(int n_seg, const void* const* t, const void* const* r, const void* const* p, const double* scalars, const double* level_scalars,
                                 void* const* const* outs, uint32_t m, int ept_method, int64_t n_per_seg, void* stream) {
    return suite_batch<EK_OPS(OpSuiteTRPm), T>("suite_trp_batch", n_seg, t, r, p, scalars, level_scalars, outs, m, ept_method, n_per_seg, stream);
}
EK_API(suite_trp_batch,
       (int n_seg, const void* const* t, const void* const* r, const void* const* p, const double* scalars, const double* level_scalars, void* const* const* outs,
        uint32_t m, int ept_method, int64_t n_per_seg, void* stream),
       (n_seg, t, r, p, scalars, level_scalars, outs, m, ept_method, n_per_seg, stream))

// used by the host-buffer pipeline in ek_api.cu
template <typename T> int ek_suite_launch_trp(const ek_operand* ins, void* const* outs, uint32_t mask, int ept_method, int64_t n, void* stream) {
    return suite<EK_OPS(OpSuiteTRPm), T>("host_suite", ins[0], ins[1], ins[2], outs, mask, ept_method, n, stream);
}
template int ek_suite_launch_trp<double>(const ek_operand*, void* const*, uint32_t, int, int64_t, void*);
template int ek_suite_launch_trp<float>(const ek_operand*, void* const*, uint32_t, int, int64_t, void*);
