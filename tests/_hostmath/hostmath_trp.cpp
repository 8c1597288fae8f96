// hostmath_trp.cpp -- TEST-ONLY host instantiation of the (t, r, p) suite functor OpSuiteTRPm (ek_thermo_ops.inc).
//
// Compiled with plain g++ (no CUDA) and loaded only by tests/test_suite_trp_cpu.py, the way hostmath.cpp serves
// tests/test_hostmath.py: the per-point logic the suite kernels execute is checked against the oracle on the CPU.  Not part of
// the product: the ek_thermo package never loads it.
#include <cstdint>

#include "../../earthkit-meteo_b200/csrc/ek_thermo_math.cuh"

using namespace ek;
using namespace ek::exactm;

template <class Op, typename T>
static void run(const void* const* ins, const double* scalars, void* const* outs, int64_t n, const Params& P) {
    for (int64_t i = 0; i < n; ++i) {
        T a[Op::NIN], r[Op::NOUT];
        for (int k = 0; k < Op::NIN; ++k) a[k] = ins[k] ? static_cast<const T*>(ins[k])[i] : static_cast<T>(scalars[k]);
        for (int o = 0; o < Op::NOUT; ++o) r[o] = T(0);
        Op::template apply<T>(a, r, P);
        for (int o = 0; o < Op::NOUT; ++o)
            if (outs[o]) static_cast<T*>(outs[o])[i] = r[o];
    }
}

template <uint32_t MASK, int M> static int both(int f32, const void* const* ins, const double* sc, void* const* outs, int64_t n, const Params& P) {
    if (f32) run<OpSuiteTRPm<MASK, M>, float>(ins, sc, outs, n, P); else run<OpSuiteTRPm<MASK, M>, double>(ins, sc, outs, n, P);
    return 0;
}

// static_mask = 0: the run-time-mask instantiation of ept method m; otherwise the compile-time-mask instantiation the library
// ships for that set (IFS only, as in ek_ops_fused_impl.cuh)
extern "C" int hostmath_trp_run(int f32, const void* const* ins, const double* scalars, void* const* outs, int64_t n, uint32_t out_mask, int m,
                                uint32_t static_mask) {
    Params P;
    P.out_mask = out_mask;
    if (static_mask != 0 && m != EPT_IFS) return -2;
    switch (static_mask) {
        case 0: break;
        case 0x1F: return both<0x1F, EPT_IFS>(f32, ins, scalars, outs, n, P);
        case 0x05: return both<0x05, EPT_IFS>(f32, ins, scalars, outs, n, P);
        case 0x2C: return both<0x2C, EPT_IFS>(f32, ins, scalars, outs, n, P);
        case 0x31F: return both<0x31F, EPT_IFS>(f32, ins, scalars, outs, n, P);
        case 0x30D: return both<0x30D, EPT_IFS>(f32, ins, scalars, outs, n, P);
        case 0x300: return both<0x300, EPT_IFS>(f32, ins, scalars, outs, n, P);
        default: return -1;
    }
    switch (m) {
        case EPT_IFS: return both<0, EPT_IFS>(f32, ins, scalars, outs, n, P);
        case EPT_BOLTON35: return both<0, EPT_BOLTON35>(f32, ins, scalars, outs, n, P);
        case EPT_BOLTON39: return both<0, EPT_BOLTON39>(f32, ins, scalars, outs, n, P);
    }
    return -2;
}
