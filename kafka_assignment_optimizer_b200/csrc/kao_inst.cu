// kao_inst.cu — explicit instantiations of the search kernels (kao_kernels.cuh) for ONE row width
// (KAO_INST_W words) and evaluation mode (KAO_INST_MODE: 0 full evaluation, row-major; 1 delta
// evaluation; 2 full evaluation, column-major evaluator of kao_device_t.cuh).
// The Makefile compiles this file once per combination; the objects build in parallel.
#include "kao_kernels.cuh"

#if !defined(KAO_INST_W) || !defined(KAO_INST_MODE)
#error "compile with -DKAO_INST_W=<1|2|4|8> -DKAO_INST_MODE=<0|1|2>"
#endif

#define KAO_INST_FULL(W, NPH, R, O)                                      \
    template __global__ void KAO_ROUND_KERNEL(W, NPH, R, O);            \
    template __global__ void KAO_PERSISTENT_KERNEL(W, NPH, R, O, threads_for<W>(), false);
#define KAO_INST_DELTA_K(W, NPH, R, O) template __global__ void KAO_PERSISTENT_KERNEL(W, NPH, R, O, kThreadsDelta, true);

#if KAO_INST_MODE == 2
#if KAO_INST_W > 2
#error "column-major evaluator: rows of up to 64 slots"
#endif
#define KAO_INST_T(S, POP, T)                                                   \
    template __global__ void KAO_PERSISTENT_KERNEL_T(KAO_INST_W, 0, S, POP, T); \
    template __global__ void KAO_PERSISTENT_KERNEL_T(KAO_INST_W, 32, S, POP, T);
KAO_FOR_SCHEDULES(KAO_INST_T)
#elif KAO_INST_MODE == 1
#if KAO_INST_W <= 2
KAO_FOR_CFGS_NARROW(KAO_INST_DELTA_K, KAO_INST_W, 5)
#else
KAO_FOR_CFGS_WIDE(KAO_INST_DELTA_K, KAO_INST_W, 5)
#endif
#elif KAO_INST_W <= 2
KAO_FOR_CFGS_NARROW(KAO_INST_FULL, KAO_INST_W, 5)
#else
KAO_FOR_CFGS_WIDE(KAO_INST_FULL, KAO_INST_W, 5)
#endif
