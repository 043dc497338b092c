// kern_inst.cu -- one group of instantiations of the thread-per-state kernels (thread_kernels.cuh), selected with -DMB_INST=<group>
// so that the groups compile in parallel (Makefile).
#include "thread_kernels.cuh"

#ifndef MB_INST
#error "compile with -DMB_INST=<group>"
#endif

namespace mb
{
#define MB_X(G, ALGO, FEXT, LAYOUT, M3) MB_INST_##G(ALGO, FEXT, LAYOUT, M3)
#define MB_EMIT(ALGO, FEXT, LAYOUT, M3) template KernelFn pick_cfg<ALGO, FEXT, LAYOUT, M3>(int);
#define MB_SKIP(ALGO, FEXT, LAYOUT, M3)
#define MB_SEL(G) (MB_INST == G)
#if MB_INST == 0
#define MB_INST_0 MB_EMIT
#else
#define MB_INST_0 MB_SKIP
#endif
#if MB_INST == 1
#define MB_INST_1 MB_EMIT
#else
#define MB_INST_1 MB_SKIP
#endif
#if MB_INST == 2
#define MB_INST_2 MB_EMIT
#else
#define MB_INST_2 MB_SKIP
#endif
#if MB_INST == 3
#define MB_INST_3 MB_EMIT
#else
#define MB_INST_3 MB_SKIP
#endif
#if MB_INST == 4
#define MB_INST_4 MB_EMIT
#else
#define MB_INST_4 MB_SKIP
#endif
#if MB_INST == 5
#define MB_INST_5 MB_EMIT
#else
#define MB_INST_5 MB_SKIP
#endif
#if MB_INST == 6
#define MB_INST_6 MB_EMIT
#else
#define MB_INST_6 MB_SKIP
#endif
#if MB_INST == 7
#define MB_INST_7 MB_EMIT
#else
#define MB_INST_7 MB_SKIP
#endif
#if MB_INST == 8
#define MB_INST_8 MB_EMIT
#else
#define MB_INST_8 MB_SKIP
#endif
#if MB_INST == 9
#define MB_INST_9 MB_EMIT
#else
#define MB_INST_9 MB_SKIP
#endif
#if MB_INST == 10
#define MB_INST_10 MB_EMIT
#else
#define MB_INST_10 MB_SKIP
#endif
#if MB_INST == 11
#define MB_INST_11 MB_EMIT
#else
#define MB_INST_11 MB_SKIP
#endif
#if MB_INST == 12
#define MB_INST_12 MB_EMIT
#else
#define MB_INST_12 MB_SKIP
#endif
#if MB_INST == 14
#define MB_INST_14 MB_EMIT
#else
#define MB_INST_14 MB_SKIP
#endif
#if MB_INST == 15
#define MB_INST_15 MB_EMIT
#else
#define MB_INST_15 MB_SKIP
#endif
#if MB_INST == 16
#define MB_INST_16 MB_EMIT
#else
#define MB_INST_16 MB_SKIP
#endif
MB_KERNEL_GROUPS(MB_X)

#if MB_INST == 13
KernelFn pick_f32(int algo)
{
   if (algo == MB_RNEA) return thread_kernel_f32<MB_RNEA, kCfg[kF32Cfg[0]].block, aux_of(MB_RNEA, 0), 0, kCfg[kF32Cfg[0]].tm>;
   if (algo == MB_ABA) return thread_kernel_f32<MB_ABA, kCfg[kF32Cfg[1]].block, aux_of(MB_ABA, 0), kAbaRec0, kCfg[kF32Cfg[1]].tm>;
   return thread_kernel_f32<MB_CRBA, kCfg[kF32Cfg[2]].block, aux_of(MB_CRBA, 0), 0, 0>;
}
#endif
} // namespace mb
