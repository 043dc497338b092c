// thread_kernels.cuh -- the thread-per-state kernel template and its launch-configuration table.  The instantiations are
// spread over several translation units (kern_inst.cu, one group each, compiled in parallel); kernels.cu declares them extern
// and owns planning and launching.
#pragma once
#include "f32_ctx.cuh"
#include "gpu_ctx.cuh"
#include "kernels.h"
#include "gravity_gradient.cuh"
#include "regressor.cuh"
#include "rnea_derivatives.cuh"

namespace mb
{
// LAYOUT (CRBA): 0 entry-major, 1 state-major, 2 packed (unique non-zero entries, entry-major rows)
// M3: the instantiation handles three-DoF joints (SphericalJoint, PlanarJoint; multidof.cuh)
template <int ALGO, bool FEXT, int LAYOUT, int BLOCK, int AUXN, int RECN, int TM, bool M3>
__device__ __forceinline__ void thread_kernel_body(const MbProgram &P, const KernelArgs &a)
{
   constexpr bool STATE_MAJOR = LAYOUT == 1;
   const int ncst = P.nb * MB_CONST_STRIDE;
   for (int i = threadIdx.x; i < ncst; i += BLOCK)
      mb_smem[i] = a.consts[i];
   using Ctx = GpuCtx2<BLOCK, TM, ring_rows(ALGO), M3>;
   thread_block_run<ALGO, STATE_MAJOR, BLOCK, AUXN, TM, M3>(a, ncst, mb_smem_stack_slots(ALGO, P, TM), P.nstack2, [&](Ctx &c2) {
      if constexpr (ALGO == MB_RNEA)
         rnea_state<double, Ctx, FEXT>(P, c2, a.grav);
      else if constexpr (ALGO == MB_ABA)
         aba_state<double, Ctx, FEXT>(P, c2, a.grav);
      else if constexpr (ALGO == MB_CRBA)
         crba_state<double, Ctx, FEXT, LAYOUT == 2>(P, c2);
      else if constexpr (ALGO == MB_REGRESSOR)
      {
         c2.yzrows = reinterpret_cast<const uint32_t *>(a.zero_entries);
         c2.nyz = a.n_zero;
         regressor_state<double, Ctx>(P, c2, a.grav);
      }
      else if constexpr (ALGO == MB_GRAVITY_GRADIENT)
         gravity_gradient_state<double, Ctx>(P, c2, a.grav);
      else if constexpr (ALGO == MB_RNEA_DERIVATIVES)
         rnea_derivatives_state<double, Ctx>(P, c2, a.grav);
      else
         coriolis_state<double, Ctx>(P, c2);
   });
}
template <int ALGO, bool FEXT, int LAYOUT, int BLOCK, int AUXN, int RECN, int TM, bool M3>
__global__ void __launch_bounds__(BLOCK) thread_kernel(const __grid_constant__ MbProgram P, const KernelArgs a)
{
   thread_kernel_body<ALGO, FEXT, LAYOUT, BLOCK, AUXN, RECN, TM, M3>(P, a);
}
// The optional fp32 variant (f32_ctx.cuh): same skeleton, constant records staged as floats, the per-state routines instantiated
// with T = float.  Plain calls only (no external wrenches / by-products), one launch configuration per algorithm.
template <int ALGO, int BLOCK, int AUXN, int RECN, int TM>
__global__ void __launch_bounds__(BLOCK) thread_kernel_f32(const __grid_constant__ MbProgram P, const KernelArgs a)
{
   const int ncst = P.nb * MB_CONST_STRIDE;
   float *cf = reinterpret_cast<float *>(mb_smem);
   for (int i = threadIdx.x; i < ncst; i += BLOCK)
      cf[i] = (float)a.consts[i];
   using Ctx = GpuCtx2<BLOCK, TM, ring_rows(ALGO)>;
   const float grav[3] = {(float)a.grav[0], (float)a.grav[1], (float)a.grav[2]};
   thread_block_run<ALGO, false, BLOCK, AUXN, TM>(a, ncst, mb_smem_stack_slots(ALGO, P, TM), P.nstack2, [&](Ctx &c2) {
      F32Ctx<Ctx> f(c2);
      if constexpr (ALGO == MB_RNEA)
         rnea_state<float, F32Ctx<Ctx>, false>(P, f, grav);
      else if constexpr (ALGO == MB_ABA)
         aba_state<float, F32Ctx<Ctx>, false>(P, f, grav);
      else
         crba_state<float, F32Ctx<Ctx>, false>(P, f);
   });
}

// compiled work-area classes (local memory per thread): {aux, rec}
//   class 0: up to 4 nested branching bodies, 32 one-DoF-equivalent records (humanoids); blocks of 256 / 128
//   class 1: up to 16 nested branching bodies, 128 bodies; blocks of 128 / 64 / 32 (deeper stacks)
__host__ __device__ constexpr int aux_of(int algo, int cls) { return mb_algo(algo).aux * (cls ? 16 : 4); }
constexpr int kAbaRec0 = MB_ABA_REC * 33, kAbaRec1 = MB_ABA_REC * 128;
// launch configurations: threads per block, work-area class, stack slots (double2) held in tensor memory
struct Cfg
{
   int block, cls, tm;
};
constexpr int kNumCfg = 15;
constexpr Cfg kCfg[kNumCfg] = {{512, 0, 32}, {384, 0, 42}, {320, 0, 42}, {256, 0, 64}, {384, 0, 0}, {320, 0, 0}, {256, 0, 0},
                               {192, 0, 0},  {128, 0, 0},  {256, 1, 64}, {128, 1, 128}, {128, 1, 0}, {64, 1, 0},  {32, 1, 0},
                               {640, 0, 24}};

typedef void (*KernelFn)(const MbProgram, const KernelArgs);

template <int ALGO, bool FEXT, int SM, bool M3> KernelFn pick_cfg(int cfg)
{
   constexpr int a0 = aux_of(ALGO, 0);
   constexpr int a1 = aux_of(ALGO, 1);
   constexpr int r0 = ALGO == MB_ABA ? kAbaRec0 : 0, r1 = ALGO == MB_ABA ? kAbaRec1 : 0;
   constexpr bool wide = mb_algo(ALGO).wide_stack;
   switch (cfg)
   {
      // without a wide stack area the TMEM configurations are never planned (mb_tm_fits) and alias the shared-memory kernels
#define MB_CFG_CASE(i) case i: return thread_kernel<ALGO, FEXT, SM, kCfg[i].block, kCfg[i].cls ? a1 : a0, kCfg[i].cls ? r1 : r0, wide ? kCfg[i].tm : 0, M3>;
      MB_CFG_CASE(0) MB_CFG_CASE(1) MB_CFG_CASE(2) MB_CFG_CASE(3) MB_CFG_CASE(4) MB_CFG_CASE(5) MB_CFG_CASE(6)
      MB_CFG_CASE(7) MB_CFG_CASE(8) MB_CFG_CASE(9) MB_CFG_CASE(10) MB_CFG_CASE(11) MB_CFG_CASE(12) MB_CFG_CASE(14)
#undef MB_CFG_CASE
      default: return thread_kernel<ALGO, FEXT, SM, kCfg[13].block, a1, r1, wide ? kCfg[13].tm : 0, M3>;
   }
}

// fp32 variant: the one configuration per algorithm that the planner picks for humanoid-sized trees (kCfg index, class 0),
// for the algorithms that are not thread-only (MbAlgoInfo)
constexpr int kF32Cfg[3] = {0, 1, 8}; // RNEA 512 threads + TMEM, ABA 384 threads + TMEM, CRBA 128 threads
KernelFn pick_f32(int algo);

// the instantiation groups: X(group, ALGO, FEXT, LAYOUT, M3).  The store-bound matrix kernels (CRBA, Coriolis, regressor, gravity
// gradient and inverse-dynamics derivatives: external wrenches tested at run time) exist only
// with the three-DoF joints compiled in (one unit-momentum column loop per multi-DoF joint either way); RNEA and ABA come in
// both forms (multidof.cuh: mb_sub_of)
#define MB_KERNEL_GROUPS(X)                                                                                             \
   X(0, MB_RNEA, false, 0, false) X(1, MB_RNEA, true, 0, false) X(2, MB_ABA, false, 0, false) X(3, MB_ABA, true, 0, false)  \
   X(4, MB_CRBA, false, 0, true) X(5, MB_CRBA, false, 1, true) X(6, MB_CRBA, false, 2, true) X(7, MB_CRBA, true, 0, true)   \
   X(8, MB_CORIOLIS, false, 0, true) X(9, MB_RNEA, false, 0, true) X(10, MB_RNEA, true, 0, true)                            \
   X(11, MB_ABA, false, 0, true) X(12, MB_ABA, true, 0, true) X(14, MB_REGRESSOR, false, 0, true)                           \
   X(15, MB_GRAVITY_GRADIENT, false, 0, true) X(16, MB_RNEA_DERIVATIVES, false, 0, true)
#define MB_NUM_KERNEL_GROUPS 16 // + group 13: the fp32 variant
} // namespace mb
