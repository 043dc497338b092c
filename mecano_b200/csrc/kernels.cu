// kernels.cu -- sm_100a kernels: one thread per state (thread-per-state variant).
//
// Layout of one block:
//   * the traversal program and topology tables arrive as a __grid_constant__ kernel parameter, i.e.
//     they live in the constant bank and are read with uniform (warp-wide) LDC;
//   * the per-body constant records (fixed transforms, inertias) are staged once into shared memory
//     and read as broadcasts;
//   * each thread owns one state: its spatial quantities stay in fp64 registers, and the data that
//     must survive from the downward to the upward sweep lives in a per-thread stack in shared memory,
//     laid out state-minor (stack[slot * blockDim + tid]) so that a warp touches 32 consecutive
//     doubles: conflict-free;
//   * q / qd / qdd / tau / wrench buffers are DoF-major, state-minor in HBM, so every global access of
//     a warp is one fully used 256-byte segment.
// No tensor cores: the recursion is not a dense contraction (SURVEY.md section 2).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <type_traits>

#include "thread_kernels.cuh"

namespace mb
{
// instantiated in kern_inst.cu
#define MB_X(G, ALGO, FEXT, LAYOUT, M3) extern template KernelFn pick_cfg<ALGO, FEXT, LAYOUT, M3>(int);
MB_KERNEL_GROUPS(MB_X)
#undef MB_X
namespace
{
// layout: 0 entry-major, 1 state-major, 2 packed (CRBA only)
// m3: the tree has three-DoF joints (MbProgram::has_3dof)
KernelFn pick(int algo, bool fext, int layout, int cfg, bool m3)
{
   if (algo == MB_RNEA)
      return m3 ? (fext ? pick_cfg<MB_RNEA, true, 0, true>(cfg) : pick_cfg<MB_RNEA, false, 0, true>(cfg))
                : (fext ? pick_cfg<MB_RNEA, true, 0, false>(cfg) : pick_cfg<MB_RNEA, false, 0, false>(cfg));
   if (algo == MB_ABA)
      return m3 ? (fext ? pick_cfg<MB_ABA, true, 0, true>(cfg) : pick_cfg<MB_ABA, false, 0, true>(cfg))
                : (fext ? pick_cfg<MB_ABA, true, 0, false>(cfg) : pick_cfg<MB_ABA, false, 0, false>(cfg));
   if (algo == MB_CORIOLIS) return pick_cfg<MB_CORIOLIS, false, 0, true>(cfg);
   if (algo == MB_REGRESSOR) return pick_cfg<MB_REGRESSOR, false, 0, true>(cfg);
   if (algo == MB_GRAVITY_GRADIENT) return pick_cfg<MB_GRAVITY_GRADIENT, false, 0, true>(cfg); // (external wrenches: tested at run time)
   if (algo == MB_RNEA_DERIVATIVES) return pick_cfg<MB_RNEA_DERIVATIVES, false, 0, true>(cfg); // (likewise)
   // CRBA: the "FEXT" instantiation is the one with by-products (centroidal momentum matrix, centre of mass), entry-major only
   if (fext && layout == 0) return pick_cfg<MB_CRBA, true, 0, true>(cfg);
   return layout == 1 ? pick_cfg<MB_CRBA, false, 1, true>(cfg) : (layout == 2 ? pick_cfg<MB_CRBA, false, 2, true>(cfg) : pick_cfg<MB_CRBA, false, 0, true>(cfg));
}

int class_of(int algo, const MbProgram &P)
{
   const int aux0 = aux_of(algo, 0), aux1 = aux_of(algo, 1);
   const int rec0 = algo == MB_ABA ? kAbaRec0 : 0, rec1 = algo == MB_ABA ? kAbaRec1 : 0;
   if (P.aux_doubles <= aux0 && P.rec_doubles <= rec0) return 0;
   if (P.aux_doubles <= aux1 && P.rec_doubles <= rec1) return 1;
   return -1;
}

size_t smem_bytes(int algo, const MbProgram &P, int block, int tm)
{
   const int ncst = (P.nb * MB_CONST_STRIDE + 1) & ~1;
   const int smem_slots = mb_smem_stack_slots(algo, P, tm);
   size_t bytes = sizeof(double) * ((size_t)ncst + (2 * (size_t)smem_slots + ring_rows(algo) * MB_PF_STAGES) * block);
   // a block with a TMEM stack allocates all 512 columns: keep it alone on its SM (a second block would spin in tcgen05.alloc)
   if (tm > 0)
      bytes = std::max<size_t>(bytes, 120 * 1024);
   return bytes;
}

// MECANO_B200_CFG="rnea=0,aba=5,crba=6" pins the launch configuration per algorithm (profiling / sweeps)
int forced_cfg(int algo)
{
   const char *e = getenv("MECANO_B200_CFG");
   if (!e) return -1;
   const std::string key = std::string(mb_algo(algo).cfg_key) + "=";
   const char *p = strstr(e, key.c_str());
   return p ? atoi(p + key.size()) : -1;
}
} // namespace

cudaError_t plan_thread_kernel(int algo, const MbProgram &P, bool fext, LaunchPlan &plan, bool *fits)
{
   *fits = false;
   bool m3 = false;
   for (int i = 0; i < P.nb; i++)
      m3 = m3 || P.body[i].sub != MB_SUB_SIX;
   plan.m3 = m3;
   const int cls = class_of(algo, P);
   if (cls < 0)
      return cudaSuccess;
   int dev = 0, max_optin = 0;
   cudaError_t e = cudaGetDevice(&dev);
   if (e != cudaSuccess) return e;
   e = cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
   if (e != cudaSuccess) return e;
   int best_threads = 0;
   const int forced = forced_cfg(algo);
   for (int cfg = 0; cfg < kNumCfg; cfg++)
   {
      if (kCfg[cfg].cls < cls)
         continue; // work areas too small
      if (forced >= 0 && cfg != forced)
         continue;
      // measured (profiles/r01l_cfg_sweep.jsonl): the TMEM stack buys RNEA 16 warps per SM (0.69 vs 0.99 ms) and ABA 12
      // (384 threads at 168 registers: 1.97 vs 2.10 ms; 512 threads would need 128 registers and spills: 2.96 ms)
      // 640 threads (five warps per sub-partition, 96 registers, deepest wide slots in shared memory) measured slower than
      // 512 (H37 RNEA 0.694 vs 0.656 ms, profiles/r01n_cfg_sweep.jsonl): kept for sweeps only
      if (forced < 0 && kCfg[cfg].block == MB_PARTIAL_TM_BLOCK)
         continue;
      if (!mb_tm_fits(algo, P, kCfg[cfg].tm, kCfg[cfg].block))
         continue; // the wide stack area (three double2 per level of the tree) exceeds the TMEM columns of one warp
      const int b = kCfg[cfg].block;
      const size_t sm = smem_bytes(algo, P, b, kCfg[cfg].tm);
      if (sm > (size_t)max_optin)
         continue;
      // every variant of this configuration gets the opt-in so that later launches cannot fail on it
      KernelFn fn = pick(algo, fext, 0, cfg, m3);
      cudaFuncAttributes fa;
      e = cudaFuncGetAttributes(&fa, (const void *)fn);
      if (e != cudaSuccess) return e;
      const int max_dyn = max_optin - (int)fa.sharedSizeBytes;
      if (sm > (size_t)max_dyn)
         continue;
      for (int f = 0; f < 2; f++)
         for (int st = 0; st < 3; st++)
         {
            e = cudaFuncSetAttribute((const void *)pick(algo, f != 0, st, cfg, m3), cudaFuncAttributeMaxDynamicSharedMemorySize, max_dyn);
            if (e != cudaSuccess) return e;
         }
      int nblk = 0;
      e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nblk, (const void *)fn, b, sm);
      if (e != cudaSuccess) return e;
      if (kCfg[cfg].tm > 0 && nblk > 1)
         nblk = 1; // cannot happen (smem_bytes), but a TMEM block must be alone on its SM
      // register spills cost more than the extra warps bring: a configuration whose kernel spills beyond its declared
      // work area only competes if nothing else fits
      const bool spills = (long)fa.localSizeBytes > 8l * aux_of(algo, kCfg[cfg].cls) + mb_algo(algo).spill_bytes;
      // warps that do not split evenly over the four sub-partitions lose more than they bring (ABA 320 threads: 3.44 ms,
      // 256 threads: 2.23 ms; profiles/r01i_cfg_sweep.jsonl): such block sizes only compete if nothing else fits
      const bool uneven = ((nblk * b) % 128) != 0 && nblk * b > 128;
      const int score = (spills || uneven) && forced < 0 ? 1 + (uneven ? 1 : 0) : nblk * b;
      // prefer more resident states; on ties the first configuration in the table wins, or the smaller block (MbAlgoInfo::small_blocks)
      if (nblk > 0 && (score > best_threads || (mb_algo(algo).small_blocks && score == best_threads && b < plan.block)))
      {
         best_threads = score;
         plan.block = b;
         plan.smem = sm;
         plan.blocks_per_sm = nblk;
         plan.size_class = cfg;
         plan.tm = kCfg[cfg].tm;
      }
   }
   if (best_threads == 0)
      return cudaSuccess; // the stack of even a 32-state block does not fit in shared memory
   cudaFuncAttributes attr;
   e = cudaFuncGetAttributes(&attr, (const void *)pick(algo, fext, 0, plan.size_class, m3));
   if (e != cudaSuccess) return e;
   int sms = 0;
   cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
   plan.grid = sms * plan.blocks_per_sm;
   plan.ws_doubles = algo == MB_ABA ? (size_t)plan.grid * plan.block * (size_t)std::max(P.rec_doubles, 1) : 0;
   plan.regs = attr.numRegs;
   plan.local_bytes = (int)attr.localSizeBytes;
   plan.static_smem = (int)attr.sharedSizeBytes;
   // the fp32 variant exists for the configuration the planner picks for humanoid-sized trees
   plan.fp32_ok = !mb_algo(algo).thread_only && plan.size_class == kF32Cfg[algo] && !m3;
   if (plan.fp32_ok)
   {
      cudaFuncAttributes fa32;
      e = cudaFuncGetAttributes(&fa32, (const void *)pick_f32(algo));
      if (e != cudaSuccess) return e;
      e = cudaFuncSetAttribute((const void *)pick_f32(algo), cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin - (int)fa32.sharedSizeBytes);
      if (e != cudaSuccess) return e;
      plan.fp32_regs = fa32.numRegs;
   }
   *fits = true;
   return cudaSuccess;
}

cudaError_t launch_thread_kernel(int algo, const MbProgram &P, const KernelArgs &a, const LaunchPlan &plan, cudaStream_t stream)
{
   if (a.n <= 0)
      return cudaSuccess;
   const int layout = algo == MB_CRBA ? ((a.flags & 4u) ? 2 : (int)(a.flags & 1u)) : 0; // MECANO_B200_CRBA_PACKED / STATE_MAJOR
   if (a.fp32)
   {
      // api.cu checked plan.fp32_ok and that the call has no optional buffers
      const long long nt = (a.n + plan.block - 1) / plan.block;
      const unsigned g = (algo == MB_ABA || plan.tm > 0) ? (unsigned)std::min<long long>(nt, plan.grid) : (unsigned)nt;
      KernelArgs b = a;
      b.ws_ld = (long long)plan.grid * plan.block;
      b.work_counter = nullptr;
      pick_f32(algo)<<<g, plan.block, plan.smem, stream>>>(P, b);
      return cudaGetLastError();
   }
   KernelFn fn = pick(algo, a.fext != nullptr || a.body_acc != nullptr || a.joint_wrench != nullptr || a.x2 != nullptr || a.cmm != nullptr || a.com != nullptr || a.root_wrench != nullptr, layout, plan.size_class, plan.m3);
   const long long ntiles = (a.n + plan.block - 1) / plan.block;
   // ABA runs as a persistent grid (its pass-two records live in a workspace with one column per resident thread), and so
   // does every kernel with a TMEM stack: a block then allocates its tensor memory, stages the constant records and
   // synchronises once instead of once per tile (H37 RNEA 0.629 -> 0.587 ms).  CRBA (shared-memory stack, several small blocks
   // per SM) measured faster with one block per tile (2.02 vs 2.20 ms): hardware block scheduling evens out its store bursts.
   static const bool persist_all = getenv("MECANO_B200_PERSIST") != nullptr;
   const unsigned grid = (algo == MB_ABA || plan.tm > 0 || persist_all) ? (unsigned)std::min<long long>(ntiles, plan.grid) : (unsigned)ntiles;
   KernelArgs b = a;
   b.ws_ld = (long long)plan.grid * plan.block;
   const bool persistent = grid < (unsigned)ntiles;
   static const bool draw = [] { const char *e = getenv("MECANO_B200_DRAW"); return !e || atoi(e) != 0; }();
   // the warps of a persistent grid draw their states from a counter that the kernel itself re-arms (gpu_ctx.cuh: thread_block_run)
   // (wide-stack kernels only: the mass-matrix kernels are launched one block per tile, and their stores carry no guard for clamped lanes)
   if (!(persistent && draw) || !mb_algo(algo).wide_stack)
      b.work_counter = nullptr;
   fn<<<grid, plan.block, plan.smem, stream>>>(P, b);
   return cudaGetLastError();
}

// ---------------------------------------------------------------------------- roofline denominators
namespace
{
__global__ void __launch_bounds__(256) dfma_chain_kernel(double *out, int iters, double seed)
{
   // 8 independent FMA chains per thread: enough ILP to saturate the FP64 pipe at modest occupancy
   double a0 = seed + threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
   const double m = 1.0000001, b = 1e-9;
   for (int i = 0; i < iters; i++)
   {
      a0 = fma(a0, m, b); a1 = fma(a1, m, b); a2 = fma(a2, m, b); a3 = fma(a3, m, b);
      a4 = fma(a4, m, b); a5 = fma(a5, m, b); a6 = fma(a6, m, b); a7 = fma(a7, m, b);
   }
   out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

__global__ void __launch_bounds__(256) copy_kernel(const double2 *__restrict__ src, double2 *__restrict__ dst, long long n2)
{
   const long long stride = (long long)gridDim.x * blockDim.x;
   for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += stride)
      dst[i] = src[i];
}
} // namespace

cudaError_t measure_fp64_peak(double *tflops)
{
   int dev = 0, sms = 0;
   cudaError_t e = cudaGetDevice(&dev);
   if (e != cudaSuccess) return e;
   cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
   const int blocks = sms * 8, threads = 256, iters = 1 << 15;
   double *out = nullptr;
   e = cudaMalloc(&out, sizeof(double) * blocks * threads);
   if (e != cudaSuccess) return e;
   cudaEvent_t t0, t1;
   cudaEventCreate(&t0);
   cudaEventCreate(&t1);
   double best = 0;
   for (int rep = 0; rep < 6; rep++)
   {
      cudaEventRecord(t0);
      dfma_chain_kernel<<<blocks, threads>>>(out, iters, 1.0 + rep);
      cudaEventRecord(t1);
      e = cudaEventSynchronize(t1);
      if (e != cudaSuccess) break;
      float ms = 0;
      cudaEventElapsedTime(&ms, t0, t1);
      const double flops = 2.0 * 8.0 * (double)iters * blocks * threads;
      if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
   }
   cudaEventDestroy(t0);
   cudaEventDestroy(t1);
   cudaFree(out);
   *tflops = best;
   return e;
}

// The same chain back to back for `seconds`: the rate over the second half, i.e. what the FP64 pipe delivers once the power
// management has settled (the denominator for kernels timed inside a long step; measure_fp64_peak above is the burst figure).
cudaError_t measure_fp64_sustained(double seconds, double *tflops)
{
   int dev = 0, sms = 0;
   cudaError_t e = cudaGetDevice(&dev);
   if (e != cudaSuccess) return e;
   cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
   const int blocks = sms * 8, threads = 256, iters = 1 << 15;
   double *out = nullptr;
   e = cudaMalloc(&out, sizeof(double) * blocks * threads);
   if (e != cudaSuccess) return e;
   cudaEvent_t t0, t1;
   cudaEventCreate(&t0);
   cudaEventCreate(&t1);
   // one launch is ~4.6 ms at the burst rate
   const int launches = std::max(4, (int)(seconds / 4.6e-3)), half = launches / 2;
   for (int rep = 0; rep < launches; rep++)
   {
      if (rep == half) cudaEventRecord(t0);
      dfma_chain_kernel<<<blocks, threads>>>(out, iters, 1.0 + rep);
   }
   cudaEventRecord(t1);
   e = cudaEventSynchronize(t1);
   float ms = 0;
   if (e == cudaSuccess) cudaEventElapsedTime(&ms, t0, t1);
   const double flops = 2.0 * 8.0 * (double)iters * blocks * threads * (launches - half);
   *tflops = ms > 0 ? flops / (ms * 1e-3) / 1e12 : 0.0;
   cudaEventDestroy(t0);
   cudaEventDestroy(t1);
   cudaFree(out);
   return e;
}

cudaError_t measure_hbm_peak(double *gbs)
{
   const long long bytes = 1ll << 31; // 2 GiB each way, far beyond L2
   double2 *src = nullptr, *dst = nullptr;
   cudaError_t e = cudaMalloc(&src, bytes);
   if (e != cudaSuccess) return e;
   e = cudaMalloc(&dst, bytes);
   if (e != cudaSuccess) { cudaFree(src); return e; }
   cudaMemset(src, 1, bytes);
   int dev = 0, sms = 0;
   cudaGetDevice(&dev);
   cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
   cudaEvent_t t0, t1;
   cudaEventCreate(&t0);
   cudaEventCreate(&t1);
   double best = 0;
   for (int rep = 0; rep < 6; rep++)
   {
      cudaEventRecord(t0);
      copy_kernel<<<sms * 16, 256>>>(src, dst, bytes / (long long)sizeof(double2));
      cudaEventRecord(t1);
      e = cudaEventSynchronize(t1);
      if (e != cudaSuccess) break;
      float ms = 0;
      cudaEventElapsedTime(&ms, t0, t1);
      if (rep > 0) best = std::max(best, 2.0 * bytes / (ms * 1e-3) / 1e9);
   }
   cudaEventDestroy(t0);
   cudaEventDestroy(t1);
   cudaFree(src);
   cudaFree(dst);
   *gbs = best;
   return e;
}
} // namespace mb
