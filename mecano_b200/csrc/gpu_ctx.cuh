// gpu_ctx.cuh -- the device-side context policy of the per-state routines (jointmath.cuh) and the skeleton of a
// thread-per-state block.  Included by kernels.cu (generic kernels, traversal program interpreted from the constant
// bank) and by the tree-specialised sources that specialize.cpp generates and NVRTC compiles at create() time, so it
// uses no host headers.
#pragma once
#include "algorithms.cuh"
#include "kernel_args.h"

// the dynamic shared memory of a block: [constant records (generic kernels only) | per-thread stack, state-minor | prefetch ring]
extern __shared__ double mb_smem[];

namespace mb
{
// 32-bit shared-space address of the dynamic shared memory, taken from the symbol: a constant in SASS.  Going through
// __cvta_generic_to_shared() instead makes the compiler derive every LDS/STS address from the generic window base
// (S2UR SR_CgaCtaId + 3 uniform instructions, re-materialised several times per op).
__device__ __forceinline__ unsigned mb_smem_u32()
{
   unsigned a;
   asm("mov.u32 %0, mb_smem;" : "=r"(a));
   return a;
}

// BLOCK (threads per block = stack stride) is a compile-time constant so that stack addresses are base + immediate;
// shared memory is addressed through the mb_smem symbol so that the compiler emits LDS/STS (a pointer kept in a
// struct degrades to generic LD/ST).
// Per-thread context: per-thread base pointers (one IMAD.WIDE per global access), stack of double2 (LDS.128 / STS.128)
// Tensor memory as stack space.  These kernels issue no tcgen05.mma, so the 256 KB of TMEM per SM would sit idle
// while shared memory (stack + rings) caps the resident states.  With TM > 0 the first TM double2 slots of each
// thread's stack live in TMEM instead: a warp owns the 32 lanes of its lane quarter (warp % 4) and a private range of
// columns, a double2 is four 32-bit columns, lane = thread: tcgen05.st/ld.32x32b.x4 (STTM/LDTM, scoreboarded like any
// load).  Slots >= TM stay in shared memory.  scripts/microbench/tmem_stack.cu measures the round trip.
// ROWS: rows of the prefetch ring per stage (program.h: MbAlgoInfo)
__host__ __device__ constexpr int ring_rows(int algo) { return mb_algo(algo).ring_rows; }

// handle of a constant record in shared memory (Ctx::cst): 32-bit shared address of the record
struct SmemCst
{
   unsigned a;
};
__device__ __forceinline__ void cst_ld2(const SmemCst C, int i2, double &a, double &b)
{
   // not volatile: the records are read-only once staged, so the loads may be scheduled, merged and dropped freely
   asm("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(a), "=d"(b) : "r"(C.a + 16u * (unsigned)i2));
}

// All shared-memory traffic of the per-state routines goes through ld/st.shared with explicit 32-bit addresses
// (base register + immediate in SASS).  The accesses to per-thread areas are `asm volatile` without a memory clobber:
// they stay ordered among themselves (and with the cp.async / tcgen05 statements), which is all a private stack needs.
__device__ __forceinline__ void mb_lds2(unsigned addr, double &a, double &b) { asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(a), "=d"(b) : "r"(addr)); }
__device__ __forceinline__ void mb_sts2(unsigned addr, double a, double b) { asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(addr), "d"(a), "d"(b)); }
__device__ __forceinline__ double mb_lds1(unsigned addr)
{
   double a;
   asm volatile("ld.shared.f64 %0, [%1];" : "=d"(a) : "r"(addr));
   return a;
}
// row `r` of a DoF-major buffer: base + r * ld8 as one IMAD.WIDE.U32
__device__ __forceinline__ const char *mb_row(const char *base, unsigned r, unsigned ld8)
{
   unsigned long long p;
   asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(p) : "r"(r), "r"(ld8), "l"((unsigned long long)base));
   return (const char *)p;
}

// the same for a base pointer shared by the grid plus a per-thread byte offset: base + r * ld8 stays on the uniform datapath, the
// thread adds its 32-bit offset (one IADD3 pair), and no 64-bit per-thread pointer has to be kept (or spilled) per buffer
__device__ __forceinline__ const char *mb_row_s(const char *ubase, unsigned r, unsigned ld8, unsigned s8)
{
   return (const char *)((unsigned long long)ubase + (unsigned long long)r * ld8 + s8);
}

__device__ __forceinline__ double mb_ldg(const char *p)
{
   double v;
   asm volatile("ld.global.nc.f64 %0, [%1];" : "=d"(v) : "l"(p));
   return v;
}
__device__ __forceinline__ void mb_stg(const char *p, double v) { asm volatile("st.global.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory"); }
__device__ __forceinline__ void mb_stg_cs(const char *p, double v) { asm volatile("st.global.cs.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory"); }

template <int BLOCK, int TM, int ROWS, bool M3 = false> struct GpuCtx2
{
   static constexpr bool kM3 = M3; // this instantiation handles three-DoF joints (multidof.cuh)
   // Two ways to address a row of an input / output buffer.  Per-thread 64-bit pointers (base + state), one IMAD.WIDE per access:
   // RNEA, CRBA.  Or the launch's base pointers (kernel parameters: uniform) plus this thread's state as a 32-bit byte offset, so that
   // base + row * ld stays on the uniform datapath and five 64-bit pointers per thread become one register: ABA, whose 168 registers
   // otherwise spill them (a reload in front of every prefetch).  Measured (r06n): ABA -0.7 %, RNEA +5 % -- hence per algorithm.
   static constexpr bool kUBase = ROWS == 2; // ring_rows(MB_ABA)
   static constexpr bool kFastQuat = ROWS == 2; // spatial.cuh: quat_to_rot
   const char *q0, *qd0, *x0;
   char *o0;
   unsigned s8; // (the launcher keeps n * 8 < 2^31)
   const char *qb, *qdb, *xb;
   char *ob;
   __device__ __forceinline__ const char *row_q(unsigned r) const { return kUBase ? mb_row_s(q0, r, ld8, s8) : mb_row(qb, r, ld8); }
   __device__ __forceinline__ const char *row_qd(unsigned r) const { return kUBase ? mb_row_s(qd0, r, ld8d, s8) : mb_row(qdb, r, ld8d); }
   __device__ __forceinline__ const char *row_x(unsigned r) const { return kUBase ? mb_row_s(x0, r, ld8x, s8) : mb_row(xb, r, ld8x); }
   __device__ __forceinline__ const char *row_o(unsigned r) const { return kUBase ? mb_row_s(o0, r, ld8, s8) : mb_row(ob, r, ld8); }
   const char *fb;
   unsigned ld8; // bytes between consecutive rows (the launcher keeps ld * 8 < 2^32)
   unsigned ld8d, ld8x; // the same for qd and x (0: one row of zeros stands in for every row)
   unsigned sb;  // shared address of this thread's element of shared-memory stack slot 0
   unsigned rb;  // shared address of this thread's element of stage 0, row 0 of the prefetch ring
   unsigned cb;  // shared address of the constant records
   unsigned tm0; // TMEM address (lane quarter << 16 | first column) of wide slot 0 of this warp
   unsigned wov; // kPartial: shared address such that wide slot w >= TM lives at wov + w * BLOCK * 16
   static constexpr int kBlock = BLOCK, kTM = TM;
   static constexpr bool kPartial = TM > 0 && BLOCK == MB_PARTIAL_TM_BLOCK;
   // warp-collective tcgen05.ld/st and the block barriers of specialised kernels need every thread to run every op: the
   // padding lanes of the last tile run the last state again and store the same values to the same addresses
#if defined(MB_SPEC)
   static constexpr bool kClamp = true;
#else
   static constexpr bool kClamp = TM > 0;
#endif
   // padding lanes of the last warp can be running a clamped state: kernels with a TMEM stack, and every persistent RNEA / ABA grid
   // (drawn states, thread_block_run); the mass-matrix kernels (one ring row) never draw, their stores stay unguarded
   static constexpr bool kMayClamp = kClamp || ROWS != 1;
   bool active;  // false for the padding lanes of the last tile (CRBA: they store nothing)
   double *aux; // local memory

   __device__ __forceinline__ double ld_q(int r) const { return mb_ldg(row_q((unsigned)r)); }
   __device__ __forceinline__ double ld_qd(int r) const { return mb_ldg(row_qd((unsigned)r)); }
   __device__ __forceinline__ double ld_x(int r) const { return mb_ldg(row_x((unsigned)r)); }
   __device__ __forceinline__ double ld_fext(int b, int k) const { return mb_ldg(mb_row(fb, (unsigned)(6 * b + k), ld8)); }
   // warm L2 with a row that a later op of this state reads directly (the floating base's rows: no ring in front of them)
   __device__ __forceinline__ void warm_q(int r) const { asm volatile("prefetch.global.L2 [%0];" ::"l"(row_q((unsigned)r))); }
   __device__ __forceinline__ void warm_qd(int r) const { asm volatile("prefetch.global.L2 [%0];" ::"l"(row_qd((unsigned)r))); }
   __device__ __forceinline__ void warm_x(int r) const { asm volatile("prefetch.global.L2 [%0];" ::"l"(row_x((unsigned)r))); }
   __device__ __forceinline__ void st_out(int r, double v) { mb_stg(row_o((unsigned)r), v); }
   // optional buffers of the FEXT instantiation (nullptr = absent): external wrenches in, RNEA by-products out
   char *accb, *wrb;
   const char *x2b;
   char *cmmb, *comb, *rwb;
   bool rootw_on, com_only_on;
   __device__ __forceinline__ bool has_rootw() const { return rootw_on; }
   // by-product CRBA launched without a matrix: centre of mass only (mecano_b200_center_of_mass)
   __device__ __forceinline__ bool com_only() const { return com_only_on; }
   __device__ __forceinline__ void st_cmm(int row, double v) { mb_stg(mb_row(cmmb, (unsigned)row, ld8), v); }
   // read-modify-write by the one thread that owns the state (the padding lanes of a clamped tile repeat the last state: not them)
   __device__ __forceinline__ void add_com(int r, double v)
   {
      if (!kMayClamp || active) { double *p = (double *)mb_row(comb, (unsigned)r, ld8); *p += v; }
   }
   __device__ __forceinline__ void add_rootw(int r, double v)
   {
      if (!kMayClamp || active) { double *p = (double *)mb_row(rwb, (unsigned)r, ld8); *p += v; }
   }
   __device__ __forceinline__ double ld_x2(int r) const { return mb_ldg(mb_row(x2b, (unsigned)r, ld8)); }
   bool fext_on, acc_on, wr_on;
   __device__ __forceinline__ bool has_fext() const { return fext_on; }
   __device__ __forceinline__ bool has_acc() const { return acc_on; }
   __device__ __forceinline__ bool has_wr() const { return wr_on; }
   __device__ __forceinline__ void st_acc(int b, int k, double v) { mb_stg(mb_row(accb, (unsigned)(6 * b + k), ld8), v); }
   __device__ __forceinline__ void st_wr(int b, int k, double v) { mb_stg(mb_row(wrb, (unsigned)(6 * b + k), ld8), v); }
   // ---- general stack access (CRBA; shared memory)
   __device__ __forceinline__ void stk_ld2(int slot2, int j, double &a, double &b) const { mb_lds2(sb + (unsigned)((slot2 + j) * (BLOCK * 16)), a, b); }
   __device__ __forceinline__ void stk_st2(int slot2, int j, double a, double b) { mb_sts2(sb + (unsigned)((slot2 + j) * (BLOCK * 16)), a, b); }
   // ---- split stack access (RNEA / ABA, MbOp2::wslot / nslot).  Tensor memory as stack space: these kernels issue no
   // tcgen05.mma, so the 256 KB of TMEM per SM would sit idle while shared memory caps the resident states.  With TM > 0
   // the wide area (the 6-vectors) lives in TMEM: a warp owns the 32 lanes of its lane quarter (warp % 4) and a private
   // range of columns, a double is two 32-bit columns, lane = thread: tcgen05.st/ld.32x32b.x2 (STTM/LDTM on aligned
   // register pairs, i.e. on the doubles where they are; scoreboarded like any load).  The narrow area stays in shared memory.
   __device__ __forceinline__ void acc_ld(int slot2, int wslot, double &x0, double &x1, double &x2, double &x3, double &x4, double &x5) const
   {
      if (TM > 0 && (!kPartial || wslot < TM))
      {
         const unsigned t = tm0 + 4u * (unsigned)wslot;
         unsigned r[12];
#pragma unroll
         for (int i = 0; i < 6; i++)
            asm volatile("tcgen05.ld.sync.aligned.32x32b.x2.b32 {%0, %1}, [%2];" : "=r"(r[2 * i]), "=r"(r[2 * i + 1]) : "r"(t + 2u * i));
         asm volatile("tcgen05.wait::ld.sync.aligned;"
                      : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]));
         x0 = __hiloint2double(r[1], r[0]); x1 = __hiloint2double(r[3], r[2]); x2 = __hiloint2double(r[5], r[4]);
         x3 = __hiloint2double(r[7], r[6]); x4 = __hiloint2double(r[9], r[8]); x5 = __hiloint2double(r[11], r[10]);
      }
      else
      {
         const unsigned t = TM > 0 ? wov + (unsigned)(wslot * (BLOCK * 16)) : sb + (unsigned)(slot2 * (BLOCK * 16));
         mb_lds2(t, x0, x1);
         mb_lds2(t + BLOCK * 16, x2, x3);
         mb_lds2(t + 2 * BLOCK * 16, x4, x5);
      }
   }
   __device__ __forceinline__ void acc_st(int slot2, int wslot, double x0, double x1, double x2, double x3, double x4, double x5)
   {
      if (TM > 0 && (!kPartial || wslot < TM))
      {
         const unsigned t = tm0 + 4u * (unsigned)wslot;
         const double x[6] = {x0, x1, x2, x3, x4, x5};
#pragma unroll
         for (int i = 0; i < 6; i++)
            asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(t + 2u * i), "r"(__double2loint(x[i])), "r"(__double2hiint(x[i])));
      }
      else
      {
         const unsigned t = TM > 0 ? wov + (unsigned)(wslot * (BLOCK * 16)) : sb + (unsigned)(slot2 * (BLOCK * 16));
         mb_sts2(t, x0, x1);
         mb_sts2(t + BLOCK * 16, x2, x3);
         mb_sts2(t + 2 * BLOCK * 16, x4, x5);
      }
   }
   __device__ __forceinline__ void jp_ld2(int slot2, int nslot, int j, double &a, double &b) const
   {
      mb_lds2(sb + (unsigned)((TM > 0 ? nslot + j : slot2 + 3 + j) * (BLOCK * 16)), a, b);
   }
   __device__ __forceinline__ void jp_st2(int slot2, int nslot, int j, double a, double b)
   {
      mb_sts2(sb + (unsigned)((TM > 0 ? nslot + j : slot2 + 3 + j) * (BLOCK * 16)), a, b);
   }
   // Tree-specialised kernels are straight-line code far larger than the instruction caches (L0 6 KB, L1.5 32 KB): left
   // alone, the warps of a block drift apart and each streams its own copy of the code from L2 (no_instructions was 46 %
   // of all stall samples).  A block-wide barrier every MB_SPEC_SYNC ops keeps them within a few KB of each other, so the
   // block fetches the code once.
   __device__ __forceinline__ void op_sync(int k) const
   {
#if defined(MB_SPEC) && MB_SPEC_SYNC > 0
      if (k % MB_SPEC_SYNC == 0)
         __syncthreads();
#endif
   }
   // Once per op: the tcgen05.st of earlier ops are complete before this op's tcgen05.ld (no op reads a slot it wrote itself)
   __device__ __forceinline__ void stk_fence() const
   {
      if (TM > 0)
         asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
   }
   __device__ __forceinline__ double aux_ld(int i) const { return aux[i]; }
   __device__ __forceinline__ void aux_st(int i, double v) { aux[i] = v; }
   // ABA pass-two records: global workspace of double2, one column per resident thread (coalesced 16-byte accesses),
   // read back in pass three through the ring below with cp.async (every thread reads only its own earlier stores)
   const char *ws0;   // workspace (uniform)
   unsigned ws_ld16;  // bytes between consecutive record slots (the launcher keeps the workspace below 4 GB)
   unsigned w16;      // byte offset of this thread's column
   __device__ __forceinline__ const char *rec_at(int i2) const { return mb_row_s(ws0, (unsigned)i2, ws_ld16, w16); }
   __device__ __forceinline__ void rec_st2(int i2, double a, double b) { *reinterpret_cast<double2 *>(const_cast<char *>(rec_at(i2))) = make_double2(a, b); }
   // direct read of a record slot in pass three (after pass_fence; the second half of a three-DoF joint's record, which
   // does not travel through the ring): L2 is the coherence point of the earlier stores
   __device__ __forceinline__ void rec_ld2(int i2, double &a, double &b) const
   {
      asm volatile("ld.global.cg.v2.f64 {%0, %1}, [%2];" : "=d"(a), "=d"(b) : "l"(rec_at(i2)) : "memory");
   }
   // pass-three ring: [stage][(q, qd) | rec0 .. rec2][BLOCK] double2, overlaid on the (then idle) stack area
   // MB_ABA_REC_VIA_L1 (default): the records come through L1 (cp.async.ca) instead of around it (.cg, = 0).  ncu counts 12
   // shared-memory wavefronts per LDGSTS.BYPASS.128 against 4 for the 512 contiguous bytes a warp writes -- 90 % of the kernel's
   // excess wavefronts, a quarter of all its shared-memory wavefronts; through L1 the fill arrives as whole lines: 1.5037 ->
   // 1.4925 ms, bit-identical (profiles/r06zu_shared_wavefronts.md).  A thread reads back only what it stored itself earlier
   // in program order (same SM, same L1: write-through, updated on a store hit), so the copy in L1 is never stale.
#ifndef MB_ABA_REC_VIA_L1
#define MB_ABA_REC_VIA_L1 1
#endif
   __device__ __forceinline__ void pf3_issue(int stage, int cfg, int dof, int rec2, int mask) const
   {
      const unsigned dst = sb + (unsigned)(stage * (MB_ABA_RING_ROWS * BLOCK * 16));
      if (mask & 1)
         asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(row_q((unsigned)cfg)) : "memory");
      if (mask & 2)
         asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + 8), "l"(row_qd((unsigned)dof)) : "memory");
#pragma unroll
      for (int j = 0; j < MB_ABA_REC / 2; j++)
      {
#if MB_ABA_REC_VIA_L1
         asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(dst + (1 + j) * BLOCK * 16), "l"(rec_at(rec2 + j)) : "memory");
#else
         asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + (1 + j) * BLOCK * 16), "l"(rec_at(rec2 + j)) : "memory");
#endif
      }
   }
   __device__ __forceinline__ void pf3_ld2(int stage, int row, double &a, double &b) const { mb_lds2(sb + (unsigned)((stage * MB_ABA_RING_ROWS + row) * (BLOCK * 16)), a, b); }
   // The record of a body is dead once pass three has read it: tell L2 so (discard.global.L2 drops the lines without writing
   // them back to HBM; the next tile of this thread overwrites them in full).  A warp's double2 row is four whole 128-byte lines.
   bool discard_on;
   __device__ __forceinline__ void rec_discard(int rec2) const
   {
      if (discard_on) // (set for one thread in eight: a 128-byte line holds the double2 of eight threads)
      {
#pragma unroll
         for (int j = 0; j < MB_ABA_REC / 2; j++)
            asm volatile("discard.global.L2 [%0], 128;" ::"l"(rec_at(rec2 + j)) : "memory");
      }
   }
   __device__ __forceinline__ void pass_fence() const { __threadfence(); }
#if defined(MB_SPEC)
   // tree-specialised kernels: the constant records are literals in the generated source (constant-bank operands)
   __device__ __forceinline__ const double *cst(int b) const { return mb_spec_consts + b * MB_CONST_STRIDE; }
#else
   __device__ __forceinline__ SmemCst cst(int b) const { return SmemCst{cb + (unsigned)(b * (MB_CONST_STRIDE * 8))}; }
#endif
   // mass matrix: entry e = row * nv + col lives at mbase + e * mstride (entry-major: mstride = ld8; state-major: 8)
   char *mbase;
   unsigned mstride;
   int nv;
   const uint4 *zlist;
   int nz8;
   __device__ __forceinline__ int n_dofs() const { return nv; }
   __device__ __forceinline__ void st_M(int e, double v) const
   {
      if (!kMayClamp || active)
         mb_stg_cs(mb_row(mbase, (unsigned)e, mstride), v);
   }
   char *corb; // Coriolis matrix (MB_CORIOLIS), entry-major; joint efforts (MB_GRAVITY_GRADIENT); d tau / dqd (MB_RNEA_DERIVATIVES)
   __device__ __forceinline__ void st_C(int e, double v) const
   {
      if (!kMayClamp || active)
         mb_stg_cs(mb_row(corb, (unsigned)e, ld8), v);
   }
   // gravity gradient (MB_GRAVITY_GRADIENT): the joint efforts tau_g, row r of `cor` (kernel_args.h); G goes through st_M
   __device__ __forceinline__ void st_tau(int r, double v) const
   {
      if (!kMayClamp || active)
         mb_stg(mb_row(corb, (unsigned)r, ld8), v);
   }
   // inverse-dynamics derivatives (MB_RNEA_DERIVATIVES): the joint efforts tau, row r of `root_wrench` (kernel_args.h); d tau / dq goes
   // through st_M, d tau / dqd through st_C
   __device__ __forceinline__ void st_jtau(int r, double v) const
   {
      if (!kMayClamp || active)
         mb_stg(mb_row(rwb, (unsigned)r, ld8), v);
   }
   __device__ __forceinline__ void zero_fill_mc_part(int k, int parts) const
   {
      const int k1 = min(nz8, (k + 1) * parts);
#pragma unroll 1
      for (int i = k * parts; i < k1; i++)
      {
         const uint4 u = __ldg(zlist + i);
         const unsigned e[8] = {u.x & 0xffffu, u.x >> 16, u.y & 0xffffu, u.y >> 16, u.z & 0xffffu, u.z >> 16, u.w & 0xffffu, u.w >> 16};
#pragma unroll
         for (int j = 0; j < 8; j++)
         {
            st_M((int)e[j], 0.0);
            st_C((int)e[j], 0.0);
         }
      }
   }
   // the zero list in `parts`-sized groups of eight entries, one group range per op of the traversal
   __device__ __forceinline__ int zero_parts(int nops) const { return (nz8 + nops - 1) / nops; }
   __device__ __forceinline__ void zero_fill_part(int k, int parts) const
   {
      const int k1 = min(nz8, (k + 1) * parts);
#pragma unroll 1
      for (int i = k * parts; i < k1; i++)
      {
         const uint4 u = __ldg(zlist + i);
         st_M(u.x & 0xffffu, 0.0); st_M(u.x >> 16, 0.0); st_M(u.y & 0xffffu, 0.0); st_M(u.y >> 16, 0.0);
         st_M(u.z & 0xffffu, 0.0); st_M(u.z >> 16, 0.0); st_M(u.w & 0xffffu, 0.0); st_M(u.w >> 16, 0.0);
      }
   }
   __device__ __forceinline__ void zero_fill() const
   {
#pragma unroll 1
      for (int k = 0; k < nz8; k++)
      {
         const uint4 u = __ldg(zlist + k);
         st_M(u.x & 0xffffu, 0.0); st_M(u.x >> 16, 0.0); st_M(u.y & 0xffffu, 0.0); st_M(u.y >> 16, 0.0);
         st_M(u.z & 0xffffu, 0.0); st_M(u.z >> 16, 0.0); st_M(u.w & 0xffffu, 0.0); st_M(u.w >> 16, 0.0);
      }
   }
   // prefetch ring: [stage][q | qd | x][BLOCK] doubles in shared memory, filled by cp.async (LDGSTS)
   // mask: 1 = q[cfg], 2 = qd[dof], 4 = x[dof]
   __device__ __forceinline__ void pf_issue(int stage, int cfg, int dof, int mask) const
   {
      const unsigned dst = rb + (unsigned)(stage * (ROWS * BLOCK * 8));
      if (mask & 1)
         asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(row_q((unsigned)cfg)) : "memory");
      if (mask & 2)
         asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + BLOCK * 8), "l"(row_qd((unsigned)dof)) : "memory");
      if (mask & 4)
         asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst + (ROWS == 3 ? 2 : 0) * BLOCK * 8), "l"(row_x((unsigned)dof)) : "memory");
   }
   __device__ __forceinline__ void pf_commit() const { asm volatile("cp.async.commit_group;" ::: "memory"); }
   template <int N> __device__ __forceinline__ void pf_wait() const { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
   __device__ __forceinline__ double pf_ld(int stage, int j) const { return mb_lds1(rb + (unsigned)((stage * ROWS + ((j == 2 && ROWS < 3) ? 0 : j)) * (BLOCK * 8))); }
   // joint-torque regressor (MB_REGRESSOR): entry e = row * 10 nb + col of Y at mbase + e * ld8, streamed past L2 like the mass matrix
   const uint32_t *yzrows; // structurally zero rows: entry of the row's first column
   int nyz;
   __device__ __forceinline__ void st_Y(int e, double v) const
   {
      if (!kMayClamp || active)
         mb_stg_cs(mb_row(mbase, (unsigned)e, ld8), v);
   }
   __device__ __forceinline__ int y_zero_parts(int nops) const { return (nyz + nops - 1) / nops; }
   __device__ __forceinline__ void y_zero_fill_part(int k, int parts) const
   {
      const int k1 = min(nyz, (k + 1) * parts);
#pragma unroll 1
      for (int i = k * parts; i < k1; i++)
      {
         const int e = (int)__ldg(yzrows + i);
#pragma unroll
         for (int j = 0; j < 10; j++)
            st_Y(e + j, 0.0);
      }
   }
};

// columns of tensor memory one warp owns when BLOCK / 32 warps share the four lane quarters
__host__ __device__ constexpr int tm_warp_cols(int block) { return (512 / ((block + 127) / 128)) & ~3; }
static_assert(MB_PARTIAL_TM_BLOCK == 640, "kCfg / tm_warp_cols assume 20 warps for the partial-TMEM block");

// Skeleton of a block: TMEM allocation, context set-up, the loop over tiles of BLOCK states; `body(ctx)` evaluates one
// state.  ncst = doubles of constant records staged at the front of shared memory (0 for specialised kernels),
// stack2 = stack slots (double2) per state.
template <int ALGO, bool STATE_MAJOR, int BLOCK, int AUXN, int TM, bool M3 = false, class Body>
__device__ __forceinline__ void thread_block_run(const KernelArgs &a, const int ncst, const int smem_slots, const int nstack2, Body body)
{
   static_assert(TM * 4 <= tm_warp_cols(BLOCK), "TMEM stack slots exceed the columns of one warp");
   static_assert(TM == 0 || mb_algo(ALGO).wide_stack, "a kernel without a wide stack area keeps its stack in shared memory");
   __shared__ unsigned tm_base_s;
   if (TM > 0)
   {
      // one warp allocates all 512 columns for the block (the launcher guarantees one resident block per SM for TM > 0)
      if (threadIdx.x < 32)
      {
         asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"((unsigned)__cvta_generic_to_shared(&tm_base_s)) : "memory");
         asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
      }
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
   }
   __syncthreads(); // also publishes the constant records staged by the caller
   if (TM > 0)
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
   double aux[AUXN > 0 ? AUXN : 1];
   GpuCtx2<BLOCK, TM, ring_rows(ALGO), M3> c2;
   c2.ld8 = (unsigned)(a.ld * 8);
   c2.ld8d = (unsigned)(a.ld_qd * 8);
   c2.ld8x = (unsigned)(a.ld_x * 8);
   // mb_smem_u32() names the symbol in inline PTX only: one (never executed) C++ reference makes sure it is declared in
   // the module even when nothing else touches it (tree-specialised kernels stage no constant records)
   if (a.n < 0)
      mb_smem[0] = 0.0;
   // [constant records | stack: smem_slots x BLOCK double2 (mb_smem_stack_slots) | prefetch ring]
   c2.cb = mb_smem_u32();
   c2.sb = c2.cb + 8u * (unsigned)((ncst + 1) & ~1) + 16u * threadIdx.x;
   c2.rb = c2.cb + 8u * (unsigned)(((ncst + 1) & ~1) + 2 * smem_slots * BLOCK) + 8u * threadIdx.x;
   c2.tm0 = 0;
   c2.wov = c2.sb + (unsigned)((nstack2 - TM) * (BLOCK * 16));
   if (TM > 0)
   {
      const unsigned warp = threadIdx.x >> 5;
      c2.tm0 = tm_base_s + (((warp & 3u) * 32u) << 16) + (warp >> 2) * (unsigned)tm_warp_cols(BLOCK);
      // warp-uniform by construction; the shuffle lets ptxas keep it (and the per-op addresses derived from it) in uniform registers
      c2.tm0 = __shfl_sync(0xffffffffu, c2.tm0, 0);
   }
   c2.active = true;
   c2.fext_on = a.fext != nullptr; c2.acc_on = a.body_acc != nullptr; c2.wr_on = a.joint_wrench != nullptr; c2.rootw_on = a.root_wrench != nullptr;
   c2.com_only_on = ALGO == MB_CRBA && a.out == nullptr;
   c2.aux = aux;
   c2.nv = a.nv;
   c2.mstride = STATE_MAJOR ? 8u : c2.ld8;
   c2.zlist = (const uint4 *)a.zero_entries;
   c2.nz8 = a.n_zero >> 3;
   c2.ws0 = reinterpret_cast<const char *>(a.ws);
   c2.w16 = (blockIdx.x * BLOCK + threadIdx.x) * 16u;
   c2.ws_ld16 = (unsigned)(a.ws_ld * 16);
   c2.q0 = (const char *)a.q; c2.qd0 = (const char *)a.qd; c2.x0 = (const char *)a.x; c2.o0 = (char *)a.out;
   c2.discard_on = ALGO == MB_ABA && (a.flags & MB_KFLAG_ABA_DISCARD) != 0 && (threadIdx.x & 7u) == 0;
   // The warps of a block start together and run the same op sequence; MECANO_B200_STAGGER_NS starts slot j of a scheduler
   // (warp / 4) j * stagger_ns late.  Measured: no effect (profiles/r06d_plain_kinds.md), the warps are not marching in phase.
   if (a.stagger_ns > 0)
      __nanosleep((threadIdx.x >> 7) * (unsigned)a.stagger_ns);
   // Work distribution.  One block per tile of BLOCK states, or -- persistent grids (TMEM stack, ABA workspace) -- every warp
   // draws the next 32 states from a counter (a.work_counter, zeroed by the launcher).  Drawing keeps the states in flight one
   // compact, advancing stretch of every row however far the warps drift apart (a static round-robin over tiles lets slow blocks
   // fall rounds behind; contiguous ranges per block -- 148 streams 57 KB apart in every row -- measured 10-12 % slower), and it
   // ends without a partial last round (2^20 states are 18.45 rounds of 148 tiles of 384: 81 SMs idle during the last one).
   // The per-state areas (stack, rings) are private to a thread and the constant records are read-only, so the threads of a block
   // never synchronise again.
   const long long ntiles = (a.n + BLOCK - 1) / BLOCK;
   using C2 = GpuCtx2<BLOCK, TM, ring_rows(ALGO), M3>;
   auto run_state = [&](long long s) {
      c2.s8 = (unsigned)s * 8u;
      c2.qb = (const char *)(a.q + s); c2.qdb = (const char *)(a.qd + s); c2.xb = (const char *)(a.x + s); c2.ob = (char *)(a.out + s);
      c2.fb = (const char *)(a.fext + s);
      c2.accb = (char *)(a.body_acc + s); c2.wrb = (char *)(a.joint_wrench + s);
      c2.x2b = (const char *)(a.x2 + s);
      c2.corb = (char *)(a.cor + s);
      c2.cmmb = (char *)(a.cmm + s); c2.comb = (char *)(a.com + s); c2.rwb = (char *)(a.root_wrench + s);
      c2.mbase = STATE_MAJOR ? (char *)(a.out + s * (long long)a.nv * a.nv) : (char *)(a.out + s);
      body(c2);
   };
   if constexpr (!C2::kMayClamp)
   {
      // the mass-matrix kernels (shared-memory stack, one block per tile): the plain loop they have had since round 1 -- at 255
      // registers the Coriolis kernel pays 16 % for any other shape of it (80 more bytes of spills, r06za)
      for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
      {
         const long long s = tile * BLOCK + threadIdx.x;
         if (s >= a.n)
            break;
         run_state(s);
      }
   }
   else
   {
      long long tile = blockIdx.x;
      for (;;)
      {
         long long s;
         const long long hi = a.n;
         if (a.work_counter != nullptr)
         {
            unsigned first = 0;
            if ((threadIdx.x & 31) == 0)
               first = atomicAdd(a.work_counter, 32u);
            first = __shfl_sync(0xffffffffu, first, 0);
            if ((long long)first >= hi)
            {
               // the last warp of the grid to run dry re-arms the counter pair for the next launch (no memset between launches)
               if ((threadIdx.x & 31) == 0 && atomicAdd(a.work_counter + 1, 1u) == gridDim.x * (BLOCK / 32) - 1)
               {
                  a.work_counter[0] = 0;
                  a.work_counter[1] = 0;
               }
               break;
            }
            s = (long long)first + (threadIdx.x & 31);
         }
         else
         {
            if (tile >= ntiles)
               break;
            s = tile * BLOCK + threadIdx.x;
            tile += gridDim.x;
         }
         // (every exit of this loop above is warp-uniform and visibly so -- a kernel parameter, the block index, a value shuffled
         // from lane 0: with a thread-dependent exit ptxas gives up the uniform datapath for the whole traversal, +12 % on RNEA / ABA)
         if (C2::kClamp || a.work_counter != nullptr)
         {
            // tcgen05.ld/st and the draw above are warp-collective: the padding lanes of the last warp run a clamped state (and
            // store nothing, or the same values to the same addresses) instead of leaving the loop on their own
            c2.active = s < hi;
            s = s < hi ? s : hi - 1;
         }
         else if (s >= hi)
            break;
         run_state(s);
      }
   }
   if (TM > 0)
   {
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncthreads();
      if (threadIdx.x < 32)
         asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tm_base_s) : "memory");
   }
}
} // namespace mb
