// program.h -- the flattened tree as the kernels see it: per-body constant records (staged in shared
// memory) and a depth-first "traversal program" (kernel parameter => constant bank).
//
// One thread evaluates one state by executing the program: DESCEND(i) ops propagate kinematics from
// the parent to body i, ASCEND(i) ops run once the whole subtree of i is finished and fold the
// subtree's force / inertia into the parent.  Interleaving the two sweeps this way means the data
// that must survive between them only has to be kept for the bodies on the current root-to-leaf
// path (a stack as deep as the tree) instead of for every body, which is what lets the per-state
// working set live in shared memory (DESIGN.md, "working set").
//
// Internal frames: every 1-DoF joint frame is re-expressed at flatten time so that the joint axis is
// the local z axis (a constant rotation Q_i absorbed into the fixed offsets and inertias).  Joint
// scalars (q, qd, qdd, tau) are invariant under this; SixDoF joints keep Q = identity so that their
// 6-vectors stay in Mecano's frameAfterJoint.
#pragma once
#if defined(__CUDACC_RTC__)
// NVRTC (tree-specialised kernels, jit.cpp) has no host headers
typedef unsigned char uint8_t;
typedef unsigned short uint16_t;
typedef unsigned int uint32_t;
typedef int int32_t;
typedef long long int64_t;
#else
#include <stdint.h>
#endif

#define MB_MAX_BODIES 128
#define MB_MAX_OPS (2 * MB_MAX_BODIES)

// joint types (after canonicalisation the 1-DoF axis is always +z)
#define MB_REVOLUTE 0
#define MB_PRISMATIC 1
#define MB_SIXDOF 2 // also the class of the other multi-DoF joints, told apart by their sub-type:
// sub-type of a multi-DoF joint: which components of the 6-vector [wx wy wz vx vy vz] in frameAfterJoint are its DoFs
#define MB_SUB_SIX 0       // SixDoFJoint: all six; configuration [qx qy qz qs x y z]
#define MB_SUB_SPHERICAL 1 // SphericalJoint: (wx wy wz); configuration [qx qy qz qs]
#define MB_SUB_PLANAR 2    // PlanarJoint: (wy vx vz); configuration [pitch x z]

// per-body constant record, in doubles
#define MB_C_R 0    // [9] row-major rotation of the joint's zero-configuration frame in the parent frame
#define MB_C_P 9    // [3] translation of the same
#define MB_C_I 12   // [6] inertia about the frame origin: xx xy xz yy yz zz
#define MB_C_H 18   // [3] first moment h = m * c
#define MB_C_M 21   // [1] mass
#define MB_C_E 22   // [9] rotation CoM frame -> internal frame (for external wrenches)
#define MB_C_C 31   // [3] CoM position in the internal frame
#define MB_C_J 34   // [6] inertia about the CoM, expressed in the internal frame: xx xy xz yy yz zz
#define MB_C_Q 40   // [9] rotation internal (canonical) frame -> the joint's frameAfterJoint (per-joint outputs in Mecano's frame)
#define MB_CONST_STRIDE 50

// op word: bit0 kind, bits 1..7 flags, bits 8..23 body
#define MB_OP_ASCEND 0x1u
#define MB_F_LEAF 0x2u         // body has no children (DESCEND keeps its data in registers; ASCEND follows immediately)
#define MB_F_LOAD_PARENT 0x4u  // DESCEND: the parent's kinematic state must be reloaded (a sibling subtree ran in between)
#define MB_F_SAVE_STATE 0x8u   // DESCEND: body has >= 2 children, save its kinematic state for the later ones
#define MB_F_ROOT_PARENT 0x10u // the parent is the root body
#define MB_F_STORE_ACC 0x20u   // ASCEND: more siblings follow, write the parent's accumulator back
#define MB_F_FIRST_CHILD 0x40u // ASCEND: first finished child of the parent (accumulator starts from the parent's own term)
#define MB_OP_BODY(w) (((w) >> 8) & 0xffffu)

struct MbBody
{
   int32_t parent;      // internal index, -1 = root body
   int32_t jtype;
   int32_t dof_off;     // Mecano DoF row of the first DoF
   int32_t cfg_off;     // Mecano configuration row
   int32_t slot;        // base of this body's stack slot (doubles), shared-memory stack
   int32_t aux;         // base of this body's branch save area (doubles), local memory; -1 if none
   int32_t rec;         // three-DoF joints: where the second half of the ABA pass-three record lives (double2 units), else -1
   int32_t subtree_end; // one past the last internal index of this body's subtree
   int32_t ext_index;   // index of this body in the caller's tree description (external wrench rows)
   int32_t depth;
   int32_t ndof;
   int32_t sub;         // MB_SUB_* of a multi-DoF joint (jtype == MB_SIXDOF), else 0
};

// Pre-decoded traversal record (28 bytes): everything an op needs, so that the kernels never
// chase MbBody fields.  Stack offsets are in double2 units (the shared-memory stack is an array of double2,
// state-minor), save-area offsets in doubles.
//   code: bit0 ASCEND, bits1-2 joint type, bit3 SC (this op also evaluates sin/cos for the next 1-DoF DESCEND),
//         bits4-5 sub-type of a multi-DoF joint (MB_SUB_*)
struct MbOp2
{
   uint8_t code;
   uint8_t flags;   // MB_F_* >> 1  (LEAF 0x1, LOAD_PARENT 0x2, SAVE_STATE 0x4, ROOT_PARENT 0x8, STORE_ACC 0x10, FIRST_CHILD 0x20)
   uint8_t body;    // internal body index (constant record)
   uint8_t pf;      // MB2_PF_*: what this op does for the ops ahead of it in the software pipeline
   uint16_t cfg, dof;    // Mecano configuration / DoF row of the joint
   uint16_t slot, pslot; // own / parent stack slot (double2 units)
   uint16_t aux, paux;   // own / parent save area (doubles)
   // split view of the same slot (RNEA / ABA): its first three double2 (the 6-vector that is read back and accumulated)
   // counted in a "wide" area, the rest (sin/cos or a SixDoF transform) in a "narrow" one.  A context may place the two
   // areas in different memories (tensor memory / shared memory) and still address them without a run-time test.
   uint16_t wslot, pwslot; // own / parent index in the wide area (double2 units)
   uint16_t nslot;         // own index in the narrow area (double2 units)
   uint16_t pfbody;        // body of op k + MB_PF_DIST (ABA pass three: its pass-two record)
   uint16_t pfcfg, pfdof;  // configuration / DoF row of op k + MB_PF_DIST (requested during this op)
};
#define MB2_PF_NEXT1 0x1u // op k+1 is a 1-DoF DESCEND (its configuration is read from the prefetch ring during this op)
#define MB2_PF_D1 0x2u    // op k + MB_PF_DIST is a 1-DoF DESCEND
#define MB2_PF_A1 0x4u    // op k + MB_PF_DIST is a 1-DoF ASCEND
#define MB2_ASCEND 0x1u
#define MB2_JT(code) (((code) >> 1) & 3u)
#define MB2_SUB(code) (((code) >> 4) & 3u)
#define MB2_SC 0x8u
#define MB2_LEAF 0x1u
#define MB2_LOAD_PARENT 0x2u
#define MB2_SAVE_STATE 0x4u
#define MB2_ROOT_PARENT 0x8u
#define MB2_STORE_ACC 0x10u
#define MB2_FIRST_CHILD 0x20u
#define MB2_ACCSRC 0x40u // ABA ASCEND and pass-three records: the joint is an ACCELERATION_SOURCE (mecano_b200_set_joint_source_modes); not part of MB_F_*

// per-body record for the CRBA ancestor walk (16 bytes; the first eight are what the dense layouts read, one aligned 64-bit load)
struct MbWalk
{
   uint8_t jtype;
   uint8_t flags;  // bit0: the parent is the root body
   uint8_t parent; // internal index of the parent body
   uint8_t above;  // packed mass-matrix layout: DoFs of the proper ancestors of this body = position of this joint's first DoF
                   // within a packed column (the non-zero rows of a column are the DoFs on the path from the root, root first)
   uint16_t dof;   // Mecano DoF row
   uint16_t slot;  // stack slot (double2 units)
   uint16_t pcol;  // packed mass-matrix layout: first packed row of the column of this joint's first DoF; the column of its
                   // r-th DoF starts at pcol + r * above + r (r + 1) / 2 and holds above + r + 1 entries
   uint16_t sub;   // MB_SUB_* of a multi-DoF joint
   uint32_t pad2;
};

// A run: consecutive ops of the same kind (code & 0xf: ASCEND bit, joint type, SC bit).  The kernels execute a run as one
// tight loop over a routine specialised on the kind, instead of dispatching every op through a switch: the loop-carried
// spatial quantities then stay in the same registers from op to op (the per-op switch cost ~40 register moves per op).
// MB_RUN_PLAIN: all ops of the run carry the flags of the common case of their kind (and no one-DoF DESCEND follows unless the SC
// bit says so), which the run loops then treat as compile-time constants.  Only for the kinds mb_run_has_plain() names.
#define MB_RUN_PLAIN 0x10u
// which kinds have a plain form (bit masks; every plain loop body is more hot code for the instruction caches, see DESIGN.md):
// RNEA 1 DESCEND of a leaf, 2 ASCEND, 4 DESCEND with SC;  ABA 1 DESCEND of a leaf, 2 ASCEND, 4 DESCEND with SC, 8 pass three
// Measured on 2^20 H37 states (profiles/r06d_plain_kinds.md): RNEA ASCEND -1.4 %; the RNEA DESCEND forms are neutral or slower
// (code placement), and every ABA form is slower (+1 ... +18 %: the hot loops of ABA already fill the 32 KB instruction cache).
#ifndef MB_PLAIN_RNEA
#define MB_PLAIN_RNEA 2
#endif
#ifndef MB_PLAIN_ABA
#define MB_PLAIN_ABA 0
#endif
// whether the ABA DESCEND runs are split by the SC bit (sin/cos of the next joint evaluated inside the op's basic block): 1, or
// tested at run time like in its ASCEND runs (one loop body less): 0
// Measured (r06o, 2^20 H37 states): 1.575 -> 1.550 ms without the split -- once pass three had lost its sin/cos (records), one loop body
// less is worth more to ABA than the overlap of the sin/cos chain with the twist propagation.
#ifndef MB_ABA_D_SC_SPLIT
#define MB_ABA_D_SC_SPLIT 0
#endif
// the same switch for RNEA (all its runs)
#ifndef MB_RNEA_SC_SPLIT
#define MB_RNEA_SC_SPLIT 1
#endif
// the flags a kind tests (rnea.cuh / aba.cuh), 0 if the kind has no plain form.  kind = MbOp2::code & 0xf; pass3: ABA pass-three list.
// Plain forms exist for revolute joints: the DESCEND of an interior body (SC set: the next joint of the chain is revolute too), the
// DESCEND of a leaf (no SC: its own ASCEND follows) and the ASCEND of an interior body with a single child.
#if defined(__CUDACC__)
__host__ __device__
#endif
static inline unsigned mb_run_plain_tested(int algo, int kind, bool pass3)
{
   if (algo == 0 /* MB_RNEA */)
   {
      if (kind == 0 && (MB_PLAIN_RNEA & 1)) return MB2_LEAF | MB2_LOAD_PARENT | MB2_SAVE_STATE | MB2_ROOT_PARENT;
      if (kind == 1 && (MB_PLAIN_RNEA & 2)) return MB2_LEAF | MB2_ROOT_PARENT | MB2_STORE_ACC;
      if (kind == 8 && (MB_PLAIN_RNEA & 4)) return MB2_LEAF | MB2_LOAD_PARENT | MB2_SAVE_STATE | MB2_ROOT_PARENT;
   }
   if (algo == 1 /* MB_ABA */)
   {
      if (pass3)
         return (kind == 0 && (MB_PLAIN_ABA & 8)) ? (MB2_ROOT_PARENT | MB2_LOAD_PARENT | MB2_SAVE_STATE | MB2_ACCSRC) : 0u;
      if ((kind == 0 && (MB_PLAIN_ABA & 1)) || (kind == 8 && (MB_PLAIN_ABA & 4))) return MB2_LEAF | MB2_LOAD_PARENT | MB2_ROOT_PARENT;
      if (kind == 1 && (MB_PLAIN_ABA & 2)) return MB2_LEAF | MB2_ROOT_PARENT | MB2_FIRST_CHILD | MB2_STORE_ACC | MB2_ACCSRC;
   }
   return 0u;
}
// MbOp2::flags of a plain op (bits outside mb_run_plain_tested are don't-cares)
#if defined(__CUDACC__)
__host__ __device__
#endif
static inline unsigned mb_run_plain_flags(int algo, int kind, bool pass3)
{
   (void)algo;
   if (pass3)
      return 0u;
   return kind == 0 ? MB2_LEAF : (kind == 1 ? MB2_FIRST_CHILD : 0u);
}
// whether the kind says if a one-DoF DESCEND follows (SC bit part of the kind; ABA keeps it out of its ASCEND kinds)
#if defined(__CUDACC__)
__host__ __device__
#endif
static inline bool mb_run_kind_has_sc(int algo, int kind, bool pass3)
{
   if (algo == 0 /* MB_RNEA */)
      return MB_RNEA_SC_SPLIT != 0;
   return !(algo == 1 /* MB_ABA */ && (pass3 || (kind & MB2_ASCEND) || !MB_ABA_D_SC_SPLIT));
}
struct MbRun
{
   uint8_t kind; // MbOp2::code & 0xf | MB_RUN_PLAIN
   uint8_t n;    // number of ops
   uint16_t k0;  // first op
};

struct MbProgram
{
   int32_t nb, nops, nv, nq;
   int32_t nruns, nruns3;
   int32_t wstack2, nstack2; // sizes of the wide / narrow stack areas per state (double2 units), see MbOp2
   int32_t stack2;        // v2 stack size per state in double2 units
   int32_t stack_doubles; // shared-memory stack per state
   int32_t aux_doubles;   // local-memory branch save area per state
   int32_t rec_doubles;   // local-memory record area per state (ABA)
   int32_t max_depth;
   MbBody body[MB_MAX_BODIES];
   uint32_t op[MB_MAX_OPS];
   MbWalk walk[MB_MAX_BODIES];
   MbRun run[MB_MAX_OPS];        // runs of op2
   MbRun run3[MB_MAX_BODIES];    // runs of op3
   MbOp2 op3[MB_MAX_BODIES + 4]; // ABA pass three: the DESCEND records only, with their own SC / pf look-ahead bits
   MbOp2 op2[MB_MAX_OPS + 4]; // trailing no-op records so that the look-ahead never reads past the end
};

// stack slot sizes (doubles) per algorithm: joint parameters needed to rebuild the joint transform
// on the way up: revolute (sin, cos), prismatic (q), SixDoF (R[9], p[3])
#if defined(__CUDACC__)
__host__ __device__
#endif
static inline int mb_jp_size(int jtype) { return jtype == MB_REVOLUTE ? 2 : (jtype == MB_PRISMATIC ? 1 : 12); }
#if defined(__CUDACC__)
__host__ __device__
#endif
static inline int mb_sub_ndof(int sub) { return sub == MB_SUB_SIX ? 6 : 3; }

// ABA pass-three record of one body, in doubles (four double2).  One-DoF joint: g = U / D without its component along the joint
// axis (which is D / D = 1), k0 = u / D, and the sin/cos of the joint angle (prismatic: q, 1) so that pass three neither reads q nor
// evaluates sin/cos again: revolute (g.ax, g.ay, g.lx, g.ly, g.lz, k0, s, c), prismatic (g.ax, g.ay, g.az, g.lx, g.ly, k0, q, 1).
// SixDoF joint: the six accelerations (last double2 unused, written as zeros).  An ACCELERATION_SOURCE joint stores its given
// acceleration (k0 / the six) and is recognised in pass three by the MB2_ACCSRC flag of its op.
#define MB_ABA_REC 8
#define MB_ABA_RING_ROWS (1 + MB_ABA_REC / 2) // pass-three ring, double2 rows per stage: (-, qd) + the record

// MB_CORIOLIS: mass matrix + Coriolis matrix (coriolis.cuh); MB_REGRESSOR: joint-torque regressor (regressor.cuh);
// MB_GRAVITY_GRADIENT: gravity torques and their configuration gradient (gravity_gradient.cuh); MB_RNEA_DERIVATIVES: joint efforts
// and their derivatives in q and qd (rnea_derivatives.cuh)
enum MbAlgo { MB_RNEA = 0, MB_ABA = 1, MB_CRBA = 2, MB_CORIOLIS = 3, MB_REGRESSOR = 4, MB_GRAVITY_GRADIENT = 5, MB_RNEA_DERIVATIVES = 6 };
#define MB_NUM_ALGOS 7

// What the flattener, the planner, the launcher and the C ABI need to know about a thread-per-state algorithm (mb_algo).
struct MbAlgoInfo
{
   const char *cfg_key; // its key in MECANO_B200_CFG (kernels.cu: forced_cfg)
   int aux;             // branch save area per nested branching body (doubles, local memory; thread_kernels.cuh: aux_of)
   bool wide_stack;     // the stack is split into a wide area, which may live in tensor memory, and a narrow one (MbOp2); without
                        // it the whole stack is in shared memory and the TMEM configurations are never planned
   bool thread_only;    // the generic thread-per-state kernel is its only form (no warp, team, tree-specialised or fp32 kernel);
                        // when it does not fit, only its own entry point fails, not the handle
   int ring_rows;       // double2 rows per stage of the prefetch ring (gpu_ctx.cuh)
   int spill_bytes;     // local memory beyond the work area that the planner accepts before it counts the kernel as spilling
   bool small_blocks;   // planner tie-break: more, smaller blocks win, as hardware block scheduling evens out the store bursts
                        // of the store-bound matrix kernels (Coriolis, H37: 2 x 128 threads 5.89 ms, 1 x 256 6.54 ms,
                        // profiles/r02h_cor_sweep.jsonl; CRBA, 4 x 128 against 2 x 256 threads: 7 / 15 / 25 / 32 / 51 bodies
                        // -2.9 / -8.4 / -0.8 / -1.4 / -4.3 %, profiles/r03g_crba_block_sweep.jsonl)
   int io_nq, io_nv, io_nv2, io_nbnv; // kernel_info bytes per state / 8: per configuration row, DoF, nv x nv and nb x nv entry
                                      // (SURVEY.md 8(d); a call with external wrenches reads 48 n_bodies bytes more)
};
#if defined(__CUDACC__)
__host__ __device__
#endif
static constexpr MbAlgoInfo mb_algo(int algo)
{
   switch (algo)
   {
      // aux: twist + spatial acceleration of a branching body; ring: q, qd, qdd
      case MB_RNEA: return {"rnea", 12, true, false, 3, 128, false, 1, 3, 0, 0};
      // aux: articulated inertia (6 + 9 + 6) + bias wrench (6), reused for (v, a) in pass three; ring: q | tau, qd (an op never
      // needs q and tau together)
      case MB_ABA: return {"aba", 27, true, false, 2, 128, false, 1, 3, 0, 0};
      // aux: composite inertia (6 + 3 + 1); ring: q
      case MB_CRBA: return {"crba", 10, false, false, 1, 128, true, 1, 0, 1, 0};
      // aux: composite inertia (10) + composite factorized inertia (4 x 9); spills: with two 46-double accumulators and three
      // force columns live, a few hundred bytes are its normal state at 255 registers
      case MB_CORIOLIS: return {"cor", 46, false, true, 1, 512, true, 1, 1, 2, 0};
      case MB_REGRESSOR: return {"reg", 12, false, true, 1, 128, true, 1, 2, 0, 10}; // aux: twist + spatial acceleration
      case MB_GRAVITY_GRADIENT: return {"gg", 16, false, true, 1, 128, true, 1, 1, 1, 0}; // aux: composite inertia (10) + external wrench (6)
      // aux: composite inertia (10), factorized inertia (4 x 9), momentum (6), RNEA force (6); spills: some 670 bytes, with four
      // accumulators of 58 doubles and four force columns live
      case MB_RNEA_DERIVATIVES: return {"rd", 58, false, true, 1, 768, true, 1, 3, 2, 0};
   }
   return {}; // not an algorithm
}

// Shared-memory stack slots (double2 per state) of a thread-per-state block.  With a tensor-memory stack (tm > 0 slots,
// wide-stack algorithms) the wide area lives in TMEM and only the narrow one in shared memory.  ABA overlays its pass-three
// ring (4 stages x MB_ABA_RING_ROWS rows) on the stack area.
#if defined(__CUDACC__)
__host__ __device__
#endif
static inline int mb_smem_stack_slots(int algo, const MbProgram &P, int tm)
{
   int s = P.stack2;
   if (tm > 0 && mb_algo(algo).wide_stack)
      s = P.nstack2 + (P.wstack2 > tm ? P.wstack2 - tm : 0); // wide slots beyond the TMEM share spill over behind the narrow area
   if (algo == MB_ABA && s < 4 * MB_ABA_RING_ROWS)
      s = 4 * MB_ABA_RING_ROWS; // the pass-three ring (4 stages) is overlaid on the stack area
   return s < 1 ? 1 : s;
}
// Blocks of MB_PARTIAL_TM_BLOCK threads (20 warps: five per TMEM lane quarter, 100 columns each) hold the first tm wide slots
// in tensor memory and the deeper ones in shared memory, chosen per access by a warp-uniform test; all other block sizes
// require the whole wide area to fit so that the test folds away at compile time.
#define MB_PARTIAL_TM_BLOCK 640
#if defined(__CUDACC__)
__host__ __device__
#endif
static inline bool mb_tm_fits(int algo, const MbProgram &P, int tm, int block)
{
   return tm == 0 || (mb_algo(algo).wide_stack && (P.wstack2 <= tm || block == MB_PARTIAL_TM_BLOCK));
}
