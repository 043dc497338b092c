// kernel_args.h -- the argument block every kernel takes (generic and tree-specialised).  No host headers: the
// specialised sources are compiled by NVRTC.
#pragma once
#include "program.h"

// KernelArgs::flags of an ABA launch (the C ABI passes 0; api.cu sets these)
#define MB_KFLAG_ABA_DISCARD 0x10000u // pass three discards the L2 lines of each record after reading it

namespace mb
{
struct KernelArgs
{
   const double *q, *qd, *x, *fext; // x = qdd (RNEA) or tau (ABA)
   const double *x2;                // ABA: given accelerations of the ACCELERATION_SOURCE joints (nullable), rows like x
   double *out;                     // tau (RNEA), qdd (ABA), mass matrix (CRBA)
   double *body_acc, *joint_wrench; // RNEA by-products (nullable), rows [6 * w + c] like fext: spatial acceleration of each body in its
                                    // CoM frame, wrench of each joint in its frameAfterJoint
   double *cmm, *com;               // CRBA by-products (nullable): centroidal momentum matrix rows [r * nv + col], r = 0..5, in the root frame;
                                    // com rows 0..3 accumulate (mass * CoM, mass) over the root's children (zeroed before the launch)
   double *cor;                     // MB_CORIOLIS: the Coriolis matrix, entry-major like the mass matrix in `out`
                                    // MB_GRAVITY_GRADIENT: the joint efforts tau_g [nv][ld]; `out` is then G, entry-major like the mass
                                    // matrix, and zero_entries / n_zero are the mass matrix's (G has its structural zeros)
                                    // MB_RNEA_DERIVATIVES: d tau / dqd, entry-major; `out` is then d tau / dq, zero_entries / n_zero the
                                    // mass matrix's (both matrices have its structural zeros) and `root_wrench` the joint efforts
   double *root_wrench;             // RNEA by-product (nullable): rows 0..5 accumulate the wrench at the root in the root frame (zeroed before)
                                    // MB_RNEA_DERIVATIVES: the joint efforts tau [nv][ld]
   int fp32;                        // optional fp32 variant (mecano_b200_set_precision): arithmetic in float, buffers stay fp64
   const double *consts;            // device copy of the per-body constant records
   double *ws;                      // ABA: pass-two records [rec][ws_ld], one column per resident thread of the persistent grid
   long long ws_ld;
   const uint16_t *zero_entries;    // CRBA: structurally zero mass-matrix entries (multiple of 8, 16-byte aligned)
   int32_t n_zero;                  // MB_REGRESSOR: `out` is the joint-torque regressor Y, [(row * 10 nb + col) * ld + s]; zero_entries
                                    // then holds n_zero uint32 entries, the first column of each structurally zero row of Y
                                    // (FlatTree::regressor_zero_rows; a row's ten columns are zero together)
   long long n, ld;
   long long ld_qd, ld_x; // row strides of qd and x (normally ld; 0 when the launcher substitutes one row of zeros)
   double grav[3];
   uint32_t flags;
   int32_t nv;
   unsigned *work_counter; // persistent thread-per-state launches (nullable): [0] next unassigned state -- warps draw 32 states at a time --,
                           // [1] warps that have run dry; both zero between launches (gpu_ctx.cuh: thread_block_run)
   int32_t stagger_ns; // thread-per-state kernels: warp slot j of a scheduler (warp / 4) starts j * stagger_ns late (gpu_ctx.cuh)
};

} // namespace mb
