// kernels.h -- launch interface between the C-ABI layer (api.cu) and the sm_100a kernels (kernels.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>

#include "kernel_args.h"
#include "program.h"

namespace mb
{
struct LaunchPlan
{
   int block = 0;        // threads per block (= states per block for the thread-per-state variant)
   size_t smem = 0;      // dynamic shared memory per block
   int tm = 0;           // stack slots held in tensor memory
   int size_class = 0;   // 0: small local work areas, 1: large
   int blocks_per_sm = 0;
   int regs = 0;
   int local_bytes = 0;
   int static_smem = 0;
   int grid = 0;         // persistent grid: resident blocks on the whole device
   size_t ws_doubles = 0; // ABA workspace size for that grid
   bool fp32_ok = false;  // the optional fp32 variant exists for this configuration
   int fp32_regs = 0;
   bool m3 = false;       // the tree has three-DoF joints: the kernels instantiated with them (thread_kernels.cuh)
};

// Picks the block size / size class for one algorithm and opts the kernel into large shared memory.
// Returns cudaSuccess or an error; *fits == false if the tree exceeds the compiled work-area classes.
cudaError_t plan_thread_kernel(int algo, const MbProgram &P, bool fext, LaunchPlan &plan, bool *fits);

cudaError_t launch_thread_kernel(int algo, const MbProgram &P, const KernelArgs &a, const LaunchPlan &plan, cudaStream_t stream);

// warp-per-state variant (warp_kernels.cu): lane = body, trees of up to 32 bodies; larger trees (up to MB_MAX_BODIES) run the
// team kernels below.  warp_variant_supports: one of the two serves this tree
bool warp_variant_supports(const MbProgram &P);
cudaError_t launch_warp_kernel(int algo, const MbProgram *device_program, const KernelArgs &a, int max_children, int max_ndof, int sm_count, cudaStream_t stream);
cudaError_t warp_kernel_attributes(int algo, bool fext, cudaFuncAttributes *attr);
// team-per-state variant (team_kernels.cu): thread = body, two to four warps per state, trees of 33 to 128 bodies
int team_threads(const MbProgram &P);
cudaError_t launch_team_kernel(int algo, const MbProgram *device_program, int nb, const KernelArgs &a, int max_children, int max_ndof, int sm_count, cudaStream_t stream);
cudaError_t team_kernel_attributes(int algo, bool fext, cudaFuncAttributes *attr);

// batched state integrator (integrate.cu): MultiBodySystemStateIntegrator.doubleIntegrateFromAcceleration
struct IntegrateJoints
{
   int32_t nb;
   uint16_t cfg[MB_MAX_BODIES], dof[MB_MAX_BODIES]; // Mecano configuration / DoF row of each joint
   uint8_t type[MB_MAX_BODIES];                     // MB_REVOLUTE / MB_PRISMATIC / MB_SIXDOF
   uint8_t sub[MB_MAX_BODIES];                      // MB_SUB_* of a multi-DoF joint
};
struct IntegrateArgs
{
   double *q, *qd, *qdd; // updated in place (qdd: SixDoF linear rows only)
   long long n, ld;
   double dt;
};
cudaError_t launch_integrate_kernel(const IntegrateJoints &J, const IntegrateArgs &a, int sm_count, cudaStream_t stream);

// forward-dynamics derivatives, last step (ltdl_solve.cu): per state, M in minv -> M^-1, d tau / dx in dq, dqd -> -M^-1 d tau / dx
struct LtdlTree;
struct LtdlArgs
{
   double *minv, *dq, *dqd; // [nv * nv][ld] entry-major each
   long long n, ld;
};
cudaError_t launch_ltdl_solve(const LtdlTree &t, const LtdlArgs &a, cudaStream_t stream);

// centroidal by-products, last step (centroidal.cu)
struct CentroidalArgs
{
   double *cols;      // [6 * ncols][ld], row r * ncols + j: column j of a 6 x ncols matrix, angular rows first (nullable if !shift)
   double *com;       // [4][ld]: (mass * CoM, mass) in, (CoM, mass) out if normalize_com; (CoM, mass) in otherwise
   long long n, ld;
   int ncols;
   int normalize_com; // divide the first three com rows by the fourth
   int shift;         // move the moments of every column from the origin of the root frame to the CoM
};
cudaError_t launch_centroidal_finish(const CentroidalArgs &a, cudaStream_t stream);

// roofline denominators
cudaError_t measure_fp64_peak(double *tflops);
cudaError_t measure_fp64_sustained(double seconds, double *tflops);
cudaError_t measure_hbm_peak(double *gbs);
} // namespace mb
