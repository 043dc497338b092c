// ltdl_solve.cu -- the last launch of mecano_b200_aba_derivatives: per state, the tree-sparse L^T D L factor of the mass matrix, the
// solve of d tau / dq and d tau / dqd against it and M^-1 (ltdl_solve.cuh), in place in the three entry-major matrices.
//
// One thread per state: a warp reads and writes 32 consecutive states of one entry, so every access is coalesced, and every lane
// follows the same DoF tree, so control flow is uniform.  No workspace: the matrices are the work area.
#include "kernels.h"
#include "ltdl_solve.cuh"

namespace mb
{
namespace
{
#define MB_LTDL_BLOCK 128

__global__ void __launch_bounds__(MB_LTDL_BLOCK) ltdl_solve_kernel(const __grid_constant__ LtdlTree t, const LtdlArgs a)
{
   const long long s = (long long)blockIdx.x * MB_LTDL_BLOCK + threadIdx.x;
   if (s >= a.n)
      return;
   const LtdlMat<double> M{a.minv + s, a.ld, t.nv}, A{a.dq + s, a.ld, t.nv}, B{a.dqd + s, a.ld, t.nv};
   ltdl_solve_state(t, M, A, B);
}
} // namespace

cudaError_t launch_ltdl_solve(const LtdlTree &t, const LtdlArgs &a, cudaStream_t stream)
{
   if (a.n <= 0)
      return cudaSuccess;
   const unsigned grid = (unsigned)((a.n + MB_LTDL_BLOCK - 1) / MB_LTDL_BLOCK);
   ltdl_solve_kernel<<<grid, MB_LTDL_BLOCK, 0, stream>>>(t, a);
   return cudaGetLastError();
}
} // namespace mb
