// ltdl_solve.cuh -- one state of the forward-dynamics derivatives' linear algebra: the tree-sparse factor M = L^T D L of the mass
// matrix (Featherstone, RBDA 6.5), the solve of the inverse-dynamics partials against it and the inverse M^-1, all in place in
// the caller's entry-major matrices.  Compiles for the device (ltdl_solve.cu) and for the host (tests/emu).
//
// DoFs are visited in the internal order of the flattened tree (depth-first pre-order, a multi-DoF joint as a chain of its DoFs):
// DoF k sits in row / column dof[k] of the matrices and its DoF parent lam[k] < k (-1 at a root joint), so the factor has M's
// sparsity, with no fill-in.  "Lower" below means entry (k, i) with i < k in that order, at row dof[k], column dof[i].
//
// The in-place order in one state (the three matrices of mecano_b200_aba_derivatives; Mi arrives holding CRBA's dense M):
//   1. factor: L (unit, strictly lower, entries (k, i) for i an ancestor of k) over M's lower triangle, 1 / D_k on the diagonal;
//      nothing else is read or written (M's upper triangle and its structural zeros are left as they are);
//   2. solve: every column of A and B (d tau / dq, d tau / dqd) becomes -M^-1 times itself, column j of A and of B together so
//      that each factor entry is read once for both;
//   3. inverse: with W = M^-1 = L^-1 D^-1 L^-T, L W = D^-1 L^-T is zero below the diagonal and 1 / D_k on it, so row k of W's
//      lower triangle follows from the rows of its ancestors:
//        W_km = -sum_{i anc k} L_ki W_im  (m < k),   W_kk = 1 / D_k - sum_{i anc k} L_ki W_ki.
//      Row k overwrites L's row k, so that row is first copied into M's upper triangle (entry (i, k)), which holds nothing needed
//      any more; rows are formed in increasing k, then the lower triangle is mirrored over the upper one.
// The sums start from +0.0, so W's entries between branches that hang separately off a fixed root come out as +0.0.
// Every lane of a warp follows the same lam: control flow is uniform.
#pragma once
#include "spatial.cuh"

namespace mb
{
#define MB_LTDL_MAX_DOFS 255 // n_dofs^2 < 2^16 (flatten.cpp)

// the DoF order of the factor (FlatTree::ltdl_dof / ltdl_parent)
struct LtdlTree
{
   int32_t nv;
   int16_t dof[MB_LTDL_MAX_DOFS];  // row / column of DoF k in the caller's matrices
   int16_t lam[MB_LTDL_MAX_DOFS];  // DoF parent of DoF k (< k), -1 at a root joint
};

// entry (r, c) of one state of an entry-major nv x nv matrix
template <class T> struct LtdlMat
{
   T *p;
   long long ld;
   int nv;
   MB_HD T &operator()(int r, int c) const { return p[((long long)r * nv + c) * ld]; }
};

// step 1: M (lower triangle and diagonal, in the order above) -> unit L below the diagonal, 1 / D on it
template <class T> MB_HD void ltdl_factor(const LtdlTree &t, const LtdlMat<T> &M)
{
#pragma unroll 1
   for (int k = t.nv - 1; k >= 0; k--)
   {
      const int rk = t.dof[k];
      const T rd = (T)1 / M(rk, rk);
      M(rk, rk) = rd;
#pragma unroll 1
      for (int i = t.lam[k]; i >= 0; i = t.lam[i])
      {
         const int ri = t.dof[i];
         const T a = M(rk, ri) * rd;
#pragma unroll 1
         for (int j = i; j >= 0; j = t.lam[j])
            M(ri, t.dof[j]) = fmad(-M(rk, t.dof[j]), a, M(ri, t.dof[j]));
         M(rk, ri) = a;
      }
   }
}

// step 2: column c of A and of B -> -M^-1 times itself (M^-1 = L^-1 D^-1 L^-T from the factor of step 1)
template <class T> MB_HD void ltdl_solve_column(const LtdlTree &t, const LtdlMat<T> &F, const LtdlMat<T> &A, const LtdlMat<T> &B, int c)
{
   // L^T z = x, from the leaves up
#pragma unroll 1
   for (int k = t.nv - 1; k >= 0; k--)
   {
      const int rk = t.dof[k];
      const T xa = A(rk, c), xb = B(rk, c);
#pragma unroll 1
      for (int i = t.lam[k]; i >= 0; i = t.lam[i])
      {
         const int ri = t.dof[i];
         const T l = F(rk, ri);
         A(ri, c) = fmad(-l, xa, A(ri, c));
         B(ri, c) = fmad(-l, xb, B(ri, c));
      }
   }
   // u = -y with L y = D^-1 z, from the root down:  u_k = -z_k / D_k - sum_i L_ki u_i
#pragma unroll 1
   for (int k = 0; k < t.nv; k++)
   {
      const int rk = t.dof[k];
      const T nrd = -F(rk, rk);
      T ua = A(rk, c) * nrd, ub = B(rk, c) * nrd;
#pragma unroll 1
      for (int i = t.lam[k]; i >= 0; i = t.lam[i])
      {
         const int ri = t.dof[i];
         const T l = F(rk, ri);
         ua = fmad(-l, A(ri, c), ua);
         ub = fmad(-l, B(ri, c), ub);
      }
      A(rk, c) = ua;
      B(rk, c) = ub;
   }
}

// step 3: the factor of step 1 -> M^-1, every entry written
template <class T> MB_HD void ltdl_inverse(const LtdlTree &t, const LtdlMat<T> &W)
{
#pragma unroll 1
   for (int k = 0; k < t.nv; k++)
   {
      const int rk = t.dof[k];
#pragma unroll 1
      for (int i = t.lam[k]; i >= 0; i = t.lam[i])
         W(t.dof[i], rk) = W(rk, t.dof[i]); // L_ki to the upper triangle
#pragma unroll 1
      for (int m = 0; m < k; m++)
      {
         const int rm = t.dof[m];
         T w = (T)0;
#pragma unroll 1
         for (int i = t.lam[k]; i >= 0; i = t.lam[i])
         {
            const int ri = t.dof[i];
            w = fmad(-W(ri, rk), m <= i ? W(ri, rm) : W(rm, ri), w);
         }
         W(rk, rm) = w;
      }
      T w = W(rk, rk);
#pragma unroll 1
      for (int i = t.lam[k]; i >= 0; i = t.lam[i])
      {
         const int ri = t.dof[i];
         w = fmad(-W(ri, rk), W(rk, ri), w);
      }
      W(rk, rk) = w;
   }
#pragma unroll 1
   for (int k = 1; k < t.nv; k++)
#pragma unroll 1
      for (int m = 0; m < k; m++)
         W(t.dof[m], t.dof[k]) = W(t.dof[k], t.dof[m]);
}

// one state of mecano_b200_aba_derivatives' last launch: Mi holds M on entry and M^-1 on return, A and B hold d tau / dq and
// d tau / dqd on entry and d qdd / dq and d qdd / dqd on return
template <class T> MB_HD void ltdl_solve_state(const LtdlTree &t, const LtdlMat<T> &Mi, const LtdlMat<T> &A, const LtdlMat<T> &B)
{
   ltdl_factor(t, Mi);
#pragma unroll 1
   for (int c = 0; c < t.nv; c++)
      ltdl_solve_column(t, Mi, A, B, c);
   ltdl_inverse(t, Mi);
}
} // namespace mb
