// emu_aba_derivatives.cpp -- the forward-dynamics derivatives' per-state linear algebra (mecano_b200/csrc/ltdl_solve.cuh) compiled
// for the host (TEST INFRASTRUCTURE, never shipped or loaded by the product), on the DoF tree the flattener builds for it
// (FlatTree::ltdl_dof / ltdl_parent).  Loaded by tests/emu_aba_derivatives_lib.py, which composes it with the emulated ABA,
// inverse-dynamics derivatives and CRBA.
#include <algorithm>
#include <cstring>
#include <string>

#include "../../mecano_b200/csrc/flatten.h"
#include "../../mecano_b200/csrc/ltdl_solve.cuh"

namespace
{
int ltdl_tree(const mecano_b200_tree_desc *d, mb::LtdlTree &t, char *err, int errlen)
{
   mb::FlatTree ft;
   std::string e;
   const int rc = mb::flatten_tree(d, ft, e);
   if (rc != 0)
   {
      if (err) { std::strncpy(err, e.c_str(), errlen - 1); err[errlen - 1] = 0; }
      return rc;
   }
   t.nv = ft.nv;
   std::copy(ft.ltdl_dof.begin(), ft.ltdl_dof.end(), t.dof);
   std::copy(ft.ltdl_parent.begin(), ft.ltdl_parent.end(), t.lam);
   return 0;
}
} // namespace

// the DoF tree: dof[k], lam[k] for k < n_dofs
extern "C" int emu_ltdl_tree(const mecano_b200_tree_desc *d, int *dof, int *lam, char *err, int errlen)
{
   mb::LtdlTree t;
   const int rc = ltdl_tree(d, t, err, errlen);
   if (rc) return rc;
   for (int k = 0; k < t.nv; k++) { dof[k] = t.dof[k]; lam[k] = t.lam[k]; }
   return 0;
}

// step 1 alone on n states of M [nv * nv][ld] (the factor of ltdl_solve.cuh in place)
extern "C" int emu_ltdl_factor(const mecano_b200_tree_desc *d, long n, long ld, double *M, char *err, int errlen)
{
   mb::LtdlTree t;
   const int rc = ltdl_tree(d, t, err, errlen);
   if (rc) return rc;
   for (long s = 0; s < n; s++)
      mb::ltdl_factor<double>(t, {M + s, ld, t.nv});
   return 0;
}

// the whole routine on n states: minv holds M on entry, M^-1 on return; dq, dqd hold d tau / dq, d tau / dqd on entry,
// -M^-1 times them on return
extern "C" int emu_ltdl_solve(const mecano_b200_tree_desc *d, long n, long ld, double *minv, double *dq, double *dqd, char *err, int errlen)
{
   mb::LtdlTree t;
   const int rc = ltdl_tree(d, t, err, errlen);
   if (rc) return rc;
   for (long s = 0; s < n; s++)
      mb::ltdl_solve_state<double>(t, {minv + s, ld, t.nv}, {dq + s, ld, t.nv}, {dqd + s, ld, t.nv});
   return 0;
}
