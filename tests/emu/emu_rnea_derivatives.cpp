// emu_rnea_derivatives.cpp -- the inverse-dynamics derivatives' per-state routine (mecano_b200/csrc/rnea_derivatives.cuh) compiled
// for the host (TEST INFRASTRUCTURE, never shipped or loaded by the product).  Builds on the emulation harness of emu.cpp, included
// whole so that its host context and counting scalar serve here unchanged; the context only gains the store of the joint efforts
// (gpu_ctx.cuh: st_jtau).  d tau / dq goes through the mass-matrix store, d tau / dqd through the Coriolis-matrix store, both
// zeroed from the context's zero list.  Loaded by tests/emu_rnea_derivatives_lib.py.
#include "emu.cpp"

#include "../../mecano_b200/csrc/rnea_derivatives.cuh"

namespace
{
template <class T> struct RdCtx : CpuCtx<T>
{
   double *tau = nullptr;
   void st_jtau(int r, T v) { tau[(long)r * this->ld + this->s] = (double)v; }
};

template <class T>
int run_rnea_derivatives(const mecano_b200_tree_desc *d, const double *g, long n, long ld, const double *q, const double *qd, const double *qdd,
                         const double *fext, double *tau, double *dq, double *dqd, char *err, int errlen)
{
   mb::FlatTree ft;
   std::string e;
   int rc = mb::flatten_tree(d, ft, e);
   if (rc != 0)
   {
      if (err) { std::strncpy(err, e.c_str(), errlen - 1); err[errlen - 1] = 0; }
      return rc;
   }
   const MbProgram &P = ft.prog[MB_RNEA_DERIVATIVES];
   std::vector<T> consts(ft.consts.begin(), ft.consts.end());
   // poison the work areas so that a read-before-write shows up as NaN
   const T nan = (T)(0.0 / 0.0);
   std::vector<T> stk(std::max(P.stack_doubles, 2 * P.stack2) + 2, nan), aux(P.aux_doubles + 1, nan);
   const T grav[3] = {(T)g[0], (T)g[1], (T)g[2]};
   for (long s = 0; s < n; s++)
   {
      std::fill(stk.begin(), stk.end(), nan);
      std::fill(aux.begin(), aux.end(), nan);
      RdCtx<T> c{{q, qd, qdd, fext, nullptr, dq, ld, s, ld, ld, ft.nv, stk.data(), aux.data(), nullptr, consts.data()}};
      c.zl = &ft.zero_entries;
      c.Cm = dqd;
      c.tau = tau;
      mb::rnea_derivatives_state<T, RdCtx<T>>(P, c, grav);
   }
   return 0;
}
} // namespace

// tau [nv][ld], dq and dqd [nv * nv][ld] entry-major, gravity g, fext [6 nb][ld] in the rows of the description (nullable)
extern "C" int emu_rnea_derivatives(const mecano_b200_tree_desc *d, const double *g, long n, long ld, const double *q, const double *qd,
                                    const double *qdd, const double *fext, double *tau, double *dq, double *dqd, char *err, int errlen)
{
   return run_rnea_derivatives<double>(d, g, n, ld, q, qd, qdd, fext, tau, dq, dqd, err, errlen);
}

// operation counts of one state without external wrenches (emu.cpp: emu_count_flops): out5 = {add, mul, div, sincos, flops}
extern "C" int emu_count_flops_rnea_derivatives(const mecano_b200_tree_desc *d, const double *q, const double *qd, const double *qdd, long *out5)
{
   const double g[3] = {0, 0, -9.81};
   std::vector<double> tau((size_t)d->n_dofs, 0.0), dq((size_t)d->n_dofs * d->n_dofs, 0.0), dqd((size_t)d->n_dofs * d->n_dofs, 0.0);
   g_cnt = {0, 0, 0, 0};
   const int rc = run_rnea_derivatives<Cnt>(d, g, 1, 1, q, qd, qdd, nullptr, tau.data(), dq.data(), dqd.data(), nullptr, 0);
   out5[0] = g_cnt.add; out5[1] = g_cnt.mul; out5[2] = g_cnt.div; out5[3] = g_cnt.sincos;
   out5[4] = g_cnt.add + g_cnt.mul + g_cnt.div;
   return rc;
}
