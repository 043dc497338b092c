// emu_regressor.cpp -- the joint-torque regressor's per-state routine (mecano_b200/csrc/regressor.cuh) compiled for the host (TEST
// INFRASTRUCTURE, never shipped or loaded by the product).  Builds on the emulation harness of emu.cpp, included whole so that its
// host context and counting scalar serve here unchanged; the context only gains the regressor's store and zero-row routines
// (gpu_ctx.cuh: st_Y, y_zero_parts, y_zero_fill_part).  Loaded by tests/emu_regressor_lib.py.
#include "emu.cpp"

#include "../../mecano_b200/csrc/regressor.cuh"

namespace
{
template <class T> struct RegCtx : CpuCtx<T>
{
   const std::vector<uint32_t> *yzl = nullptr;
   // Y entry-major like the mass matrix in emu.cpp, entry e = row * 10 nb + col
   void st_Y(int e, T v) { this->M[(long)e * this->ld + this->s] = (double)v; }
   int y_zero_parts(int nops) const { return ((int)yzl->size() + nops - 1) / nops; }
   void y_zero_fill_part(int k, int parts)
   {
      const int k1 = std::min((int)yzl->size(), (k + 1) * parts);
      for (int i = k * parts; i < k1; i++)
         for (int j = 0; j < 10; j++) st_Y((int)(*yzl)[i] + j, (T)0);
   }
};

template <class T>
int run_regressor(const mecano_b200_tree_desc *d, const double *g, long n, long ld, const double *q, const double *qd, const double *qdd, double *Y,
                  char *err, int errlen)
{
   mb::FlatTree ft;
   std::string e;
   int rc = mb::flatten_tree(d, ft, e);
   if (rc != 0)
   {
      if (err) { std::strncpy(err, e.c_str(), errlen - 1); err[errlen - 1] = 0; }
      return rc;
   }
   const MbProgram &P = ft.prog[MB_REGRESSOR];
   for (int i = 0; i < P.nb; i++)
      if (P.body[i].ext_index >= P.nb)
      {
         if (err) { std::strncpy(err, "wrench_index ranks must be below n_bodies", errlen - 1); err[errlen - 1] = 0; }
         return MECANO_B200_ERR_SHAPE;
      }
   std::vector<T> consts(ft.consts.begin(), ft.consts.end());
   // poison the work areas so that a read-before-write shows up as NaN
   const T nan = (T)(0.0 / 0.0);
   std::vector<T> stk(std::max(P.stack_doubles, 2 * P.stack2) + 2, nan), aux(P.aux_doubles + 1, nan);
   const T grav[3] = {(T)g[0], (T)g[1], (T)g[2]};
   for (long s = 0; s < n; s++)
   {
      std::fill(stk.begin(), stk.end(), nan);
      std::fill(aux.begin(), aux.end(), nan);
      RegCtx<T> c{{q, qd, qdd, nullptr, nullptr, Y, ld, s, ld, ld, ft.nv, stk.data(), aux.data(), nullptr, consts.data()}};
      c.yzl = &ft.regressor_zero_rows;
      mb::regressor_state<T, RegCtx<T>>(P, c, grav);
   }
   return 0;
}
} // namespace

// Y [nv * 10 nb][ld] entry-major, gravity g
extern "C" int emu_joint_torque_regressor(const mecano_b200_tree_desc *d, const double *g, long n, long ld, const double *q, const double *qd,
                                          const double *qdd, double *Y, char *err, int errlen)
{
   return run_regressor<double>(d, g, n, ld, q, qd, qdd, Y, err, errlen);
}

// operation counts of one state (emu.cpp: emu_count_flops): out5 = {add, mul, div, sincos, flops = add + mul + div}
extern "C" int emu_count_flops_regressor(const mecano_b200_tree_desc *d, const double *q, const double *qd, const double *qdd, long *out5)
{
   const double g[3] = {0, 0, -9.81};
   std::vector<double> Y((size_t)10 * d->n_bodies * d->n_dofs, 0.0);
   g_cnt = {0, 0, 0, 0};
   const int rc = run_regressor<Cnt>(d, g, 1, 1, q, qd, qdd, Y.data(), nullptr, 0);
   out5[0] = g_cnt.add; out5[1] = g_cnt.mul; out5[2] = g_cnt.div; out5[3] = g_cnt.sincos;
   out5[4] = g_cnt.add + g_cnt.mul + g_cnt.div;
   return rc;
}
