// regressor.cuh -- one state of the joint-torque regressor Y(q, qd, qdd) (Mecano's JointTorqueRegressorCalculator: the
// inertial-parameter regressor of inverse dynamics, tau = Y pi for every set of inertial parameters pi).
//
// Definition (include/mecano_b200.h, mecano_b200_joint_torque_regressor): Y is nv x 10 nb; column block w (ten columns)
// belongs to the body whose external-wrench rows are [6 w, 6 w + 6); its parameters, in the column order of the
// MECANO_B200_REGRESSOR_* table, are m, m c, and the moment of inertia about the origin, all in the body's CoM frame.
//
// Organisation: the DESCEND ops carry the twist and the acceleration of the body (RNEA pass one, rnea.cuh).  At body w they
// are re-expressed in its CoM frame, where the ten columns of the 6 x 10 body regressor are formed:
//   m:        (0, g)                       g = a_lin + w x v_lin, the classical acceleration of the frame origin
//   h = m c:  (e_j x g, K e_j)             K = al~ + w w^T - |w|^2 1   (al: angular acceleration)
//   I:        (I al + w x (I w), 0)        for the six unit symmetric I
// The columns are mapped to the joint frame, projected on the body's own S, then carried up the ancestors together, each
// ancestor's transform formed once for all ten (the walk of crba.cuh: crba_walk).  The six inertia columns are pure couples
// and stay so on the way up: only their rotation is applied.  The ancestors' sin/cos (SixDoF: transforms) are on the stack
// during the descent, so the walk runs in the DESCEND op and the ASCEND ops only spread the structural zeros.
#pragma once
#include "jointmath.cuh"
#include "../../include/mecano_b200.h"

namespace mb
{
// the ten columns of one body, in its current frame: m and the three first moments as wrenches, the six inertias as couples
template <class T> struct RegCols
{
   SvT<T> m, h[3];
   V3T<T> I[6];
};

template <class T> MB_HD T v3_get(const V3T<T> &v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : v.z); }

// the body regressor in the CoM frame (twist v, acceleration a of that frame), re-expressed in the joint frame X = (E, c)
template <class T> MB_HD RegCols<T> reg_body(const XfT<T> &X, const SvT<T> &v, const SvT<T> &a)
{
   const V3T<T> w = v.a, al = a.a;
   const V3T<T> g = cross_add(w, v.l, a.l);
   const T ww = dot(w, w);
   RegCols<T> F;
   F.m.a = v3<T>((T)0, (T)0, (T)0);
   F.m.l = g;
   // K e_j: column j of al~ + w w^T - |w|^2 1;  e_j x g
   F.h[0].a = v3<T>((T)0, -g.z, g.y);
   F.h[0].l = v3<T>(w.x * w.x - ww, al.z + w.y * w.x, -al.y + w.z * w.x);
   F.h[1].a = v3<T>(g.z, (T)0, -g.x);
   F.h[1].l = v3<T>(-al.z + w.x * w.y, w.y * w.y - ww, al.x + w.z * w.y);
   F.h[2].a = v3<T>(-g.y, g.x, (T)0);
   F.h[2].l = v3<T>(al.y + w.x * w.z, -al.x + w.y * w.z, w.z * w.z - ww);
   // I al + w x (I w) for I = the unit symmetric matrices xx, xy, xz, yy, yz, zz
   const V3T<T> Iw[6] = {v3<T>(w.x, (T)0, (T)0), v3<T>(w.y, w.x, (T)0), v3<T>(w.z, (T)0, w.x),
                         v3<T>((T)0, w.y, (T)0), v3<T>((T)0, w.z, w.y), v3<T>((T)0, (T)0, w.z)};
   const V3T<T> Ia[6] = {v3<T>(al.x, (T)0, (T)0), v3<T>(al.y, al.x, (T)0), v3<T>(al.z, (T)0, al.x),
                         v3<T>((T)0, al.y, (T)0), v3<T>((T)0, al.z, al.y), v3<T>((T)0, (T)0, al.z)};
#pragma unroll
   for (int k = 0; k < 6; k++)
      F.I[k] = mul(X.R, cross_add(w, Iw[k], Ia[k]));
   F.m = force_to_parent(X, F.m);
#pragma unroll
   for (int j = 0; j < 3; j++)
      F.h[j] = force_to_parent(X, F.h[j]);
   return F;
}

// the ten columns carried from a body's frame to its parent's: X = the body's joint transform
template <class T> MB_HD void reg_up(const XfT<T> &X, RegCols<T> &F)
{
   F.m = force_to_parent(X, F.m);
#pragma unroll
   for (int j = 0; j < 3; j++)
      F.h[j] = force_to_parent(X, F.h[j]);
#pragma unroll
   for (int k = 0; k < 6; k++)
      F.I[k] = mul(X.R, F.I[k]);
}

// row e0 / e0 + 1 .. of Y: component `comp` ([wx wy wz vx vy vz]) of the ten columns
template <class T, class Ctx> MB_HD void reg_store_row(Ctx &c, int e0, int comp, const RegCols<T> &F)
{
   c.st_Y(e0 + MECANO_B200_REGRESSOR_M, sv_get(F.m, comp));
#pragma unroll
   for (int j = 0; j < 3; j++)
      c.st_Y(e0 + MECANO_B200_REGRESSOR_MC + j, sv_get(F.h[j], comp));
#pragma unroll
   for (int k = 0; k < 6; k++)
      c.st_Y(e0 + MECANO_B200_REGRESSOR_I + k, comp < 3 ? v3_get(F.I[k], comp) : (T)0);
}

// S_j^T of the ten columns into the rows of joint j (first DoF row dj); cb = first column of the body's block, ncol = 10 nb
template <class T, class Ctx> MB_HD void reg_project(Ctx &c, int jt, int sub, int dj, int cb, int ncol, const RegCols<T> &F)
{
   if (jt == MB_REVOLUTE)
      reg_store_row<T>(c, dj * ncol + cb, 2, F);
   else if (jt == MB_PRISMATIC)
      reg_store_row<T>(c, dj * ncol + cb, 5, F);
   else
   {
      const int nd = mb_sub_ndof(sub);
#pragma unroll 1
      for (int r = 0; r < nd; r++)
         reg_store_row<T>(c, (dj + r) * ncol + cb, sub == MB_SUB_SIX ? r : mb_sub_component(sub, r), F);
   }
}

template <class T, class Ctx> MB_HD void regressor_state(const MbProgram &P, Ctx &c, const T *grav)
{
   // rows of joints off the path from the root to a body are zero in that body's block, spread over the ops
   const int zpart = c.y_zero_parts(P.nops);
   const int ncol = 10 * P.nb;
   SvT<T> v = sv_zero<T>(), a = sv_zero<T>();
   const int nops = P.nops;
#pragma unroll 1
   for (int k = 0; k < nops; k++)
   {
      const MbOp2 o = P.op2[k];
      c.y_zero_fill_part(k, zpart);
      if (o.code & MB2_ASCEND)
         continue;
      const int jt = MB2_JT(o.code);
      const auto C = c.cst(o.body);
      // ---- pass one of RNEA (rnea.cuh): twist and acceleration of the body in its joint frame; the root accelerates at -gravity
      if (o.flags & MB2_ROOT_PARENT)
      {
         v = sv_zero<T>();
         a = sv_zero<T>();
         a.l = v3<T>(-grav[0], -grav[1], -grav[2]);
      }
      else if (o.flags & MB2_LOAD_PARENT)
      {
         v = aux_ld_sv<T>(c, o.paux);
         a = aux_ld_sv<T>(c, o.paux + 6);
      }
      XfT<T> X;
      T s = (T)0, cs = (T)1;
      if (jt == MB_SIXDOF)
      {
         const int sub = mb_sub_of<Ctx>(o);
         X = joint_xf_multi<T>(c, C, o.cfg, sub);
         const SvT<T> vj = ld_svj<T>(o.dof, sub, [&](int r) { return c.ld_qd(r); });
         const SvT<T> aj = ld_svj<T>(o.dof, sub, [&](int r) { return c.ld_x(r); });
         v = motion_to_child(X, v) + vj;
         a = motion_to_child(X, a) + cross_motion(v, vj) + aj;
         stk_st_xf<T>(c, o.slot, X);
      }
      else
      {
         const T q = c.ld_q(o.cfg), qd = c.ld_qd(o.dof), qdd = c.ld_x(o.dof);
         SvT<T> vj = sv_zero<T>(), aj = sv_zero<T>();
         if (jt == MB_REVOLUTE)
         {
            mb_sincos(mb_reduce_angle(q), &s, &cs);
            X = joint_xf_1dof<T, true>(C, s, cs);
            vj.a.z = qd;
            aj.a.z = qdd;
         }
         else
         {
            s = q;
            X = joint_xf_1dof<T, false>(C, s, cs);
            vj.l.z = qd;
            aj.l.z = qdd;
         }
         v = motion_to_child(X, v) + vj;
         a = motion_to_child(X, a) + cross_motion(v, vj) + aj;
         if (!(o.flags & MB2_LEAF))
            c.stk_st2(o.slot, 0, s, cs);
      }
      if (o.flags & MB2_SAVE_STATE)
      {
         aux_st_sv<T>(c, o.aux, v);
         aux_st_sv<T>(c, o.aux + 6, a);
      }
      // ---- the body's block: the ten columns in its CoM frame, mapped to the joint frame, projected on S and on every ancestor's S
      XfT<T> Xc;
      ld_com<T>(C, Xc.R, Xc.p);
      RegCols<T> F = reg_body<T>(Xc, motion_to_child(Xc, v), motion_to_child(Xc, a));
      const int cb = 10 * P.body[o.body].ext_index;
      reg_project<T>(c, jt, mb_sub_of<Ctx>(o), o.dof, cb, ncol, F);
      int b = o.body;
      MbWalk w = P.walk[b];
#pragma unroll 1
      while (!(w.flags & 1u)) // until the parent is the root body; X = the joint transform of body b
      {
         reg_up<T>(X, F);
         b = w.parent;
         w = P.walk[b];
         reg_project<T>(c, w.jtype, mb_sub_of<Ctx>(w), w.dof, cb, ncol, F);
         if (w.flags & 1u)
            break;
         if (w.jtype == MB_SIXDOF)
            X = stk_ld_xf<T>(c, w.slot);
         else
         {
            c.stk_ld2(w.slot, 0, s, cs);
            X = w.jtype == MB_REVOLUTE ? joint_xf_1dof<T, true>(c.cst(b), s, cs) : joint_xf_1dof<T, false>(c.cst(b), s, cs);
         }
      }
   }
}
} // namespace mb
