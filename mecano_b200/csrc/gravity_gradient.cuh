// gravity_gradient.cuh -- one state of the gravity gradient (Mecano's MultiBodyGravityGradientCalculator): the joint efforts that
// gravity and the external wrenches cause, tau_g(q), and their configuration gradient G = d tau_g / dq (nv x nv).
//
// Definition (include/mecano_b200.h, mecano_b200_gravity_gradient): tau_g is RNEA at qd = qdd = 0; column j of G is the derivative
// along q (+) eps e_j, the step mecano_b200_integrate takes with qd = e_j (a multi-DoF joint moves along its body-frame velocity
// coordinate j).  DESIGN.md 4.7 derives the recursion.  With a0 = (0, g) the root acceleration (g = -gravity) carried into the
// frame of body d, I^c_d its composite inertia, F_d = I^c_d a0 - (composite external wrench), for DoF r of joint d with unit twist S:
//   tau_(d,r)       = S . F_d
//   n               = (I^c_d S)_lin x g                 (= -(a0 x* I^c_d S): a pure couple)
//   u               = S x* F_d - I^c_d (S x a0)
//   G[(d,r)][x]     = S_x . (n, 0)  for every DoF x of joint d and of its ancestors
//   G[x][(d,r)]     = S_x . u       for every DoF x of a strict ancestor
// n and u are carried up the ancestors together, each ancestor's transform formed once per walk step (the walk of crba.cuh:
// crba_walk).  G couples only joints on a common root path: its structural zeros are those of the mass matrix and come from
// the CRBA zero list (FlatTree::zero_entries), spread over the ops.
//
// Organisation: the DESCEND ops carry g into each body's frame and leave the joint's sin/cos (SixDoF / three-DoF: the transform)
// on the stack, like CRBA.  The ASCEND ops accumulate the composite inertia and, when external wrenches are given (tested at run
// time), the composite external wrench, form tau, n, u and walk, then fold the subtree into the parent and rotate g back into the
// parent's frame -- so that the next sibling's DESCEND finds it there (it is never saved in the branch area).
#pragma once
#include "crba.cuh"

namespace mb
{
// G[col][x] = S_x . (n, 0) and G[x][col] = S_x . u for the DoFs x of joint (jt, sub) whose first DoF row is dj
template <class T, class Ctx> MB_HD void gg_project(Ctx &c, int jt, int sub, int dj, int col, const V3T<T> &n, const SvT<T> &u)
{
   const int nv = c.n_dofs();
   if (jt == MB_REVOLUTE)
   {
      c.st_M(col * nv + dj, n.z);
      c.st_M(dj * nv + col, u.a.z);
   }
   else if (jt == MB_PRISMATIC)
   {
      c.st_M(col * nv + dj, (T)0);
      c.st_M(dj * nv + col, u.l.z);
   }
   else
   {
      SvT<T> nc;
      nc.a = n;
      nc.l = v3<T>((T)0, (T)0, (T)0);
      const int nd = mb_sub_ndof(sub);
#pragma unroll 1
      for (int r = 0; r < nd; r++)
      {
         const int comp = sub == MB_SUB_SIX ? r : mb_sub_component(sub, r);
         c.st_M(col * nv + dj + r, sv_get(nc, comp));
         c.st_M((dj + r) * nv + col, sv_get(u, comp));
      }
   }
}

// column `col` of G: from body b (transform given by (s, cs) / the stack) up to the child of the root body
template <class T, class Ctx> MB_HD void gg_walk(const MbProgram &P, Ctx &c, int b, int col, T s, T cs, V3T<T> n, SvT<T> u)
{
   MbWalk w = P.walk[b];
#pragma unroll 1
   while (!(w.flags & 1u)) // until the parent is the root body
   {
      const auto C = c.cst(b);
      XfT<T> X;
      if (w.jtype == MB_REVOLUTE)
         X = joint_xf_1dof<T, true>(C, s, cs);
      else if (w.jtype == MB_PRISMATIC)
         X = joint_xf_1dof<T, false>(C, s, cs);
      else
         X = stk_ld_xf<T>(c, w.slot);
      n = mul(X.R, n);
      u = force_to_parent(X, u);
      b = w.parent;
      w = P.walk[b];
      gg_project<T>(c, w.jtype, mb_sub_of<Ctx>(w), w.dof, col, n, u);
      if (w.jtype != MB_SIXDOF)
         c.stk_ld2(w.slot, 0, s, cs);
   }
}

template <class T, class Ctx> MB_HD void gravity_gradient_state(const MbProgram &P, Ctx &c, const T *grav)
{
   const int zpart = c.zero_parts(P.nops);
   const bool fx = c.has_fext();
   const int nv = c.n_dofs();
   RbiT<T> acc = RbiT<T>();        // composite inertia of the finished children of the body ascended next
   SvT<T> accf = sv_zero<T>();     // the same for the external wrenches
   V3T<T> g = v3<T>(-grav[0], -grav[1], -grav[2]);
   T ls = (T)0, lc = (T)1;         // sin/cos of the last DESCEND (a leaf's ASCEND follows immediately)
   const int nops = P.nops;
#pragma unroll 1
   for (int k = 0; k < nops; k++)
   {
      const MbOp2 o = P.op2[k];
      c.zero_fill_part(k, zpart);
      const int jt = MB2_JT(o.code);
      const auto C = c.cst(o.body);
      if (!(o.code & MB2_ASCEND))
      {
         // ---- joint transform; g into the body's frame (a DESCEND that reloads its parent finds g there: see the top)
         if (o.flags & MB2_ROOT_PARENT)
            g = v3<T>(-grav[0], -grav[1], -grav[2]);
         XfT<T> X;
         if (jt == MB_SIXDOF)
         {
            X = joint_xf_multi<T>(c, C, o.cfg, mb_sub_of<Ctx>(o));
            stk_st_xf<T>(c, o.slot, X);
         }
         else
         {
            const T q = c.ld_q(o.cfg);
            T s = q, cs = (T)1; // a prismatic displacement is not an angle
            if (jt == MB_REVOLUTE)
            {
               mb_sincos(mb_reduce_angle(q), &s, &cs);
               X = joint_xf_1dof<T, true>(C, s, cs);
            }
            else
               X = joint_xf_1dof<T, false>(C, s, cs);
            ls = s;
            lc = cs;
            if (!(o.flags & MB2_LEAF))
               c.stk_st2(o.slot, 0, s, cs);
         }
         g = mulT(X.R, g);
         continue;
      }
      // ---- composite inertia and external wrench of the subtree, about this joint frame
      RbiT<T> Ic = ld_rbi<T>(C);
      if (!(o.flags & MB2_LEAF))
         Ic = Ic + acc;
      SvT<T> Fx = sv_zero<T>();
      if (fx)
      {
         Fx = external_wrench<T>(c, P.body[o.body].ext_index, C);
         if (!(o.flags & MB2_LEAF))
            Fx = Fx + accf;
      }
      T js = ls, jc = lc;
      if (jt != MB_SIXDOF && !(o.flags & MB2_LEAF))
         c.stk_ld2(o.slot, 0, js, jc);
      // F = Ic a0 - Fx with a0 = (0, g)
      SvT<T> F;
      F.a = cross(Ic.h, g);
      F.l = Ic.m * g;
      if (fx)
         F = F - Fx;
      const int d = o.dof;
      const bool walk = !(o.flags & MB2_ROOT_PARENT);
      if (jt == MB_REVOLUTE)
      {
         // S = (e_z, 0): Ic S = (I e_z, e_z x h); S x a0 = (0, e_z x g)
         c.st_tau(d, F.a.z);
         const V3T<T> hl = v3<T>(-Ic.h.y, Ic.h.x, (T)0);
         const V3T<T> n = cross(hl, g);
         const V3T<T> wz = v3<T>(-g.y, g.x, (T)0);
         SvT<T> u;
         u.a = v3<T>(-F.a.y, F.a.x, (T)0) - cross(Ic.h, wz);
         u.l = v3<T>(-F.l.y, F.l.x, (T)0) - Ic.m * wz;
         c.st_M(d * nv + d, n.z);
         if (walk)
            gg_walk<T>(P, c, o.body, d, js, jc, n, u);
      }
      else if (jt == MB_PRISMATIC)
      {
         // S = (0, e_z): Ic S = (h x e_z, m e_z), S x a0 = 0, S x* F = (e_z x F_lin, 0)
         c.st_tau(d, F.l.z);
         const V3T<T> n = v3<T>(-Ic.m * g.y, Ic.m * g.x, (T)0);
         SvT<T> u;
         u.a = v3<T>(-F.l.y, F.l.x, (T)0);
         u.l = v3<T>((T)0, (T)0, (T)0);
         c.st_M(d * nv + d, (T)0);
         if (walk)
            gg_walk<T>(P, c, o.body, d, js, jc, n, u);
      }
      else
      {
         // multi-DoF joint: DoF r is component comp(r) of the spatial vector in frameAfterJoint (multidof.cuh)
         const int sub = mb_sub_of<Ctx>(o), nd = mb_sub_ndof(sub);
#pragma unroll 1
         for (int r = 0; r < nd; r++)
         {
            const int cc = mb_sub_component(sub, r);
            SvT<T> e = sv_zero<T>();
            if (cc == 0) e.a.x = 1; else if (cc == 1) e.a.y = 1; else if (cc == 2) e.a.z = 1;
            else if (cc == 3) e.l.x = 1; else if (cc == 4) e.l.y = 1; else e.l.z = 1;
            c.st_tau(d + r, sv_get(F, cc));
            const V3T<T> n = cross(mul(Ic, e).l, g);
            const V3T<T> w = cross(e.a, g);
            SvT<T> Iw;
            Iw.a = cross(Ic.h, w);
            Iw.l = Ic.m * w;
            const SvT<T> u = cross_force(e, F) - Iw;
            // the joint's own block, row (d, r): G[(d,r)][(d,x)] = S_x . (n, 0)
            SvT<T> nc;
            nc.a = n;
            nc.l = v3<T>((T)0, (T)0, (T)0);
#pragma unroll 1
            for (int x = 0; x < nd; x++)
               c.st_M((d + r) * nv + d + x, sv_get(nc, mb_sub_component(sub, x)));
            if (walk)
               gg_walk<T>(P, c, o.body, d + r, js, jc, n, u);
         }
      }
      if (walk)
      {
         // fold the subtree into the parent; g back into the parent's frame
         XfT<T> X;
         if (jt == MB_REVOLUTE) X = joint_xf_1dof<T, true>(C, js, jc);
         else if (jt == MB_PRISMATIC) X = joint_xf_1dof<T, false>(C, js, jc);
         else X = stk_ld_xf<T>(c, o.slot);
         const RbiT<T> K = rbi_to_parent(X, Ic);
         acc = (o.flags & MB2_FIRST_CHILD) ? K : aux_ld_rbi<T>(c, o.paux) + K;
         if (o.flags & MB2_STORE_ACC)
            aux_st_rbi<T>(c, o.paux, acc);
         if (fx)
         {
            const SvT<T> Kf = force_to_parent(X, Fx);
            accf = (o.flags & MB2_FIRST_CHILD) ? Kf : aux_ld_sv<T>(c, o.paux + 10) + Kf;
            if (o.flags & MB2_STORE_ACC)
               aux_st_sv<T>(c, o.paux + 10, accf);
         }
         g = mul(X.R, g);
      }
   }
}
} // namespace mb
