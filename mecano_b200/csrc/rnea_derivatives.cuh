// rnea_derivatives.cuh -- one state of the first-order partial derivatives of inverse dynamics: the joint efforts tau(q, qd, qdd)
// of RNEA together with d tau / dq and d tau / dqd (nv x nv each).  d tau / dqdd is the mass matrix (crba.cuh).
//
// Definition (include/mecano_b200.h, mecano_b200_rnea_derivatives): column j of d tau / dq is the derivative along q (+) eps e_j,
// the step mecano_b200_integrate takes with qd = e_j (a multi-DoF joint moves along its body-frame velocity coordinate j), the
// convention of the gravity gradient (gravity_gradient.cuh), which this extends to a moving state.  DESIGN.md 4.7 derives the
// recursion.  With, for a joint x with DoF column S (unit twist) and parent twist / acceleration vl, al in x's frame,
//   Psid_x = vl x S,   Psidd_x = al x S + vl x Psid_x,   Sd_x = v_x x S,
// the composites of the subtree of joint j (I^C inertia, B^C factorized inertia of coriolis.cuh, h^C = sum I_k v_k momentum,
// F^C the RNEA force including -fext) and K^C = B^C + B^C^T + (h^C)xbar with (f)xbar x = x x* f, for DoF r of joint j:
//   tau_(j,r) = S . F^C
//   row forces      p1 = I^C S,   p2 = K^C^T S = (B^C + B^C^T) S - S x* h^C
//   column forces   uq = I^C Psidd + K^C Psid + S x* F^C,   uv = I^C (Psid + Sd) + K^C S
//   dq [(j,r)][x]  = S_x . (vl x* (vl x* p1 - p2) - al x* p1)   = p1 . Psidd_x + p2 . Psid_x
//   dqd[(j,r)][x]  = S_x . (p2 - (vl + v_x) x* p1)             = p1 . (Psid_x + Sd_x) + p2 . S_x
//     for every DoF x of joint j and of its ancestors, with x's own vl, al, v_x;
//   dq [x][(j,r)]  = S_x . uq,   dqd[x][(j,r)] = S_x . uv       for every DoF x of a strict ancestor.
// For a one-DoF joint Psid = Sd = v x S and Psidd = a x S + v x Psid with the body's own twist and acceleration (the joint's
// velocity terms cancel), so it keeps only (v, a).  The four forces are carried up the ancestors together, each
// ancestor's transform formed once per walk step.  Both matrices couple only joints on a common root path: their structural
// zeros are those of the mass matrix and come from the CRBA zero list (FlatTree::zero_entries), spread over the ops.
//
// Organisation: the DESCEND ops run pass one of RNEA (twist and acceleration of each body) and leave v and the joint's sin/cos --
// multi-DoF joints: v, vl, al and the transform -- on the shared-memory stack, and a in a per-depth area of the local save area
// (a 60-body chain would otherwise need more shared memory than a block of 32 states has).  The ASCEND ops accumulate the four composites,
// write tau and the joint's own block, fold the composites into the parent and walk the four forces up (a multi-DoF joint
// walks each DoF first and folds after).  The branch save area holds the four accumulators (10 + 36 + 6 + 6 doubles).
#pragma once
#include "coriolis.cuh"

namespace mb
{
// stack slot of a body (double2 units): [v: 3 | sin/cos: 1] or, multi-DoF, [v: 3 | vl: 3 | al: 3 | transform: 6] (a joint
// attached to the root body keeps no transform: no walk leaves it)
#define MB_RD_V 0
#define MB_RD_SC 3
#define MB_RD_VL 3
#define MB_RD_AL 6
#define MB_RD_X 9

// the acceleration of body b: six doubles per depth behind the branch save area (flatten.cpp adds them to aux_doubles)
MB_HD int rd_acc_at(const MbProgram &P, int b) { return P.aux_doubles - 6 * (P.max_depth + 1) + 6 * P.body[b].depth; }

template <class T> MB_HD SvT<T> sv_twice(const SvT<T> &v)
{
   SvT<T> r;
   r.a = (T)2 * v.a;
   r.l = (T)2 * v.l;
   return r;
}

// the forces whose projections onto S_x are the entries of row (j, r) at the DoFs x of a joint with parent twist / acceleration
// vl, al in its frame and vs = vl + v_x:  wq = vl x* (vl x* p1 - p2) - al x* p1,  wv = p2 - vs x* p1
template <class T>
MB_HD void rd_row_forces(const SvT<T> &vl, const SvT<T> &al, const SvT<T> &vs, const SvT<T> &p1, const SvT<T> &p2, SvT<T> &wq, SvT<T> &wv)
{
   wq = cross_force(vl, cross_force(vl, p1) - p2) - cross_force(al, p1);
   wv = p2 - cross_force(vs, p1);
}

// (vl, al, vs) of the joint of body b, whose stack slot is `slot`
template <class T, class Ctx> MB_HD void rd_ld_state(const MbProgram &P, Ctx &c, int b, int jt, int slot, SvT<T> &vl, SvT<T> &al, SvT<T> &vs)
{
   if (jt == MB_SIXDOF)
   {
      vl = stk_ld_sv<T>(c, slot + MB_RD_VL);
      al = stk_ld_sv<T>(c, slot + MB_RD_AL);
      vs = vl + stk_ld_sv<T>(c, slot + MB_RD_V);
   }
   else
   {
      vl = stk_ld_sv<T>(c, slot + MB_RD_V);
      al = aux_ld_sv<T>(c, rd_acc_at(P, b));
      vs = sv_twice(vl);
   }
}

// dq[row][x] = S_x . wq, dqd[row][x] = S_x . wv, dq[x][row] = S_x . uq, dqd[x][row] = S_x . uv for the DoFs x of joint (jt, sub)
// whose first DoF row is dx
template <class T, class Ctx>
MB_HD void rd_project(Ctx &c, int jt, int sub, int dx, int row, const SvT<T> &wq, const SvT<T> &wv, const SvT<T> &uq, const SvT<T> &uv)
{
   const int nv = c.n_dofs();
   if (jt == MB_REVOLUTE)
   {
      c.st_M(row * nv + dx, wq.a.z);
      c.st_C(row * nv + dx, wv.a.z);
      c.st_M(dx * nv + row, uq.a.z);
      c.st_C(dx * nv + row, uv.a.z);
   }
   else if (jt == MB_PRISMATIC)
   {
      c.st_M(row * nv + dx, wq.l.z);
      c.st_C(row * nv + dx, wv.l.z);
      c.st_M(dx * nv + row, uq.l.z);
      c.st_C(dx * nv + row, uv.l.z);
   }
   else
   {
      const int nd = mb_sub_ndof(sub);
#pragma unroll 1
      for (int x = 0; x < nd; x++)
      {
         const int cx = sub == MB_SUB_SIX ? x : mb_sub_component(sub, x);
         c.st_M(row * nv + dx + x, sv_get(wq, cx));
         c.st_C(row * nv + dx + x, sv_get(wv, cx));
         c.st_M((dx + x) * nv + row, sv_get(uq, cx));
         c.st_C((dx + x) * nv + row, sv_get(uv, cx));
      }
   }
}

// row / column `row`: from body b (transform given by (s, cs) / the stack) up to the child of the root body
template <class T, class Ctx>
MB_HD void rd_walk(const MbProgram &P, Ctx &c, int b, int row, T s, T cs, SvT<T> p1, SvT<T> p2, SvT<T> uq, SvT<T> uv)
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
         X = stk_ld_xf<T>(c, w.slot + MB_RD_X);
      p1 = force_to_parent(X, p1);
      p2 = force_to_parent(X, p2);
      uq = force_to_parent(X, uq);
      uv = force_to_parent(X, uv);
      b = w.parent;
      w = P.walk[b];
      SvT<T> vl, al, vs, wq, wv;
      rd_ld_state<T>(P, c, b, w.jtype, w.slot, vl, al, vs);
      rd_row_forces(vl, al, vs, p1, p2, wq, wv);
      rd_project<T>(c, w.jtype, mb_sub_of<Ctx>(w), w.dof, row, wq, wv, uq, uv);
      if (w.jtype != MB_SIXDOF)
         c.stk_ld2(w.slot, MB_RD_SC, s, cs);
   }
}

template <class T, class Ctx> MB_HD void rnea_derivatives_state(const MbProgram &P, Ctx &c, const T *grav)
{
   const int zpart = c.zero_parts(P.nops);
   const bool fx = c.has_fext();
   const int nv = c.n_dofs();
   // composites of the finished children of the body ascended next: inertia, factorized inertia, momentum, RNEA force
   RbiT<T> acc = RbiT<T>();
   FbiT<T> bacc;
   bacc.A = bacc.TR = bacc.BL = bacc.L = m3_zero<T>();
   SvT<T> hacc = sv_zero<T>(), facc = sv_zero<T>();
   SvT<T> v = sv_zero<T>(), a = sv_zero<T>();
   T ls = (T)0, lc = (T)1; // sin/cos of the last DESCEND (a leaf's ASCEND follows immediately)
   const int nops = P.nops;
#pragma unroll 1
   for (int k = 0; k < nops; k++)
   {
      const MbOp2 o = P.op2[k];
      c.stk_fence();
      c.zero_fill_mc_part(k, zpart);
      const int jt = MB2_JT(o.code);
      const auto C = c.cst(o.body);
      if (!(o.code & MB2_ASCEND))
      {
         // ---- pass one of RNEA: joint transform, twist and acceleration of the body (rnea.cuh), gravity as the root acceleration
         if (o.flags & MB2_ROOT_PARENT)
         {
            v = sv_zero<T>();
            a = sv_zero<T>();
            a.l = v3<T>(-grav[0], -grav[1], -grav[2]);
         }
         else if (o.flags & MB2_LOAD_PARENT)
         {
            v = stk_ld_sv<T>(c, o.pslot + MB_RD_V);
            a = aux_ld_sv<T>(c, rd_acc_at(P, P.body[o.body].parent));
         }
         if (jt == MB_SIXDOF)
         {
            const int sub = mb_sub_of<Ctx>(o);
            const XfT<T> X = joint_xf_multi<T>(c, C, o.cfg, sub);
            const SvT<T> vl = motion_to_child(X, v), al = motion_to_child(X, a);
            const SvT<T> vj = ld_svj<T>(o.dof, sub, [&](int r) { return c.ld_qd(r); });
            const SvT<T> aj = ld_svj<T>(o.dof, sub, [&](int r) { return c.ld_x(r); });
            v = vl + vj;
            a = al + cross_motion(v, vj) + aj;
            stk_st_sv<T>(c, o.slot + MB_RD_V, v);
            aux_st_sv<T>(c, rd_acc_at(P, o.body), a);
            stk_st_sv<T>(c, o.slot + MB_RD_VL, vl);
            stk_st_sv<T>(c, o.slot + MB_RD_AL, al);
            if (!(o.flags & MB2_ROOT_PARENT))
               stk_st_xf<T>(c, o.slot + MB_RD_X, X);
         }
         else
         {
            const T q = c.ld_q(o.cfg), qd = c.ld_qd(o.dof), qdd = c.ld_x(o.dof);
            XfT<T> X;
            if (jt == MB_REVOLUTE)
            {
               mb_sincos(mb_reduce_angle(q), &ls, &lc);
               X = joint_xf_1dof<T, true>(C, ls, lc);
               v = motion_to_child(X, v);
               a = motion_to_child(X, a);
               // a += v x (S qd) + S qdd with S = [e_z; 0]
               a.a.x += v.a.y * qd; a.a.y -= v.a.x * qd;
               a.l.x += v.l.y * qd; a.l.y -= v.l.x * qd;
               v.a.z += qd;
               a.a.z += qdd;
            }
            else
            {
               ls = q; // a prismatic displacement is not an angle
               lc = (T)1;
               X = joint_xf_1dof<T, false>(C, ls, lc);
               v = motion_to_child(X, v);
               a = motion_to_child(X, a);
               // S = [0; e_z]
               a.l.x += v.a.y * qd; a.l.y -= v.a.x * qd;
               v.l.z += qd;
               a.l.z += qdd;
            }
            if (!(o.flags & MB2_LEAF))
            {
               stk_st_sv<T>(c, o.slot + MB_RD_V, v);
               aux_st_sv<T>(c, rd_acc_at(P, o.body), a);
               c.stk_st2(o.slot, MB_RD_SC, ls, lc);
            }
         }
         continue;
      }
      // ---- the body's RNEA force and the four composites of the subtree, about this joint frame
      SvT<T> vb = v, ab = a;
      T js = ls, jc = lc;
      if (jt == MB_SIXDOF || !(o.flags & MB2_LEAF))
      {
         vb = stk_ld_sv<T>(c, o.slot + MB_RD_V);
         ab = aux_ld_sv<T>(c, rd_acc_at(P, o.body));
         if (jt != MB_SIXDOF)
            c.stk_ld2(o.slot, MB_RD_SC, js, jc);
      }
      const RbiT<T> Ib = ld_rbi<T>(C);
      SvT<T> hc = mul(Ib, vb);
      SvT<T> Fc = mul(Ib, ab) + cross_force(vb, hc);
      if (fx)
         Fc = Fc - external_wrench<T>(c, P.body[o.body].ext_index, C);
      RbiT<T> Ic = Ib;
      FbiT<T> Bc = fbi_from_rbi(Ib, vb);
      if (!(o.flags & MB2_LEAF))
      {
         Ic = Ic + acc;
         Bc = Bc + bacc;
         hc = hc + hacc;
         Fc = Fc + facc;
      }
      const int d = o.dof;
      const bool walk = !(o.flags & MB2_ROOT_PARENT);
      auto fold = [&]() {
         XfT<T> X;
         if (jt == MB_REVOLUTE) X = joint_xf_1dof<T, true>(C, js, jc);
         else if (jt == MB_PRISMATIC) X = joint_xf_1dof<T, false>(C, js, jc);
         else X = stk_ld_xf<T>(c, o.slot + MB_RD_X);
         const RbiT<T> K = rbi_to_parent(X, Ic);
         const FbiT<T> KB = fbi_to_parent(X, Bc);
         const SvT<T> Kh = force_to_parent(X, hc), KF = force_to_parent(X, Fc);
         if (o.flags & MB2_FIRST_CHILD)
         {
            acc = K;
            bacc = KB;
            hacc = Kh;
            facc = KF;
         }
         else
         {
            acc = aux_ld_rbi<T>(c, o.paux) + K;
            bacc = aux_ld_fbi<T>(c, o.paux + 10) + KB;
            hacc = aux_ld_sv<T>(c, o.paux + 46) + Kh;
            facc = aux_ld_sv<T>(c, o.paux + 52) + KF;
         }
         if (o.flags & MB2_STORE_ACC)
         {
            aux_st_rbi<T>(c, o.paux, acc);
            aux_st_fbi<T>(c, o.paux + 10, bacc);
            aux_st_sv<T>(c, o.paux + 46, hacc);
            aux_st_sv<T>(c, o.paux + 52, facc);
         }
      };
      if (jt != MB_SIXDOF)
      {
         SvT<T> S = sv_zero<T>();
         if (jt == MB_REVOLUTE) S.a.z = (T)1;
         else S.l.z = (T)1;
         c.st_jtau(d, jt == MB_REVOLUTE ? Fc.a.z : Fc.l.z);
         const SvT<T> psid = cross_motion(vb, S);
         const SvT<T> psidd = cross_motion(ab, S) + cross_motion(vb, psid);
         const SvT<T> bs = mul(Bc, S) + mulT(Bc, S), sh = cross_force(S, hc);
         const SvT<T> p1 = mul(Ic, S), p2 = bs - sh;
         const SvT<T> uq = mul(Ic, psidd) + mul(Bc, psid) + mulT(Bc, psid) + cross_force(psid, hc) + cross_force(S, Fc);
         const SvT<T> uv = mul(Ic, sv_twice(psid)) + bs + sh;
         SvT<T> wq, wv;
         rd_row_forces(vb, ab, sv_twice(vb), p1, p2, wq, wv);
         c.st_M(d * nv + d, jt == MB_REVOLUTE ? wq.a.z : wq.l.z);
         c.st_C(d * nv + d, jt == MB_REVOLUTE ? wv.a.z : wv.l.z);
         if (walk)
         {
            // the accumulators first, so that the composites are dead while the four forces walk up the ancestors
            fold();
            rd_walk<T>(P, c, o.body, d, js, jc, p1, p2, uq, uv);
         }
      }
      else
      {
         // multi-DoF joint: DoF r is component comp(r) of the spatial vector in frameAfterJoint (multidof.cuh)
         const int sub = mb_sub_of<Ctx>(o), nd = mb_sub_ndof(sub);
         const SvT<T> vl = stk_ld_sv<T>(c, o.slot + MB_RD_VL), al = stk_ld_sv<T>(c, o.slot + MB_RD_AL);
#pragma unroll 1
         for (int r = 0; r < nd; r++)
         {
            const int cc = mb_sub_component(sub, r);
            SvT<T> S = sv_zero<T>();
            if (cc == 0) S.a.x = (T)1; else if (cc == 1) S.a.y = (T)1; else if (cc == 2) S.a.z = (T)1;
            else if (cc == 3) S.l.x = (T)1; else if (cc == 4) S.l.y = (T)1; else S.l.z = (T)1;
            c.st_jtau(d + r, sv_get(Fc, cc));
            const SvT<T> psid = cross_motion(vl, S), sd = cross_motion(vb, S);
            const SvT<T> psidd = cross_motion(al, S) + cross_motion(vl, psid);
            const SvT<T> bs = mul(Bc, S) + mulT(Bc, S), sh = cross_force(S, hc);
            const SvT<T> p1 = mul(Ic, S), p2 = bs - sh;
            const SvT<T> uq = mul(Ic, psidd) + mul(Bc, psid) + mulT(Bc, psid) + cross_force(psid, hc) + cross_force(S, Fc);
            const SvT<T> uv = mul(Ic, psid + sd) + bs + sh;
            // the joint's own block, row (d, r)
            SvT<T> wq, wv;
            rd_row_forces(vl, al, vl + vb, p1, p2, wq, wv);
#pragma unroll 1
            for (int x = 0; x < nd; x++)
            {
               const int cx = mb_sub_component(sub, x);
               c.st_M((d + r) * nv + d + x, sv_get(wq, cx));
               c.st_C((d + r) * nv + d + x, sv_get(wv, cx));
            }
            if (walk)
               rd_walk<T>(P, c, o.body, d + r, js, jc, p1, p2, uq, uv);
         }
         if (walk)
            fold();
      }
   }
}
} // namespace mb
