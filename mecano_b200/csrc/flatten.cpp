// flatten.cpp -- see flatten.h.  Plain host C++ (no CUDA).
#include "flatten.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

namespace mb
{
namespace
{
struct M3
{
   double m[9];
};

M3 identity()
{
   M3 r{};
   r.m[0] = r.m[4] = r.m[8] = 1.0;
   return r;
}

M3 mul(const M3 &a, const M3 &b)
{
   M3 r{};
   for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++)
         r.m[3 * i + j] = a.m[3 * i] * b.m[j] + a.m[3 * i + 1] * b.m[3 + j] + a.m[3 * i + 2] * b.m[6 + j];
   return r;
}

M3 transpose(const M3 &a)
{
   M3 r{};
   for (int i = 0; i < 3; i++)
      for (int j = 0; j < 3; j++)
         r.m[3 * i + j] = a.m[3 * j + i];
   return r;
}

void mulv(const M3 &a, const double *x, double *y)
{
   double t[3];
   for (int i = 0; i < 3; i++)
      t[i] = a.m[3 * i] * x[0] + a.m[3 * i + 1] * x[1] + a.m[3 * i + 2] * x[2];
   y[0] = t[0];
   y[1] = t[1];
   y[2] = t[2];
}

// rotation Q with Q e_z = u (|u| = 1): shortest arc
M3 align_z_to(const double *u)
{
   const double c = u[2];
   if (c > 1.0 - 1e-14)
      return identity();
   if (c < -1.0 + 1e-14)
   {
      M3 r = identity();
      r.m[4] = -1.0;
      r.m[8] = -1.0; // rotation by pi about x
      return r;
   }
   // v = e_z x u = (-uy, ux, 0); Q = I + [v]x + [v]x^2 / (1 + c)
   const double vx = -u[1], vy = u[0];
   const double k = 1.0 / (1.0 + c);
   M3 K{};
   K.m[0] = 0; K.m[1] = 0; K.m[2] = vy;
   K.m[3] = 0; K.m[4] = 0; K.m[5] = -vx;
   K.m[6] = -vy; K.m[7] = vx; K.m[8] = 0;
   M3 K2 = mul(K, K);
   M3 r = identity();
   for (int i = 0; i < 9; i++)
      r.m[i] += K.m[i] + k * K2.m[i];
   return r;
}

int joint_ndof(int api_type) { return api_type == MECANO_B200_SIXDOF ? 6 : (api_type >= MECANO_B200_SPHERICAL ? 3 : 1); }
int joint_ncfg(int api_type) { return api_type == MECANO_B200_SIXDOF ? 7 : (api_type == MECANO_B200_SPHERICAL ? 4 : (api_type == MECANO_B200_PLANAR ? 3 : 1)); }

int slot_size(int algo, int jtype)
{
   const int jp = mb_jp_size(jtype);
   const int nd = jtype == MB_SIXDOF ? 6 : 1;
   switch (algo)
   {
      case MB_RNEA: return 6 + jp;       // accumulated wrench + joint parameters
      case MB_ABA: return 6 + jp + nd;   // twist + joint parameters + joint velocity
      case MB_CORIOLIS: return 6 + jp;   // twist + joint parameters
      default: return jp;                // CRBA, regressor, gravity gradient: joint parameters only
   }
}

// v2 stack slots, in double2 units (rnea.cuh / aba.cuh / crba.cuh)
int slot2_size(int algo, int jtype, bool root_parent)
{
   switch (algo)
   {
      case MB_RNEA: // wrench (3) + sin/cos (1); SixDoF: wrench (3) + transform (6) unless attached to the root body
         return jtype == MB_SIXDOF ? (root_parent ? 3 : 9) : 4;
      case MB_ABA: // twist (3) + sin/cos (1); SixDoF: twist (3) + transform (6) unless attached to the root body
         return jtype == MB_SIXDOF ? (root_parent ? 3 : 9) : 4;
      case MB_CORIOLIS: // twist (3) + sin/cos (1); SixDoF: twist (3) + transform (6)
         return jtype == MB_SIXDOF ? 9 : 4;
      case MB_RNEA_DERIVATIVES: // twist (3) + sin/cos (1); SixDoF: twist, the parent's twist and acceleration (9) + transform (6) unless
                                // attached to the root body (the body's acceleration: a per-depth area behind the branch save area)
         return jtype == MB_SIXDOF ? (root_parent ? 9 : 15) : 4;
      default: // CRBA, regressor, gravity gradient: sin/cos (1); SixDoF: transform (6)
         return jtype == MB_SIXDOF ? 6 : 1;
   }
}

// Runs of consecutive ops of the same kind (MbRun).  RNEA runs are split by the SC bit (its routines schedule the sin/cos of the
// next joint inside the op's basic block).  ABA splits only its DESCEND ops that way (pass three evaluates no sin/cos: they
// travel in the pass-two records); its ASCEND ops are large,
// the SC test there is a warp-uniform branch taken a few times per state, and one loop body per joint type keeps the hot code of
// the kernel inside the instruction cache (no_instructions was 12.8 % of the stall samples with SC-split ASCEND runs).  Runs whose
// ops all carry the common flags of their kind are marked MB_RUN_PLAIN (program.h).
void build_runs(int algo, MbProgram &P, int n3)
{
   auto make_runs = [algo](const MbOp2 *ops, int n, MbRun *runs, bool pass3) {
      int nr = 0;
      for (int k = 0; k < n; k++)
      {
         uint8_t kind = ops[k].code & (mb_run_kind_has_sc(algo, ops[k].code & 0xf, pass3) ? 0xfu : 0x7u);
         const unsigned tested = mb_run_plain_tested(algo, kind, pass3);
         if (tested)
         {
            const bool next1 = (ops[k].pf & MB2_PF_NEXT1) != 0, sc = (kind & MB2_SC) != 0;
            if ((ops[k].flags & tested) == (mb_run_plain_flags(algo, kind, pass3) & tested) && (!mb_run_kind_has_sc(algo, kind, pass3) || next1 == sc))
               kind |= MB_RUN_PLAIN;
         }
         if (nr > 0 && runs[nr - 1].kind == kind && runs[nr - 1].n < 255)
            runs[nr - 1].n++;
         else
         {
            runs[nr].kind = kind;
            runs[nr].n = 1;
            runs[nr].k0 = (uint16_t)k;
            nr++;
         }
      }
      return nr;
   };
   P.nruns = make_runs(P.op2, P.nops, P.run, false);
   P.nruns3 = make_runs(P.op3, n3, P.run3, true);
}

// Pre-decode the op words into MbOp2 records (program.h).
void build_op2(int algo, MbProgram &P, const std::vector<int> &nchild)
{
   const int nb = P.nb;
   std::vector<int> slot2(nb, 0), wslot(nb, 0), nslot(nb, 0);
   P.stack2 = 1;
   P.wstack2 = P.nstack2 = 0;
   for (int i = 0; i < nb; i++)
   {
      const MbBody &B = P.body[i];
      int s = 0;
      if (B.parent >= 0)
      {
         const MbBody &Bp = P.body[B.parent];
         s = slot2[B.parent] + slot2_size(algo, Bp.jtype, Bp.parent < 0);
         if (mb_algo(algo).wide_stack)
         {
            wslot[i] = wslot[B.parent] + 3;
            nslot[i] = nslot[B.parent] + slot2_size(algo, Bp.jtype, Bp.parent < 0) - 3;
         }
      }
      slot2[i] = s;
      // leaves keep their data in registers, except SixDoF joints which always use their slot
      if (nchild[i] > 0 || B.jtype == MB_SIXDOF)
      {
         P.stack2 = std::max(P.stack2, s + slot2_size(algo, B.jtype, B.parent < 0));
         if (mb_algo(algo).wide_stack)
         {
            P.wstack2 = std::max(P.wstack2, wslot[i] + 3);
            P.nstack2 = std::max(P.nstack2, nslot[i] + slot2_size(algo, B.jtype, B.parent < 0) - 3);
         }
      }
   }
   if (algo == MB_ABA)
      P.stack2 = std::max(P.stack2, 4 * MB_ABA_RING_ROWS); // pass three overlays a 4-stage ring of double2 rows on the stack area
   std::memset(P.op2, 0, sizeof P.op2);
   for (int k = 0; k < P.nops; k++)
   {
      const uint32_t w = P.op[k];
      const int i = MB_OP_BODY(w);
      const MbBody &B = P.body[i];
      MbOp2 &o = P.op2[k];
      o.code = (uint8_t)((w & MB_OP_ASCEND) | ((uint32_t)B.jtype << 1) | ((uint32_t)B.sub << 4));
      o.flags = (uint8_t)((w & 0xfeu) >> 1);
      o.body = (uint8_t)i;
      o.cfg = (uint16_t)B.cfg_off;
      o.dof = (uint16_t)B.dof_off;
      o.slot = (uint16_t)slot2[i];
      o.pslot = (uint16_t)(B.parent >= 0 ? slot2[B.parent] : 0);
      o.aux = (uint16_t)(B.aux >= 0 ? B.aux : 0);
      o.paux = (uint16_t)(B.parent >= 0 && P.body[B.parent].aux >= 0 ? P.body[B.parent].aux : 0);
      o.wslot = (uint16_t)wslot[i];
      o.pwslot = (uint16_t)(B.parent >= 0 ? wslot[B.parent] : 0);
      o.nslot = (uint16_t)nslot[i];
   }
   for (int i = 0; i < nb; i++)
   {
      const MbBody &B = P.body[i];
      MbWalk &w = P.walk[i];
      w.jtype = (uint8_t)B.jtype;
      w.flags = (uint8_t)(B.parent < 0 ? 1 : 0);
      w.parent = (uint8_t)(B.parent < 0 ? 0 : B.parent);
      w.sub = (uint16_t)B.sub;
      w.pad2 = 0;
      w.dof = (uint16_t)B.dof_off;
      w.slot = (uint16_t)slot2[i];
      // packed layout: bodies are in depth-first order, so the parent's record is complete
      w.above = (uint8_t)(B.parent < 0 ? 0 : P.walk[B.parent].above + P.body[B.parent].ndof);
      w.pcol = (uint16_t)(i == 0 ? 0 : P.walk[i - 1].pcol + P.body[i - 1].ndof * P.walk[i - 1].above + P.body[i - 1].ndof * (P.body[i - 1].ndof + 1) / 2);
   }
   // trailing records: ASCEND of a SixDoF joint can never be mistaken for a 1-DoF DESCEND by the look-ahead
   for (int k = P.nops; k < P.nops + 4; k++)
      P.op2[k].code = (uint8_t)(MB2_ASCEND | (MB_SIXDOF << 1));
   // pass-three list: one DESCEND record per body.  Pass two writes the pass-three records of the bodies in post-order; pass
   // three reads them in the REVERSE of that order -- a pre-order walk that visits the children of a body last child first --
   // so that the workspace behaves like a stack: what was written last (and is still in L2) is read first, and a record is
   // dead (and discarded from L2) as soon as it has been read.  The forward order (MECANO_B200_ABA_P3_FORWARD=1, kept for
   // measurements) reads the records in roughly the order they were written, i.e. each one after the whole workspace has
   // passed through L2 in between.
   int n3 = 0;
   {
      static const bool forward = getenv("MECANO_B200_ABA_P3_FORWARD") != nullptr;
      std::vector<int> desc_of(nb, -1);
      for (int k = 0; k < P.nops; k++)
         if (!(P.op2[k].code & MB2_ASCEND))
            desc_of[P.op2[k].body] = k;
      std::vector<std::vector<int>> kids(nb + 1);
      for (int i = 0; i < nb; i++)
         kids[P.body[i].parent + 1].push_back(i);
      std::vector<int> stack;
      // a stack pops the last pushed first: push in reverse for the forward order, as listed for the reversed one
      auto push_kids = [&](int b) {
         const std::vector<int> &c = kids[b + 1];
         if (forward && algo == MB_ABA) stack.insert(stack.end(), c.rbegin(), c.rend());
         else if (algo == MB_ABA) stack.insert(stack.end(), c.begin(), c.end());
         else stack.insert(stack.end(), c.rbegin(), c.rend());
      };
      push_kids(-1);
      int prev = -2;
      while (!stack.empty())
      {
         const int i = stack.back();
         stack.pop_back();
         MbOp2 o = P.op2[desc_of[i]];
         // the parent's kinematic state is in registers only if the parent was the op just before
         o.flags = (uint8_t)(o.flags & ~MB2_LOAD_PARENT);
         if (P.body[i].parent >= 0 && prev != P.body[i].parent)
            o.flags |= MB2_LOAD_PARENT;
         P.op3[n3++] = o;
         prev = i;
         push_kids(i);
      }
   }
   auto look_ahead = [](MbOp2 *ops, int n) {
      for (int k = 0; k < n; k++)
      {
         const MbOp2 &n1 = ops[k + 1];
         if (!(n1.code & MB2_ASCEND) && MB2_JT(n1.code) == MB_REVOLUTE)
            ops[k].code |= MB2_SC;
         if (!(n1.code & MB2_ASCEND) && MB2_JT(n1.code) != MB_SIXDOF)
            ops[k].pf |= MB2_PF_NEXT1;
         // what op k requests for op k + 3 (MB_PF_DIST, rnea.cuh); the trailing records are SixDoF ASCENDs: nothing
         const MbOp2 &nd = ops[k + 3];
         if (MB2_JT(nd.code) != MB_SIXDOF)
            ops[k].pf |= (nd.code & MB2_ASCEND) ? MB2_PF_A1 : MB2_PF_D1;
         ops[k].pfcfg = nd.cfg;
         ops[k].pfdof = nd.dof;
         ops[k].pfbody = nd.body;
      }
   };
   look_ahead(P.op2, P.nops);
   look_ahead(P.op3, n3);
   P.nruns3 = n3; // (the number of pass-three ops until build_runs() replaces it by the number of runs)
   build_runs(algo, P, n3);
}
} // namespace

int flatten_tree(const mecano_b200_tree_desc *d, FlatTree &out, std::string &err)
{
   if (!d)
   {
      err = "tree description is NULL";
      return MECANO_B200_ERR_INVALID_ARGUMENT;
   }
   if (d->struct_size != (int32_t)sizeof(mecano_b200_tree_desc))
   {
      err = "mecano_b200_tree_desc.struct_size mismatch (ABI version)";
      return MECANO_B200_ERR_INVALID_ARGUMENT;
   }
   const int nb = d->n_bodies;
   if (nb <= 0)
   {
      err = "tree has no joints";
      return MECANO_B200_ERR_INVALID_ARGUMENT;
   }
   if ((long)d->n_dofs * d->n_dofs > 65535)
   {
      err = "mass matrix has more than 65535 entries";
      return MECANO_B200_ERR_TOO_LARGE;
   }
   if (nb > MB_MAX_BODIES)
   {
      err = "tree has more than " + std::to_string(MB_MAX_BODIES) + " bodies";
      return MECANO_B200_ERR_TOO_LARGE;
   }
   if (!d->parent || !d->joint_type || !d->axis || !d->offset_rot || !d->offset_pos || !d->com_rot || !d->com_pos || !d->inertia
       || !d->mass || !d->dof_offset || !d->cfg_offset)
   {
      err = "tree description has a NULL table";
      return MECANO_B200_ERR_INVALID_ARGUMENT;
   }

   // ---- validation
   int nv = 0, nq = 0;
   for (int b = 0; b < nb; b++)
   {
      const int jt = d->joint_type[b];
      if (jt < MECANO_B200_REVOLUTE || jt > MECANO_B200_PLANAR)
      {
         err = "body " + std::to_string(b) + ": unsupported joint type " + std::to_string(jt)
               + " (RevoluteJoint, PrismaticJoint, SixDoFJoint, SphericalJoint, PlanarJoint; no CPU fallback)";
         return MECANO_B200_ERR_UNSUPPORTED_TOPOLOGY;
      }
      if (d->parent[b] < -1 || d->parent[b] >= b)
      {
         err = "body " + std::to_string(b) + ": parent index must satisfy -1 <= parent < body (kinematic loops are not supported)";
         return MECANO_B200_ERR_UNSUPPORTED_TOPOLOGY;
      }
      nv += joint_ndof(jt);
      nq += joint_ncfg(jt);
      if (jt == MECANO_B200_REVOLUTE || jt == MECANO_B200_PRISMATIC)
      {
         const double *u = d->axis + 3 * b;
         const double n = std::sqrt(u[0] * u[0] + u[1] * u[1] + u[2] * u[2]);
         if (!(n > 1e-12))
         {
            err = "body " + std::to_string(b) + ": zero joint axis";
            return MECANO_B200_ERR_INVALID_ARGUMENT;
         }
      }
      const double *J = d->inertia + 9 * b;
      const double scale = std::fabs(J[0]) + std::fabs(J[4]) + std::fabs(J[8]) + 1e-300;
      if (std::fabs(J[1] - J[3]) > 1e-9 * scale || std::fabs(J[2] - J[6]) > 1e-9 * scale || std::fabs(J[5] - J[7]) > 1e-9 * scale)
      {
         err = "body " + std::to_string(b) + ": moment of inertia is not symmetric";
         return MECANO_B200_ERR_INVALID_ARGUMENT;
      }
   }
   if (d->wrench_index)
   {
      // ranks in the caller's joint list: distinct, and small enough for 6 * w + 5 to stay a 16-bit row (a list may hold more
      // joints than the tree has bodies: fixed joints are folded away by the host model before the tables are built)
      std::vector<char> used(10922, 0);
      for (int b = 0; b < nb; b++)
         if (d->wrench_index[b] < 0 || d->wrench_index[b] >= 10922 || used[d->wrench_index[b]]++)
         {
            err = "wrench_index must hold distinct ranks in [0, 10922)";
            return MECANO_B200_ERR_SHAPE;
         }
   }
   if (nv != d->n_dofs || nq != d->n_cfg)
   {
      err = "n_dofs / n_cfg do not match the joint types";
      return MECANO_B200_ERR_SHAPE;
   }
   {
      std::vector<char> used_v(nv, 0), used_q(nq, 0);
      for (int b = 0; b < nb; b++)
      {
         const int nd = joint_ndof(d->joint_type[b]), nc = joint_ncfg(d->joint_type[b]);
         if (d->dof_offset[b] < 0 || d->dof_offset[b] + nd > nv || d->cfg_offset[b] < 0 || d->cfg_offset[b] + nc > nq)
         {
            err = "body " + std::to_string(b) + ": dof/cfg offset out of range";
            return MECANO_B200_ERR_SHAPE;
         }
         for (int k = 0; k < nd; k++)
            if (used_v[d->dof_offset[b] + k]++)
            {
               err = "dof offsets overlap";
               return MECANO_B200_ERR_SHAPE;
            }
         for (int k = 0; k < nc; k++)
            if (used_q[d->cfg_offset[b] + k]++)
            {
               err = "cfg offsets overlap";
               return MECANO_B200_ERR_SHAPE;
            }
      }
   }

   // ---- depth-first pre-order, children visited in increasing DoF row (Mecano's insertion order,
   //      JointIterator.java:153-162 / JointMatrixIndexProvider.java:77-101)
   std::vector<std::vector<int>> children(nb + 1);
   for (int b = 0; b < nb; b++)
      children[d->parent[b] + 1].push_back(b);
   for (auto &c : children)
      std::sort(c.begin(), c.end(), [&](int a, int b) { return d->dof_offset[a] < d->dof_offset[b]; });
   std::vector<int> order; // internal -> caller index
   order.reserve(nb);
   {
      std::vector<int> stack(children[0].rbegin(), children[0].rend());
      while (!stack.empty())
      {
         const int b = stack.back();
         stack.pop_back();
         order.push_back(b);
         for (auto it = children[b + 1].rbegin(); it != children[b + 1].rend(); ++it)
            stack.push_back(*it);
      }
   }
   out = FlatTree();
   out.nb = nb;
   out.nv = nv;
   out.nq = nq;
   out.internal_of.assign(nb, -1);
   for (int i = 0; i < nb; i++)
      out.internal_of[order[i]] = i;

   // ---- canonical frames and constant records
   std::vector<M3> Q(nb);
   out.consts.assign((size_t)nb * MB_CONST_STRIDE, 0.0);
   std::vector<int> parent_i(nb), nchild(nb, 0), depth(nb, 0), subtree_end(nb, 0);
   for (int i = 0; i < nb; i++)
   {
      const int b = order[i];
      const int pb = d->parent[b];
      parent_i[i] = pb < 0 ? -1 : out.internal_of[pb];
      if (parent_i[i] >= 0)
      {
         nchild[parent_i[i]]++;
         depth[i] = depth[parent_i[i]] + 1;
      }
      out.max_depth = std::max(out.max_depth, depth[i] + 1);

      double u[3] = {0, 0, 1};
      if (d->joint_type[b] == MECANO_B200_REVOLUTE || d->joint_type[b] == MECANO_B200_PRISMATIC)
      {
         const double *a = d->axis + 3 * b;
         const double n = std::sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
         u[0] = a[0] / n; u[1] = a[1] / n; u[2] = a[2] / n;
         Q[i] = align_z_to(u);
      }
      else
         Q[i] = identity();

      M3 RT, Rc;
      std::memcpy(RT.m, d->offset_rot + 9 * b, sizeof RT.m);
      std::memcpy(Rc.m, d->com_rot + 9 * b, sizeof Rc.m);
      const M3 QpT = parent_i[i] < 0 ? identity() : transpose(Q[parent_i[i]]);
      const M3 R = mul(mul(QpT, RT), Q[i]);
      double p[3];
      mulv(QpT, d->offset_pos + 3 * b, p);
      const M3 QiT = transpose(Q[i]);
      const M3 E = mul(QiT, Rc);
      double c[3];
      mulv(QiT, d->com_pos + 3 * b, c);
      M3 J;
      std::memcpy(J.m, d->inertia + 9 * b, sizeof J.m);
      // symmetrise (validated above)
      J.m[3] = J.m[1] = 0.5 * (J.m[1] + J.m[3]);
      J.m[6] = J.m[2] = 0.5 * (J.m[2] + J.m[6]);
      J.m[7] = J.m[5] = 0.5 * (J.m[5] + J.m[7]);
      const M3 Ib = mul(mul(E, J), transpose(E));
      const double m = d->mass[b];
      const double cc = c[0] * c[0] + c[1] * c[1] + c[2] * c[2];
      double *rec = out.consts.data() + (size_t)i * MB_CONST_STRIDE;
      std::memcpy(rec + MB_C_R, R.m, sizeof R.m);
      std::memcpy(rec + MB_C_P, p, sizeof p);
      rec[MB_C_I + 0] = Ib.m[0] + m * (cc - c[0] * c[0]);
      rec[MB_C_I + 1] = 0.5 * (Ib.m[1] + Ib.m[3]) - m * c[0] * c[1];
      rec[MB_C_I + 2] = 0.5 * (Ib.m[2] + Ib.m[6]) - m * c[0] * c[2];
      rec[MB_C_I + 3] = Ib.m[4] + m * (cc - c[1] * c[1]);
      rec[MB_C_I + 4] = 0.5 * (Ib.m[5] + Ib.m[7]) - m * c[1] * c[2];
      rec[MB_C_I + 5] = Ib.m[8] + m * (cc - c[2] * c[2]);
      rec[MB_C_H + 0] = m * c[0];
      rec[MB_C_H + 1] = m * c[1];
      rec[MB_C_H + 2] = m * c[2];
      rec[MB_C_M] = m;
      std::memcpy(rec + MB_C_E, E.m, sizeof E.m);
      std::memcpy(rec + MB_C_C, c, sizeof c);
      std::memcpy(rec + MB_C_Q, Q[i].m, sizeof Q[i].m);
      rec[MB_C_J + 0] = Ib.m[0];
      rec[MB_C_J + 1] = 0.5 * (Ib.m[1] + Ib.m[3]);
      rec[MB_C_J + 2] = 0.5 * (Ib.m[2] + Ib.m[6]);
      rec[MB_C_J + 3] = Ib.m[4];
      rec[MB_C_J + 4] = 0.5 * (Ib.m[5] + Ib.m[7]);
      rec[MB_C_J + 5] = Ib.m[8];
   }
   for (int i = nb - 1; i >= 0; i--)
   {
      if (subtree_end[i] == 0)
         subtree_end[i] = i + 1;
      if (parent_i[i] >= 0)
         subtree_end[parent_i[i]] = std::max(subtree_end[parent_i[i]], subtree_end[i]);
   }

   // ---- level tables (warp-per-state variant)
   out.level_of = depth;
   out.level_order.resize(nb);
   for (int i = 0; i < nb; i++)
      out.level_order[i] = i;
   std::stable_sort(out.level_order.begin(), out.level_order.end(), [&](int a, int b) { return depth[a] < depth[b]; });
   out.level_start.assign(out.max_depth + 1, 0);
   for (int i = 0; i < nb; i++)
      out.level_start[depth[i] + 1]++;
   for (int l = 0; l < out.max_depth; l++)
      out.level_start[l + 1] += out.level_start[l];

   // ---- traversal programs
   for (int algo = 0; algo < MB_NUM_ALGOS; algo++)
   {
      MbProgram &P = out.prog[algo];
      std::memset(&P, 0, sizeof P);
      P.nb = nb;
      P.nv = nv;
      P.nq = nq;
      P.max_depth = out.max_depth;
      int rec_extra = 0; // three-DoF joints: second half of the ABA pass-three record, behind the regular records
      for (int i = 0; i < nb; i++)
      {
         MbBody &B = P.body[i];
         const int b = order[i];
         B.parent = parent_i[i];
         // multi-DoF joints share the SixDoF class of the kernels (transform on the stack, rows read directly) and differ by sub-type
         B.jtype = d->joint_type[b] >= MECANO_B200_SIXDOF ? MB_SIXDOF : d->joint_type[b];
         B.sub = d->joint_type[b] == MECANO_B200_SPHERICAL ? MB_SUB_SPHERICAL : (d->joint_type[b] == MECANO_B200_PLANAR ? MB_SUB_PLANAR : MB_SUB_SIX);
         B.dof_off = d->dof_offset[b];
         B.cfg_off = d->cfg_offset[b];
         B.subtree_end = subtree_end[i];
         B.ext_index = d->wrench_index ? d->wrench_index[b] : b;
         B.depth = depth[i];
         B.ndof = joint_ndof(d->joint_type[b]);
         // stack slot: leaves keep everything in registers; others stack up along the current path
         const int pslot = parent_i[i] < 0 ? 0 : P.body[parent_i[i]].slot + (nchild[parent_i[i]] > 0 ? slot_size(algo, P.body[parent_i[i]].jtype) : 0);
         B.slot = pslot;
         if (nchild[i] > 0)
            P.stack_doubles = std::max(P.stack_doubles, B.slot + slot_size(algo, B.jtype));
         // branch save area, nested like a stack of branching ancestors
         int paux = 0;
         for (int a = parent_i[i]; a >= 0; a = parent_i[a])
            if (nchild[a] >= 2)
               paux += mb_algo(algo).aux;
         B.aux = nchild[i] >= 2 ? paux : -1;
         if (nchild[i] >= 2)
            P.aux_doubles = std::max(P.aux_doubles, paux + mb_algo(algo).aux);
         B.rec = -1;
         if (B.jtype == MB_SIXDOF && B.sub != MB_SUB_SIX)
         {
            B.rec = (nb + rec_extra) * (MB_ABA_REC / 2);
            rec_extra++;
         }
      }
      P.rec_doubles = algo == MB_ABA ? MB_ABA_REC * (nb + rec_extra) : 0;
      if (algo == MB_RNEA_DERIVATIVES)
         P.aux_doubles += 6 * (P.max_depth + 1); // the spatial acceleration of the open body at each depth (rnea_derivatives.cuh)

      // ops: iterative DFS emitting DESCEND on entry and ASCEND on exit
      int nops = 0;
      std::vector<int> path;            // bodies whose subtree is open
      std::vector<int> done_children(nb, 0);
      int prev_descend = -2;            // body of the previous op if it was a DESCEND, else -2
      for (int i = 0; i < nb; i++)
      {
         // close finished subtrees
         while (!path.empty() && subtree_end[path.back()] <= i)
         {
            const int c = path.back();
            path.pop_back();
            uint32_t w = MB_OP_ASCEND | ((uint32_t)c << 8);
            if (nchild[c] == 0) w |= MB_F_LEAF;
            const int p = parent_i[c];
            if (p < 0)
               w |= MB_F_ROOT_PARENT;
            else
            {
               if (done_children[p] == 0) w |= MB_F_FIRST_CHILD;
               done_children[p]++;
               if (done_children[p] < nchild[p]) w |= MB_F_STORE_ACC;
            }
            P.op[nops++] = w;
            prev_descend = -2;
         }
         uint32_t w = ((uint32_t)i << 8);
         if (nchild[i] == 0) w |= MB_F_LEAF;
         if (nchild[i] >= 2) w |= MB_F_SAVE_STATE;
         if (parent_i[i] < 0)
            w |= MB_F_ROOT_PARENT;
         else if (prev_descend != parent_i[i])
            w |= MB_F_LOAD_PARENT;
         P.op[nops++] = w;
         prev_descend = i;
         path.push_back(i);
      }
      while (!path.empty())
      {
         const int c = path.back();
         path.pop_back();
         uint32_t w = MB_OP_ASCEND | ((uint32_t)c << 8);
         if (nchild[c] == 0) w |= MB_F_LEAF;
         const int p = parent_i[c];
         if (p < 0)
            w |= MB_F_ROOT_PARENT;
         else
         {
            if (done_children[p] == 0) w |= MB_F_FIRST_CHILD;
            done_children[p]++;
            if (done_children[p] < nchild[p]) w |= MB_F_STORE_ACC;
         }
         P.op[nops++] = w;
      }
      P.nops = nops;
      build_op2(algo, P, nchild);
   }
   // ---- structural zeros of the mass matrix: DoF pairs of bodies on unrelated branches
   {
      const MbProgram &P = out.prog[MB_CRBA];
      for (int i = 0; i < nb; i++)
         for (int j = 0; j < nb; j++)
         {
            if (i == j)
               continue;
            const bool related = (j > i && j < subtree_end[i]) || (i > j && i < subtree_end[j]);
            if (related)
               continue;
            for (int r = 0; r < P.body[i].ndof; r++)
               for (int s = 0; s < P.body[j].ndof; s++)
                  out.zero_entries.push_back((uint16_t)((P.body[i].dof_off + r) * nv + P.body[j].dof_off + s));
         }
      while (!out.zero_entries.empty() && out.zero_entries.size() % 8 != 0)
         out.zero_entries.push_back(out.zero_entries.back());
      // packed layout index map: for every column (DoF r of body i) the DoFs on the path from the root down to and including
      // that DoF, in the order the kernel's packed row numbers follow (MbWalk::pcol / above)
      for (int i = 0; i < nb; i++)
         for (int r = 0; r < P.body[i].ndof; r++)
         {
            std::vector<int> path;
            for (int a = i; a >= 0; a = P.body[a].parent)
               path.push_back(a);
            for (auto it = path.rbegin(); it != path.rend(); ++it)
               for (int k = 0; k < (*it == i ? r + 1 : P.body[*it].ndof); k++)
               {
                  out.packed_row.push_back(P.body[*it].dof_off + k);
                  out.packed_col.push_back(P.body[i].dof_off + r);
               }
            if (r == 0 && (int)out.packed_row.size() - (P.walk[i].above + 1) != P.walk[i].pcol)
            {
               err = "internal error: packed mass-matrix column table";
               return MECANO_B200_ERR_INVALID_ARGUMENT;
            }
         }
      // DoF order of the L^T D L factor: bodies in pre-order, a joint's DoFs as a chain, so every DoF parent comes first
      std::vector<int> last_dof(nb, -1);
      for (int i = 0; i < nb; i++)
         for (int r = 0; r < P.body[i].ndof; r++)
         {
            const int k = (int)out.ltdl_dof.size();
            out.ltdl_parent.push_back((int16_t)(r > 0 ? k - 1 : (P.body[i].parent >= 0 ? last_dof[P.body[i].parent] : -1)));
            out.ltdl_dof.push_back((int16_t)(P.body[i].dof_off + r));
            last_dof[i] = k;
         }
   }
   // ---- structural zeros of the joint-torque regressor: in the block of body i, the DoF rows of the joints that are not on the
   //      path from the root to i (flatten.h); only for wrench_index ranks that fit the 10 nb columns (api.cu refuses the others)
   {
      const MbProgram &P = out.prog[MB_REGRESSOR];
      bool cols_ok = true;
      for (int i = 0; i < nb; i++)
         cols_ok = cols_ok && P.body[i].ext_index < nb;
      for (int i = 0; i < nb && cols_ok; i++)
         for (int j = 0; j < nb; j++)
         {
            if (j <= i && i < subtree_end[j])
               continue; // j is i or an ancestor of i
            for (int r = 0; r < P.body[j].ndof; r++)
               out.regressor_zero_rows.push_back((uint32_t)((P.body[j].dof_off + r) * 10 * nb + 10 * P.body[i].ext_index));
         }
   }
   return MECANO_B200_OK;
}
int apply_source_modes(FlatTree &t, const int32_t *accel_source, std::vector<std::pair<int, int>> &effort_dof_runs)
{
   MbProgram &P = t.prog[MB_ABA];
   std::vector<char> locked((size_t)t.nb, 0); // by internal index
   int count = 0;
   if (accel_source)
      for (int b = 0; b < t.nb; b++)
         if (accel_source[b])
         {
            locked[(size_t)t.internal_of[(size_t)b]] = 1;
            count++;
         }
   for (int k = 0; k < P.nops; k++)
      if (P.op2[k].code & MB2_ASCEND)
         P.op2[k].flags = (uint8_t)((P.op2[k].flags & ~MB2_ACCSRC) | (locked[P.op2[k].body] ? MB2_ACCSRC : 0u));
   for (int k = 0; k < P.nb; k++) // pass three: one record per body
      P.op3[k].flags = (uint8_t)((P.op3[k].flags & ~MB2_ACCSRC) | (locked[P.op3[k].body] ? MB2_ACCSRC : 0u));
   build_runs(MB_ABA, P, P.nb); // a locked joint is not a plain op
   // DoF rows of the joints that stay EFFORT_SOURCE, as runs of consecutive rows
   std::vector<char> effort((size_t)t.nv, 1);
   for (int i = 0; i < t.nb; i++)
      if (locked[(size_t)i])
         for (int k = 0; k < P.body[i].ndof; k++)
            effort[(size_t)(P.body[i].dof_off + k)] = 0;
   effort_dof_runs.clear();
   for (int r = 0; r < t.nv;)
   {
      if (!effort[(size_t)r]) { r++; continue; }
      int e = r;
      while (e < t.nv && effort[(size_t)e]) e++;
      effort_dof_runs.emplace_back(r, e - r);
      r = e;
   }
   return count;
}
} // namespace mb
