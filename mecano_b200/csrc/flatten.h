// flatten.h -- host-side construction of the kernel tables from a mecano_b200_tree_desc.
// The analogue of Mecano's calculator constructors mirroring the body tree into RecursionStep objects
// (M/algorithms/InverseDynamicsCalculator.java:253-282, ForwardDynamicsCalculator.java:198-222,
//  CompositeRigidBodyMassMatrixCalculator.java:242-266), done once per handle.
#pragma once
#include <string>
#include <utility>
#include <vector>

#include "../../include/mecano_b200.h"
#include "program.h"

namespace mb
{
struct FlatTree
{
   int nb = 0, nv = 0, nq = 0, max_depth = 0;
   std::vector<double> consts;      // [nb][MB_CONST_STRIDE], internal (DFS) order
   std::vector<int> internal_of;    // caller's body index -> internal index
   std::vector<int> level_of;       // internal index -> tree level (0 = attached to the root body)
   std::vector<int> level_order;    // internal indices sorted by level (for the warp-per-state variant)
   std::vector<int> level_start;    // [n_levels + 1] into level_order
   std::vector<uint16_t> zero_entries; // mass-matrix entries (row * nv + col) that are structurally zero, padded to a multiple of 8
   // packed mass-matrix layout (MECANO_B200_CRBA_PACKED): packed row p holds M[packed_row[p]][packed_col[p]] (= the mirrored
   // entry); one row per unique entry that is not structurally zero, column by column, path from the root first
   std::vector<int32_t> packed_row, packed_col;
   // the DoF tree of the forward-dynamics derivatives' L^T D L factor (ltdl_solve.cuh): DoF k in internal pre-order (a multi-DoF
   // joint as a chain of its DoFs) is row ltdl_dof[k] of the matrices; its DoF parent ltdl_parent[k] < k, -1 at a root joint
   std::vector<int16_t> ltdl_dof, ltdl_parent;
   // joint-torque regressor (MB_REGRESSOR): the structurally zero rows of each body's block, as the entry of the row's first
   // column (row * 10 nb + 10 w); a row's ten columns are zero together.  Empty if a wrench_index rank is >= nb.
   std::vector<uint32_t> regressor_zero_rows;
   MbProgram prog[MB_NUM_ALGOS];    // MB_RNEA, MB_ABA, MB_CRBA, MB_CORIOLIS, MB_REGRESSOR, MB_GRAVITY_GRADIENT, MB_RNEA_DERIVATIVES
};

// Returns MECANO_B200_OK or a negative error code; `err` receives the message.
int flatten_tree(const mecano_b200_tree_desc *desc, FlatTree &out, std::string &err);

// ForwardDynamicsCalculator.setJointSourceMode (ForwardDynamicsCalculator.java:400-403) on the flattened ABA program:
// accel_source [nb] in the caller's body order (NULL = every joint back to EFFORT_SOURCE) marks the ASCEND ops of the
// ACCELERATION_SOURCE joints; effort_dof_runs receives the (first row, count) runs of DoF rows that stay EFFORT_SOURCE.
// Returns the number of ACCELERATION_SOURCE joints.
int apply_source_modes(FlatTree &t, const int32_t *accel_source, std::vector<std::pair<int, int>> &effort_dof_runs);
} // namespace mb
