// emu_layout.cpp -- the per-state stack sizes of the flattened traversal programs, as the launch planner reads them
// (TEST INFRASTRUCTURE, never shipped or loaded by the product).  tests/test_launch_configurations.py checks the planner's
// refusals of the tensor-memory configurations against program.h: mb_tm_fits, which depends on the wide stack area.
#include <string>

#include "../../mecano_b200/csrc/flatten.h"

// wide (TMEM-capable) and narrow stack areas of one algorithm, double2 slots per state; returns the flattener's error code
extern "C" int emu_stack_areas(const mecano_b200_tree_desc *d, int algo, int *wide, int *narrow)
{
   mb::FlatTree ft;
   std::string e;
   const int rc = mb::flatten_tree(d, ft, e);
   if (rc != 0) return rc;
   *wide = ft.prog[algo].wstack2;
   *narrow = ft.prog[algo].nstack2;
   return 0;
}
