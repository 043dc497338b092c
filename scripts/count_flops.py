"""Flops per state of RNEA / ABA / CRBA / the joint-torque regressor / the gravity gradient / the inverse-dynamics derivatives: the per-state kernel
routines instantiated with a counting scalar (tests/emu).

Two files, both read by bench.py:
  profiles/algorithmic_flops.json  FROZEN.  The ALGORITHMIC work of SURVEY.md 8d: the count of the plain local-transform
      formulation (f = I a + v x* I v about the joint origin, full 3-block congruence, no structural shortcuts) as the
      kernels implemented it at commit b11b22e.  It defines the problem, not the program: the FP64 roofline fraction is
      (this count) / time / peak, so a kernel that needs fewer operations for the same result scores higher, the way a
      GEMM is rated at 2 N^3 whatever the algorithm.  Not rewritten by this script.
  profiles/executed_flops.json     what the current routines execute (Newton-Euler from CoM quantities, exact zeros of the
      downdated articulated inertia, accumulating multiply-add chains); rewritten by this script."""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import emu_gravity_gradient_lib as egl  # noqa: E402
import emu_lib as el  # noqa: E402
import emu_regressor_lib as erl  # noqa: E402
import emu_rnea_derivatives_lib as erd  # noqa: E402
import treedesc as td  # noqa: E402

out = {"_definition": "add/sub/mul/div = 1 flop (FMA = 2); sin/cos pairs counted separately; the CURRENT routines of "
                      "mecano_b200/csrc/{rnea,aba,crba,regressor,gravity_gradient,rnea_derivatives}.cuh instantiated with a counting scalar "
                      "(tests/emu/emu.cpp, emu_regressor.cpp, emu_gravity_gradient.cpp, emu_rnea_derivatives.cpp; the gravity gradient and the "
                      "inverse-dynamics derivatives without external wrenches)"}
rng = np.random.default_rng(1)
for key, tree in (("A7", td.chain(rng, 7)), ("H36", td.humanoid(rng, 1)), ("H37", td.humanoid(rng, 2))):
    e = el.Emu(tree)
    q, qd, qdd, tau = td.random_states(rng, tree, 1)
    r = {"rnea": e.count_flops(0, q, qd, qdd), "aba": e.count_flops(1, q, qd, tau), "crba": e.count_flops(2, q, qd, tau),
         "regressor": erl.count_flops(tree, q, qd, qdd), "gravity_gradient": egl.count_flops(tree, q),
         "rnea_derivatives": erd.count_flops(tree, q, qd, qdd)}
    out[key] = {k: v["flops"] for k, v in r.items()}
    out[key + "_detail"] = r
    print(key, out[key], {k: v["sincos"] for k, v in r.items()})
json.dump(out, open(os.path.join(ROOT, "profiles", "executed_flops.json"), "w"), indent=1)
