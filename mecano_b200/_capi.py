"""ctypes binding of the C ABI (include/mecano_b200.h).

The shared library holds hand-written sm_100a kernels only.  If it is missing this module raises at
import time: there is no CPU fallback and none is wanted.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MECANO_B200_LIB") or os.path.join(_HERE, "libmecano_b200.so")  # (override: kernel variants of scripts/build_variants.sh)

if not os.path.exists(LIB_PATH):
    raise ImportError(
        "mecano_b200: %s not found. Build the CUDA extension first (python -c 'import __graft_entry__ as g; g.build()' "
        "or make -C mecano_b200/csrc). There is no CPU fallback." % LIB_PATH)

lib = ctypes.CDLL(LIB_PATH)

c_dp = ctypes.POINTER(ctypes.c_double)
c_ip = ctypes.POINTER(ctypes.c_int32)
c_vp = ctypes.c_void_p
c_i64 = ctypes.c_int64
c_u32 = ctypes.c_uint32

REVOLUTE, PRISMATIC, SIXDOF = 0, 1, 2
RNEA_NO_CORIOLIS, RNEA_NO_ACCELERATIONS = 1, 2
CRBA_ENTRY_MAJOR, CRBA_STATE_MAJOR = 0, 1
CRBA_ZEROS_PRESENT = 2  # structurally zero entries already hold zeros (same tree, same buffer): not written / transferred again
CRBA_PACKED = 4  # one row per unique, structurally non-zero entry (mecano_b200_crba_packed_index gives the map)
ALGO_RNEA, ALGO_ABA, ALGO_CRBA = 0, 1, 2
ALGO_REGRESSOR = 4
ALGO_GRAVITY_GRADIENT = 5
ALGO_RNEA_DERIVATIVES = 6
# column order of a body's ten inertial parameters in the joint-torque regressor (MECANO_B200_REGRESSOR_*): mass, first of the
# first moments m c (x y z), first of the moments of inertia about the origin (xx xy xz yy yz zz)
REGRESSOR_M, REGRESSOR_MC, REGRESSOR_I = 0, 1, 4
FRAME_WORLD, FRAME_CENTER_OF_MASS = 0, 1


class TreeDesc(ctypes.Structure):
    """mecano_b200_tree_desc"""
    _fields_ = [
        ("struct_size", ctypes.c_int32), ("n_bodies", ctypes.c_int32), ("n_dofs", ctypes.c_int32), ("n_cfg", ctypes.c_int32),
        ("n_levels", ctypes.c_int32), ("level_start", c_ip), ("parent", c_ip), ("joint_type", c_ip), ("axis", c_dp),
        ("offset_rot", c_dp), ("offset_pos", c_dp), ("com_rot", c_dp), ("com_pos", c_dp), ("inertia", c_dp), ("mass", c_dp),
        ("dof_offset", c_ip), ("cfg_offset", c_ip), ("wrench_index", c_ip),
    ]


class KernelInfo(ctypes.Structure):
    """mecano_b200_kernel_info"""
    _fields_ = [
        ("variant", ctypes.c_int32), ("block_threads", ctypes.c_int32), ("states_per_block", ctypes.c_int32),
        ("regs_per_thread", ctypes.c_int32), ("static_smem_bytes", ctypes.c_int32), ("dynamic_smem_bytes", ctypes.c_int32),
        ("local_bytes_per_thread", ctypes.c_int32), ("blocks_per_sm", ctypes.c_int32), ("sm_count", ctypes.c_int32),
        ("stack_doubles", ctypes.c_int32), ("max_depth", ctypes.c_int32), ("specialized", ctypes.c_int32),
        ("bytes_per_state", ctypes.c_double), ("tmem_stack_slots", ctypes.c_int32), ("reserved", ctypes.c_int32),
        ("jit_seconds", ctypes.c_double),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_ if name != "reserved"}


EXPORTS = [
    "mecano_b200_version", "mecano_b200_device_count", "mecano_b200_create", "mecano_b200_destroy", "mecano_b200_last_error",
    "mecano_b200_set_gravity", "mecano_b200_set_variant", "mecano_b200_n_dofs", "mecano_b200_n_cfg", "mecano_b200_n_bodies",
    "mecano_b200_rnea", "mecano_b200_aba", "mecano_b200_crba", "mecano_b200_rnea_host", "mecano_b200_aba_host",
    "mecano_b200_crba_host", "mecano_b200_kernel_info_get", "mecano_b200_measure_fp64_peak", "mecano_b200_measure_fp64_sustained", "mecano_b200_measure_hbm_peak",
    "mecano_b200_integrate", "mecano_b200_integrate_host", "mecano_b200_host_alloc", "mecano_b200_host_free", "mecano_b200_generate_source", "mecano_b200_jit_check", "mecano_b200_specialize",
    "mecano_b200_rnea_full", "mecano_b200_rnea_full_host",
    "mecano_b200_set_joint_source_modes", "mecano_b200_aba_sources", "mecano_b200_aba_sources_host",
    "mecano_b200_crba_centroidal", "mecano_b200_centroidal_convective_term", "mecano_b200_crba_centroidal_host",
    "mecano_b200_centroidal_convective_term_host", "mecano_b200_center_of_mass", "mecano_b200_center_of_mass_host", "mecano_b200_coriolis", "mecano_b200_coriolis_host", "mecano_b200_set_grid_limit", "mecano_b200_set_precision",
    "mecano_b200_crba_packed_size", "mecano_b200_crba_packed_index", "mecano_b200_step_host",
    "mecano_b200_multi_create", "mecano_b200_multi_destroy", "mecano_b200_multi_last_error", "mecano_b200_multi_size", "mecano_b200_multi_handle",
    "mecano_b200_multi_slice", "mecano_b200_multi_set_gravity", "mecano_b200_multi_rnea_host", "mecano_b200_multi_aba_host",
    "mecano_b200_multi_crba_host", "mecano_b200_multi_step_host",
    "mecano_b200_joint_torque_regressor", "mecano_b200_joint_torque_regressor_host",
    "mecano_b200_gravity_gradient", "mecano_b200_gravity_gradient_host",
    "mecano_b200_rnea_derivatives", "mecano_b200_rnea_derivatives_host",
    "mecano_b200_aba_derivatives", "mecano_b200_aba_derivatives_host",
]

lib.mecano_b200_create.argtypes = [ctypes.POINTER(TreeDesc), ctypes.c_int, ctypes.POINTER(c_vp)]
lib.mecano_b200_destroy.argtypes = [c_vp]
lib.mecano_b200_destroy.restype = None
lib.mecano_b200_last_error.argtypes = [c_vp]
lib.mecano_b200_last_error.restype = ctypes.c_char_p
lib.mecano_b200_set_gravity.argtypes = [c_vp, ctypes.c_double, ctypes.c_double, ctypes.c_double]
lib.mecano_b200_set_variant.argtypes = [c_vp, ctypes.c_int]
lib.mecano_b200_set_precision.argtypes = [c_vp, ctypes.c_int]
lib.mecano_b200_set_grid_limit.argtypes = [c_vp, ctypes.c_int, ctypes.c_int]
lib.mecano_b200_specialize.argtypes = [c_vp, c_u32]
lib.mecano_b200_jit_check.argtypes = [ctypes.POINTER(TreeDesc), ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.POINTER(c_i64)]
for _f in ("mecano_b200_n_dofs", "mecano_b200_n_cfg", "mecano_b200_n_bodies"):
    getattr(lib, _f).argtypes = [c_vp]
lib.mecano_b200_rnea.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_u32, c_vp]
lib.mecano_b200_rnea_full.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_u32, c_vp]
lib.mecano_b200_rnea_full_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_u32]
lib.mecano_b200_aba.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_u32, c_vp]
lib.mecano_b200_set_joint_source_modes.argtypes = [c_vp, c_vp]
lib.mecano_b200_aba_sources.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]
lib.mecano_b200_aba_sources_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]
lib.mecano_b200_crba_centroidal.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, ctypes.c_int, c_vp]
lib.mecano_b200_centroidal_convective_term.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, ctypes.c_int, c_vp]
lib.mecano_b200_crba_centroidal_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, ctypes.c_int]
lib.mecano_b200_centroidal_convective_term_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, ctypes.c_int]
lib.mecano_b200_center_of_mass.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp]
lib.mecano_b200_center_of_mass_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp]
lib.mecano_b200_coriolis.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]
lib.mecano_b200_coriolis_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp]
lib.mecano_b200_joint_torque_regressor.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]
lib.mecano_b200_joint_torque_regressor_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp]
lib.mecano_b200_gravity_gradient.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]
lib.mecano_b200_gravity_gradient_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp]
lib.mecano_b200_rnea_derivatives.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]
lib.mecano_b200_rnea_derivatives_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]
lib.mecano_b200_aba_derivatives.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]
lib.mecano_b200_aba_derivatives_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]
lib.mecano_b200_crba.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_u32, c_vp]
lib.mecano_b200_rnea_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_u32]
lib.mecano_b200_aba_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_u32]
lib.mecano_b200_crba_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_u32]
lib.mecano_b200_integrate.argtypes = [c_vp, c_i64, c_i64, ctypes.c_double, c_vp, c_vp, c_vp, c_vp]
lib.mecano_b200_integrate_host.argtypes = [c_vp, c_i64, c_i64, ctypes.c_double, c_vp, c_vp, c_vp]
lib.mecano_b200_kernel_info_get.argtypes = [c_vp, ctypes.c_int, c_i64, ctypes.POINTER(KernelInfo)]
lib.mecano_b200_measure_fp64_peak.argtypes = [ctypes.c_int, c_dp]
lib.mecano_b200_measure_fp64_sustained.argtypes = [ctypes.c_int, ctypes.c_double, c_dp]
lib.mecano_b200_measure_hbm_peak.argtypes = [ctypes.c_int, c_dp]
lib.mecano_b200_host_alloc.argtypes = [ctypes.POINTER(c_vp), c_i64]
lib.mecano_b200_host_free.argtypes = [c_vp]
lib.mecano_b200_crba_packed_size.argtypes = [c_vp]
lib.mecano_b200_crba_packed_index.argtypes = [c_vp, c_vp, c_vp]
lib.mecano_b200_step_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_u32]
lib.mecano_b200_multi_create.argtypes = [ctypes.POINTER(TreeDesc), c_vp, ctypes.c_int, ctypes.POINTER(c_vp)]
lib.mecano_b200_multi_destroy.argtypes = [c_vp]
lib.mecano_b200_multi_destroy.restype = None
lib.mecano_b200_multi_last_error.argtypes = [c_vp]
lib.mecano_b200_multi_last_error.restype = ctypes.c_char_p
lib.mecano_b200_multi_size.argtypes = [c_vp]
lib.mecano_b200_multi_handle.argtypes = [c_vp, ctypes.c_int]
lib.mecano_b200_multi_handle.restype = c_vp
lib.mecano_b200_multi_slice.argtypes = [c_vp, c_i64, ctypes.c_int, ctypes.POINTER(c_i64), ctypes.POINTER(c_i64)]
lib.mecano_b200_multi_set_gravity.argtypes = [c_vp, ctypes.c_double, ctypes.c_double, ctypes.c_double]
lib.mecano_b200_multi_rnea_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_u32]
lib.mecano_b200_multi_aba_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_u32]
lib.mecano_b200_multi_crba_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_u32]
lib.mecano_b200_multi_step_host.argtypes = [c_vp, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_u32]
lib.mecano_b200_generate_source.argtypes = [ctypes.POINTER(TreeDesc), ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_char_p, c_i64, ctypes.POINTER(c_i64)]


class MecanoB200Error(RuntimeError):
    def __init__(self, code, message):
        super().__init__("mecano_b200 error %d: %s" % (code, message))
        self.code = code


def check(rc, handle=None):
    if rc != 0:
        msg = lib.mecano_b200_last_error(handle)
        raise MecanoB200Error(rc, msg.decode() if msg else "")
