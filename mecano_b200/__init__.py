"""mecano_b200 -- B200-native batched rigid-body dynamics behind Mecano's calculator API.

Only what the hot path needs: the C-ABI binding (_capi), the low-level engine and the host-side mirror
of the reference interface (multibody / calculators).  Importing fails loudly when the CUDA library has
not been built: there is no CPU fallback.
"""
from . import _capi  # noqa: F401  (raises ImportError if libmecano_b200.so is missing)
from ._capi import MecanoB200Error  # noqa: F401
from .calculators import (CompositeRigidBodyMassMatrixCalculator, ForwardDynamicsCalculator,  # noqa: F401
                          ForwardDynamicsDerivativesCalculator, InverseDynamicsCalculator, InverseDynamicsDerivativesCalculator,
                          JointSourceMode, JointTorqueRegressorCalculator, MatrixDimensionException, MultiBodyDynamicsStep,
                          MultiBodyGravityGradientCalculator, MultiBodySystemStateIntegrator)
from .engine import Engine, MultiDeviceEngine, measure_fp64_peak, measure_fp64_sustained, measure_hbm_peak  # noqa: F401
from .multibody import (FixedJoint, JointMatrixIndexProvider, MultiBodySystem, MultiBodySystemRandomTools, PlanarJoint, PrismaticJoint,  # noqa: F401
                        RevoluteJoint, RigidBody, RigidBodyTransform, ScrewTheoryException, SixDoFJoint, SphericalJoint)
