"""Batched mirrors of Mecano's three calculators (Python face; the C++ face is csrc/host/calculators.hpp).

    InverseDynamicsCalculator                 M/algorithms/InverseDynamicsCalculator.java:201-251, 291-306, 343-403, 469-472, 496-501, 567-570
    ForwardDynamicsCalculator                 M/algorithms/ForwardDynamicsCalculator.java:128-196, 313-319, 508-520, 556-567
    CompositeRigidBodyMassMatrixCalculator    M/algorithms/CompositeRigidBodyMassMatrixCalculator.java:182-233, 286-291, 344-348
    JointTorqueRegressorCalculator            the inertial-parameter regressor of inverse dynamics (project definition, see the class)
    MultiBodyGravityGradientCalculator        gravity torques and their configuration gradient (project definition, see the class)
    InverseDynamicsDerivativesCalculator      d tau / dq and d tau / dqd of inverse dynamics (project definition, see the class)
    ForwardDynamicsDerivativesCalculator      d qdd / dq, d qdd / dqd and M^-1 of forward dynamics (project definition, see the class)

Same names, argument meaning and error behaviour as the reference; the batching changes are that the joint state
is passed explicitly as [rows, N] matrices (Mecano reads it from the joint objects) and that results come back as
[rows, N] matrices.  Inputs may be float64 torch CUDA tensors (device path, asynchronous on the current stream) or
float64 numpy arrays (host path through the *_host C-ABI entry points, which stage through the GPU).  There is no
CPU implementation behind these classes.
"""
import numpy as np

from . import _capi
from .engine import Engine, MultiDeviceEngine
from .multibody import MultiBodySystem, RigidBody


class MatrixDimensionException(ValueError):
    """EJML's MatrixDimensionException (ForwardDynamicsCalculator.java:522-533)."""


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _make_engine(input, device):
    """device: one CUDA device index, or a list of them (MultiDeviceEngine: host matrices sliced across the GPUs of the box)."""
    if isinstance(device, (list, tuple)):
        return MultiDeviceEngine(input.tables().contents, device, keepalive=input)
    return Engine(input.tables().contents, device, keepalive=input)


class _BatchedCalculator:
    def __init__(self, input, device=0):
        if isinstance(input, RigidBody):  # InverseDynamicsCalculator(RigidBodyReadOnly rootBody), :186
            input = MultiBodySystem.toMultiBodySystemBasics(input)
        self._input = input
        self._device = device
        self._engine = _make_engine(input, device)
        self._xengine = None  # engine over the expanded tables (systems with fixed / ignored joints; lazy)
        self._fext = None
        self._gravity = (0.0, 0.0, 0.0)

    def getInput(self):
        return self._input

    def setGravitationalAcceleration(self, *gravity):
        """setGravitationalAcceleration(gz) | (gx, gy, gz) | (tuple3)  (InverseDynamicsCalculator.java:343-403)"""
        if len(gravity) == 1:
            g = gravity[0]
            g = (0.0, 0.0, float(g)) if np.isscalar(g) else tuple(float(v) for v in g)
        else:
            g = tuple(float(v) for v in gravity)
        if len(g) != 3:
            raise ValueError("gravity must have 3 components")
        self._gravity = g
        self._engine.set_gravity(*g)

    def setExternalWrenches(self, wrenches):
        """External wrench on the successor of every joint, [6 * nJoints, N] in JointMatrixIndexProvider order, each
        expressed in its body's CoM frame (setExternalWrench, InverseDynamicsCalculator.java:469-472, :819)."""
        self._fext = wrenches

    # ---- systems with fixed / ignored joints.  Their tables weld the successors of FixedJoints and the ignored subtrees into the
    # bodies that carry them (the fast path of every plain call).  A call with external wrenches or per-body results needs those
    # bodies back -- a wrench on a FixedJoint's successor acts where it is applied, every body reports its acceleration in its
    # own frame, a FixedJoint transmits a wrench (InverseDynamicsCalculator.java:469-472, :578-602 with :832-860) -- and runs on
    # the expanded tables instead (MultiBodySystem.expanded(): nothing welded, the fixed / ignored joints held at their
    # configuration with zero velocity and acceleration, their rows appended behind the system's own).
    def _expanded(self):
        if isinstance(self._device, (list, tuple)):
            raise NotImplementedError("external wrenches / per-body results on systems with fixed or ignored joints run on one device")
        x = self._input.expanded()
        if self._xengine is None:
            self._xengine = Engine(x.tables().contents, self._device, keepalive=self._input)
        self._xengine.set_gravity(*self._gravity)
        return self._xengine, x

    @staticmethod
    def _extended(m, extra_rows, fill=None):
        """[rows + extra_rows, N]: m on top; below it `fill` (one value per row, the same for every state) or zeros."""
        rows, n = m.shape
        if _is_torch(m):
            import torch

            out = torch.empty((rows + extra_rows, n), dtype=torch.float64, device=m.device)
            out[:rows] = m
            if extra_rows:
                out[rows:] = 0.0 if fill is None else torch.as_tensor(np.asarray(fill), dtype=torch.float64, device=m.device)[:, None]
            return out
        out = np.empty((rows + extra_rows, n), dtype=np.float64)
        out[:rows] = m
        if extra_rows:
            out[rows:] = 0.0 if fill is None else np.asarray(fill, dtype=np.float64)[:, None]
        return out

    def setExternalWrenchesToZero(self):
        self._fext = None

    def _check(self, name, m, rows, n):
        if m is None or m.ndim != 2 or m.shape[0] != rows or m.shape[1] != n:
            raise MatrixDimensionException("%s: expected a %d x %d matrix, got %s" % (name, rows, n, None if m is None else tuple(m.shape)))

    def _empty_like(self, ref, rows, n, match_ld=True):
        """Output matrix with the same leading dimension as `ref` (all matrices of one call share it)."""
        if _is_torch(ref):
            import torch

            ld = max(n, ref.stride(0)) if (match_ld and ref.dim() == 2 and ref.shape[0] > 1) else n
            return torch.empty((rows, ld), dtype=torch.float64, device=ref.device)[:, :n]
        ld = max(n, ref.strides[0] // 8) if (match_ld and ref.ndim == 2 and ref.shape[0] > 1) else n
        return np.empty((rows, ld), dtype=np.float64)[:, :n]

    def kernelInfo(self, n_states=0):
        return self._engine.kernel_info(self._ALGO, n_states)

    def setKernelVariant(self, variant):
        """"auto" (default: by batch size), "thread" (one thread per state) or "warp" (body-parallel, lane = body: one warp per state for
        trees of up to 32 bodies, a team of two to four warps up to 128; one-DoF and SixDoF joints; for small batches)."""
        self._engine.set_variant({"auto": 0, "thread": 1, "warp": 2}[variant] if isinstance(variant, str) else int(variant))
        return self

    def setPrecision(self, precision):
        """"fp64" (Mecano's, the default) or "fp32": the optional single-precision variant (arithmetic in float, matrices stay
        float64); plain compute() / getMassMatrix() calls only, tolerance 1e-5 (RNEA, CRBA) / 1e-4 (ABA).  Returns self."""
        self._engine.set_precision(precision)
        return self

    def setGridLimit(self, maxBlocks):
        """Cap this calculator's persistent grid at maxBlocks blocks (one block owns one SM; 0 = whole device), so that another
        calculator running at the same time on another stream finds free SMs (mecano_b200_set_grid_limit).  Returns self."""
        self._engine.set_grid_limit(self._ALGO, maxBlocks)
        return self

    def specialize(self, force=False):
        """Optional second half of the constructor: compile a kernel unrolled for this tree (mecano_b200_specialize).
        Trees whose unrolled code would overflow the instruction caches keep the generic kernel; kernelInfo()["specialized"]
        tells which one runs.  Returns self."""
        self._engine.specialize([self._ALGO], force=force)
        return self


class InverseDynamicsCalculator(_BatchedCalculator):
    _ALGO = _capi.ALGO_RNEA

    def __init__(self, input, device=0):
        super().__init__(input, device)
        self._coriolis = True
        self._accelerations = True
        self._tau = None
        self._want_acc = self._want_wrench = False
        self._body_acc = self._joint_wrench = None

    def setConsiderCoriolisAndCentrifugalForces(self, value):
        self._coriolis = bool(value)

    def setConsiderJointAccelerations(self, value):
        self._accelerations = bool(value)

    def areCoriolisAndCentrifugalForcesConsidered(self):
        return self._coriolis

    def areJointAccelerationsConsidered(self):
        return self._accelerations

    def setComputeByProducts(self, bodyAccelerations=True, jointWrenches=True):
        """Mecano's calculator always keeps the rigid-body accelerations and the joint wrenches of its last compute()
        (getBodyAcceleration, getComputedJointWrench; InverseDynamicsCalculator.java:578-602).  For N states these are two
        [6 * nJoints, N] matrices (12 * nBodies more rows of HBM traffic than the joint efforts), so the batched calculator
        writes them only on request.  Returns self."""
        self._want_acc, self._want_wrench = bool(bodyAccelerations), bool(jointWrenches)
        return self

    def compute(self, q, qd, qdd, tau=None):
        """compute(jointAccelerationMatrix) for N states; returns getJointTauMatrix() ([nDoFs, N])."""
        nv, nq = self._input.getNumberOfDoFs(), self._input.getConfigurationMatrixSize()
        n = q.shape[1] if q.ndim == 2 else -1
        self._check("q", q, nq, n)
        self._check("qd", qd, nv, n)
        self._check("qdd", qdd, nv, n)
        if tau is None:
            tau = self._empty_like(q, nv, n)
        self._check("tau", tau, nv, n)
        if self._fext is not None:
            self._check("externalWrenches", self._fext, 6 * self._input.getNumberOfJoints(), n)
        flags = (0 if self._coriolis else _capi.RNEA_NO_CORIOLIS) | (0 if self._accelerations else _capi.RNEA_NO_ACCELERATIONS)
        rows = 6 * self._input.getNumberOfJoints()
        if self._input.hasWeldedBodies() and (self._fext is not None or self._want_acc or self._want_wrench):
            # fixed / ignored joints: on the expanded tables (see _expanded)
            eng, x = self._expanded()
            q2 = self._extended(q, x.n_extra_cfg, x.q_extra)
            qd2, qdd2 = self._extended(qd, x.n_extra_dof), self._extended(qdd, x.n_extra_dof)
            tau2 = self._empty_like(q2, nv + x.n_extra_dof, n, match_ld=False)
            f2 = None if self._fext is None else self._extended(self._fext, 6 * x.n_extra_wrench_blocks)
            rows2 = rows + 6 * x.n_extra_wrench_blocks
            acc2 = self._empty_like(q2, rows2, n, match_ld=False) if self._want_acc else None
            wr2 = self._empty_like(q2, rows2, n, match_ld=False) if self._want_wrench else None
            (eng.rnea if _is_torch(q) else eng.rnea_host)(q2, qd2, qdd2, tau2, fext=f2, flags=flags, body_acc=acc2, joint_wrench=wr2)
            tau[:] = tau2[:nv]
            # the considered joints' blocks lead (the ignored bodies' follow): [6 * nJoints, N] views
            self._body_acc = None if acc2 is None else acc2[:rows]
            self._joint_wrench = None if wr2 is None else wr2[:rows]
            self._tau = tau
            return tau
        self._body_acc = self._empty_like(q, rows, n) if self._want_acc else None
        self._joint_wrench = self._empty_like(q, rows, n) if self._want_wrench else None
        if _is_torch(q):
            self._engine.rnea(q, qd, qdd, tau, fext=self._fext, flags=flags, body_acc=self._body_acc, joint_wrench=self._joint_wrench)
        else:
            self._engine.rnea_host(q, qd, qdd, tau, fext=self._fext, flags=flags, body_acc=self._body_acc, joint_wrench=self._joint_wrench)
        self._tau = tau
        return tau

    def getJointTauMatrix(self):
        return self._tau

    def getComputedJointTau(self, joint):
        """getComputedJointTau(joint) (InverseDynamicsCalculator.java:594-604) for N states: the [nDoFs(joint), N] rows of the joint."""
        if self._tau is None:
            return None
        rows = self._input.getJointMatrixIndexProvider().getJointDoFIndices(joint)
        return self._tau[rows[0]:rows[0] + len(rows)] if rows else self._tau[0:0]

    def getBodyAccelerationMatrix(self):
        """[6 * nJoints, N]: rows [6 j, 6 j + 6) = spatial acceleration (angular, linear) of the successor of joint j
        (JointMatrixIndexProvider order) expressed in its CoM frame; None unless setComputeByProducts() asked for it."""
        return self._body_acc

    def getComputedJointWrenchMatrix(self):
        """[6 * nJoints, N]: rows [6 j, 6 j + 6) = wrench (moment, force) transmitted by joint j, in its frameAfterJoint."""
        return self._joint_wrench

    def getBodyAcceleration(self, body):
        """getBodyAcceleration(body) (InverseDynamicsCalculator.java:578-591) for N states: [6, N], None for the root body."""
        if body.isRootBody() or self._body_acc is None:
            return None
        j = self._input.getAllJoints().index(body.getParentJoint())
        return self._body_acc[6 * j:6 * j + 6]

    def getComputedJointWrench(self, joint):
        """getComputedJointWrench(joint) (InverseDynamicsCalculator.java:593-602) for N states: [6, N]."""
        if self._joint_wrench is None:
            return None
        j = self._input.getAllJoints().index(joint)
        return self._joint_wrench[6 * j:6 * j + 6]


class JointSourceMode:
    """ForwardDynamicsCalculator.JointSourceMode (ForwardDynamicsCalculator.java:45-57)."""
    EFFORT_SOURCE = "EFFORT_SOURCE"
    ACCELERATION_SOURCE = "ACCELERATION_SOURCE"


class ForwardDynamicsCalculator(_BatchedCalculator):
    _ALGO = _capi.ALGO_ABA
    JointSourceMode = JointSourceMode

    def __init__(self, input, device=0):
        super().__init__(input, device)
        self._qdd = None
        self._tau = None
        self._modes = {}  # joint -> JointSourceMode, ACCELERATION_SOURCE entries only

    # ---- joint source modes (ForwardDynamicsCalculator.java:400-465)
    def setJointSourceMode(self, joint, mode):
        if mode not in (JointSourceMode.EFFORT_SOURCE, JointSourceMode.ACCELERATION_SOURCE):
            raise ValueError("unknown JointSourceMode %r" % (mode,))
        if self._input.tableRow(joint) < 0:
            raise ValueError("joint %s is not considered by this calculator" % joint.getName())
        if mode == JointSourceMode.ACCELERATION_SOURCE:
            self._modes[joint] = mode
        else:
            self._modes.pop(joint, None)
        self._push_modes()

    def setJointSourceModes(self, jointSourceModeFunction):
        """The function may return None for a joint to leave its mode unchanged (:422-433)."""
        for joint in self._input.getJointsToConsider():
            if self._input.tableRow(joint) < 0:
                continue
            mode = jointSourceModeFunction(joint)
            if mode == JointSourceMode.ACCELERATION_SOURCE:
                self._modes[joint] = mode
            elif mode == JointSourceMode.EFFORT_SOURCE:
                self._modes.pop(joint, None)
        self._push_modes()

    def resetJointSourceModes(self):
        self._modes.clear()
        self._push_modes()

    def getJointSourceMode(self, joint):
        return self._modes.get(joint, JointSourceMode.EFFORT_SOURCE)

    def _push_modes(self):
        if not self._modes:
            self._engine.set_joint_source_modes(None)
            return
        src = np.zeros(self._engine.nb, dtype=np.int32)
        for joint in self._modes:
            src[self._input.tableRow(joint)] = 1
        self._engine.set_joint_source_modes(src)

    def compute(self, q, qd, tau, qdd=None, jointAccelerationInput=None):
        """compute(jointTauMatrix[, jointAccelerationMatrix]) for N states (:489-520); returns getJointAccelerationMatrix()
        ([nDoFs, N]).  jointAccelerationInput ([nDoFs, N]) is only read at the rows of ACCELERATION_SOURCE joints, and is
        required when there are any; the efforts of those joints are then available from getJointTauMatrix()."""
        nv, nq = self._input.getNumberOfDoFs(), self._input.getConfigurationMatrixSize()
        n = q.shape[1] if q.ndim == 2 else -1
        self._check("q", q, nq, n)
        self._check("qd", qd, nv, n)
        self._check("tau", tau, nv, n)
        if qdd is None:
            qdd = self._empty_like(q, nv, n)
        self._check("qdd", qdd, nv, n)
        if self._fext is not None:
            self._check("externalWrenches", self._fext, 6 * self._input.getNumberOfJoints(), n)
        if self._modes:
            self._check("jointAccelerationInput", jointAccelerationInput, nv, n)
        if self._fext is not None and self._input.hasWeldedBodies():
            # fixed / ignored joints with external wrenches: on the expanded tables (see _expanded), the held joints locked
            # (ACCELERATION_SOURCE with zero acceleration, next to the caller's own ACCELERATION_SOURCE joints)
            eng, x = self._expanded()
            locked = x.locked.copy()
            considered = self._input.getJointsToConsider()
            for joint in self._modes:
                locked[x.row_of_considered[considered.index(joint)]] = 1
            eng.set_joint_source_modes(locked)
            q2 = self._extended(q, x.n_extra_cfg, x.q_extra)
            qd2, tau2 = self._extended(qd, x.n_extra_dof), self._extended(tau, x.n_extra_dof)
            acc_in = jointAccelerationInput if self._modes else (qd * 0.0)
            acc_in2 = self._extended(acc_in, x.n_extra_dof)
            qdd2 = self._empty_like(q2, nv + x.n_extra_dof, n, match_ld=False)
            tau_out2 = self._empty_like(q2, nv + x.n_extra_dof, n, match_ld=False)
            f2 = self._extended(self._fext, 6 * x.n_extra_wrench_blocks)
            (eng.aba_sources if _is_torch(q) else eng.aba_sources_host)(q2, qd2, tau2, acc_in2, qdd2, tau_out2, fext=f2)
            qdd[:] = qdd2[:nv]
            self._tau = tau_out2[:nv] if self._modes else tau
            self._qdd = qdd
            return qdd
        if self._modes:
            tau_out = self._empty_like(q, nv, n)
            run = self._engine.aba_sources if _is_torch(q) else self._engine.aba_sources_host
            run(q, qd, tau, jointAccelerationInput, qdd, tau_out, fext=self._fext)
            self._tau = tau_out
        else:
            if _is_torch(q):
                self._engine.aba(q, qd, tau, qdd, fext=self._fext)
            else:
                self._engine.aba_host(q, qd, tau, qdd, fext=self._fext)
            self._tau = tau  # every joint is an EFFORT_SOURCE: the efforts are the input
        self._qdd = qdd
        return qdd

    def getJointAccelerationMatrix(self):
        return self._qdd

    def getJointTauMatrix(self):
        """The joint efforts (:566-590): the input for EFFORT_SOURCE joints, computed for ACCELERATION_SOURCE joints."""
        return self._tau

    def _rows(self, matrix, joint):
        if matrix is None:
            return None
        rows = self._input.getJointMatrixIndexProvider().getJointDoFIndices(joint)
        return matrix[rows[0]:rows[0] + len(rows)] if rows else matrix[0:0]

    def getComputedJointAcceleration(self, joint):
        """getComputedJointAcceleration(joint) (:600-608) for N states: [nDoFs(joint), N]."""
        return self._rows(self._qdd, joint)

    def getJointTau(self, joint):
        """getJointTau(joint) (:622-630) for N states: [nDoFs(joint), N].  (The reference returns the joint's acceleration matrix
        there, `recursionStep.qdd`, against its own documentation; this returns the effort.)"""
        return self._rows(self._tau, joint)


class CompositeRigidBodyMassMatrixCalculator(_BatchedCalculator):
    _ALGO = _capi.ALGO_CRBA

    WORLD_FRAME = "worldFrame"                 # the inertial frame of the system
    CENTER_OF_MASS_FRAME = "centerOfMassFrame"  # axes of the inertial frame, origin at the centre of mass of each state

    def __init__(self, input, centroidalMomentumFrame=None, device=0):
        """CompositeRigidBodyMassMatrixCalculator(input[, centroidalMomentumFrame]) (:182-233).  Mecano takes any ReferenceFrame;
        the batched calculator offers the two that make sense for N states at once: WORLD_FRAME (the default, Mecano's is the
        inertial frame too, :184) and CENTER_OF_MASS_FRAME (Mecano's CenterOfMassReferenceFrame)."""
        super().__init__(input, device)
        self._M = None
        self._owned = {}
        self._cmm = self._com = self._convective = self._com_q = None
        self._frame = self.WORLD_FRAME
        if centroidalMomentumFrame is not None:
            self.setCentroidalMomentumFrame(centroidalMomentumFrame)

    def setCentroidalMomentumFrame(self, centroidalMomentumFrame):
        """setCentroidalMomentumFrame (:380-387)."""
        if centroidalMomentumFrame not in (self.WORLD_FRAME, self.CENTER_OF_MASS_FRAME):
            raise ValueError("centroidalMomentumFrame must be WORLD_FRAME or CENTER_OF_MASS_FRAME")
        if centroidalMomentumFrame != self._frame:
            self._cmm = self._convective = None
        self._frame = centroidalMomentumFrame

    def getCentroidalMomentumFrame(self):
        return self._frame

    def _frame_code(self):
        return _capi.FRAME_CENTER_OF_MASS if self._frame == self.CENTER_OF_MASS_FRAME else _capi.FRAME_WORLD

    def setEnableCoriolisMatrixCalculation(self, enableCoriolisMatrixCalculation):
        """setEnableCoriolisMatrixCalculation (:278-281); disabled by default, like the reference."""
        self._coriolis_enabled = bool(enableCoriolisMatrixCalculation)

    def getCoriolisMatrix(self, q, qd):
        """getCoriolisMatrix() (:358-366) for N states: [nDoFs * nDoFs, N], entry (i, j) of state s at [i * nDoFs + j, s]; times
        the joint velocities it gives the Coriolis and centrifugal joint efforts.  The mass matrix of the same states comes out
        of the same recursion (getMassMatrix() without an argument returns it).  Raises like the reference
        (UnsupportedOperationException) unless setEnableCoriolisMatrixCalculation(True) was called."""
        if not getattr(self, "_coriolis_enabled", False):
            raise RuntimeError("Coriolis matrix calculation is disabled.")
        nv, nq = self._input.getNumberOfDoFs(), self._input.getConfigurationMatrixSize()
        n = q.shape[1] if q.ndim == 2 else -1
        self._check("q", q, nq, n)
        self._check("qd", qd, nv, n)
        self._M = self._empty_like(q, nv * nv, n)
        self._C = self._empty_like(q, nv * nv, n)
        self._engine.coriolis(q, qd, self._M, self._C)
        return self._C

    def getCentroidalMomentumMatrix(self, q):
        """getCentroidalMomentumMatrix() (:411-416, :801-809) for N states: [6 * nDoFs, N], entry (r, j) of the 6 x nDoFs matrix of
        state s at [r * nDoFs + j, s] (angular rows first); times the joint velocities it gives the momentum of the system in the
        centroidal momentum frame.  The mass matrix of the same states is computed on the way (getMassMatrix() without an
        argument returns it), as are the centre of mass and total mass (getCenterOfMass())."""
        nv, nq = self._input.getNumberOfDoFs(), self._input.getConfigurationMatrixSize()
        n = q.shape[1] if q.ndim == 2 else -1
        self._check("q", q, nq, n)
        self._M = self._empty_like(q, nv * nv, n)
        self._cmm = self._empty_like(q, 6 * nv, n)
        self._com = self._empty_like(q, 4, n)
        self._engine.crba_centroidal(q, self._M, self._cmm, self._com, self._frame_code())
        self._com_q = q  # the configuration matrix the centre of mass belongs to (getCentroidalConvectiveTermMatrix)
        return self._cmm

    def getCenterOfMass(self, q=None):
        """[4, N]: centre of mass of the system in the root frame (x, y, z) and its total mass.  Without an argument: of the
        states last handed to getCentroidalMomentumMatrix() / getCentroidalConvectiveTermMatrix().  With `q`: computed for these
        states by the centre-of-mass-only launch (CenterOfMassCalculator.getCenterOfMass() + getTotalMass(),
        CenterOfMassCalculator.java:70-124; mecano_b200_center_of_mass) -- no matrix is computed or written, the rows are
        bit-identical to those getCentroidalMomentumMatrix(q) leaves."""
        if q is not None:
            nq = self._input.getConfigurationMatrixSize()
            n = q.shape[1] if q.ndim == 2 else -1
            self._check("q", q, nq, n)
            self._com = self._empty_like(q, 4, n)
            self._engine.center_of_mass(q, self._com)
            self._com_q = q
        return self._com

    def getCentroidalConvectiveTermMatrix(self, q, qd, reuseCenterOfMass=False):
        """getCentroidalConvectiveTermMatrix() (:423-440, :811-839) for N states: [6, N], moment first, in the centroidal momentum
        frame.  In CENTER_OF_MASS_FRAME the centre of mass is that of the `q` passed here: getCenterOfMass(q) runs first (the
        reference derives both from the same joint state after reset()).  reuseCenterOfMass=True skips that when the
        caller has just called getCentroidalMomentumMatrix() or getCenterOfMass() with this very `q` (same object, same batch); it is the caller's
        statement that the configuration has not changed since."""
        nv, nq = self._input.getNumberOfDoFs(), self._input.getConfigurationMatrixSize()
        n = q.shape[1] if q.ndim == 2 else -1
        self._check("q", q, nq, n)
        self._check("qd", qd, nv, n)
        com = None
        if self._frame == self.CENTER_OF_MASS_FRAME:
            fresh = reuseCenterOfMass and self._com is not None and self._com_q is q and self._com.shape[1] == n
            if not fresh:
                self.getCenterOfMass(q)
            com = self._com
        out = self._empty_like(q, 6, n)
        self._engine.centroidal_convective_term(q, qd, com, out, self._frame_code())
        self._convective = out
        return out

    def reset(self):
        """Mecano caches the mass matrix until reset(); the batched calculator recomputes on every getMassMatrix(q)."""
        self._M = None
        self._com = self._com_q = None

    def getMassMatrixPackedIndex(self):
        """(row, col) int32 arrays of the packed layout: packed row p of getMassMatrix(q, packed=True) is entry (row[p], col[p])
        of the symmetric mass matrix, and every entry the arrays do not list (in either order) is structurally zero."""
        return self._engine.packed_index()

    def getMassMatrix(self, q=None, massMatrix=None, stateMajor=False, packed=False):
        """Mass matrices for N states.  Default layout [nDoFs*nDoFs, N] (entry (i, j) of state s at [i*nDoFs + j, s]);
        stateMajor=True gives [N, nDoFs*nDoFs], i.e. one Mecano-style dense row-major nDoFs x nDoFs matrix per state;
        packed=True gives [P, N] with one row per unique entry that is not structurally zero (getMassMatrixPackedIndex() maps
        rows to entries; 362 rows instead of 1,369 for a 37-DoF humanoid), for callers that scatter into their own matrices.

        Without `massMatrix` the calculator owns the result like Mecano's does (getMassMatrix() returns a reference to the
        internal matrix, CompositeRigidBodyMassMatrixCalculator.java:344-348): one buffer per batch shape, reused by later
        calls.  The entries coupling joints of unrelated branches depend on the topology only, so they are written once and
        from the second call on neither rewritten nor (host path) transferred again (MECANO_B200_CRBA_ZEROS_PRESENT).  A
        caller-supplied `massMatrix` is always written in full."""
        if q is None:
            return self._M  # the matrices of the last call, like Mecano's cached getMassMatrix()
        nv, nq = self._input.getNumberOfDoFs(), self._input.getConfigurationMatrixSize()
        n = q.shape[1] if q.ndim == 2 else -1
        self._check("q", q, nq, n)
        if packed:
            if stateMajor:
                raise ValueError("packed and stateMajor are different layouts")
            if massMatrix is None:
                massMatrix = self._empty_like(q, self._engine.packed_size(), n)
            self._check("massMatrix", massMatrix, self._engine.packed_size(), n)
            (self._engine.crba if _is_torch(q) else self._engine.crba_host)(q, massMatrix, _capi.CRBA_PACKED)
            self._M = massMatrix
            return massMatrix
        shape = (n, nv * nv) if stateMajor else (nv * nv, n)
        layout = _capi.CRBA_STATE_MAJOR if stateMajor else _capi.CRBA_ENTRY_MAJOR
        owned_key = None
        if massMatrix is None:
            # entry-major: [nv*nv, n] sharing the leading dimension of q; state-major: one contiguous [n, nv*nv]
            ld = shape[1] if stateMajor or q.shape[0] < 2 else max(n, q.stride(0) if _is_torch(q) else q.strides[0] // 8)
            key = (n, ld, bool(stateMajor), str(q.device) if _is_torch(q) else "host")
            if key not in self._owned:
                self._owned.clear()  # one live result, like the reference
                self._owned[key] = [self._new_owned(q, shape, ld), False]
            massMatrix, primed = self._owned[key]
            if primed:
                layout |= _capi.CRBA_ZEROS_PRESENT
            owned_key = key
        self._check("massMatrix", massMatrix, *shape)
        if _is_torch(q):
            self._engine.crba(q, massMatrix, layout)
        else:
            self._engine.crba_host(q, massMatrix, layout)
        if owned_key is not None:
            self._owned[owned_key][1] = True  # (only once a call has been issued without error: a failed first call wrote no zeros)
        self._M = massMatrix
        return massMatrix

    @staticmethod
    def _new_owned(q, shape, ld):
        """[rows, ld] storage viewed as [rows, n]: all matrices of one call share the leading dimension of q."""
        rows, n = shape
        if _is_torch(q):
            import torch

            return torch.empty((rows, ld), dtype=torch.float64, device=q.device)[:, :n]
        try:  # page-locked, so that the device -> host copies run at full speed and asynchronously
            import torch

            return torch.empty((rows, ld), dtype=torch.float64).pin_memory().numpy()[:, :n]
        except Exception:
            return np.empty((rows, ld), dtype=np.float64)[:, :n]


class JointTorqueRegressorCalculator(_BatchedCalculator):
    """Mecano's JointTorqueRegressorCalculator for N states: the inertial-parameter regressor Y(q, qd, qdd) of inverse dynamics,
    tau = Y pi for any inertial parameters pi of the bodies (with gravity, without external wrenches).  What system
    identification stacks over a log of states to fit masses, centres of mass and inertias.

    Y is [nDoFs * 10 nBodies, N], entry (i, c) of state s at [i * 10 nBodies + c, s]: row i = DoF row, column block w (ten
    columns) = the successor of joint w (JointMatrixIndexProvider order), parameters m, m cx, m cy, m cz, Ixx, Ixy, Ixz, Iyy,
    Iyz, Izz in the order of the _capi.REGRESSOR_* table, c and I (about the origin) in the body's CoM frame.  On systems with
    fixed or ignored joints every body of the tree has its own block (the expanded tables, see _BatchedCalculator._expanded):
    nBodies counts them all, and the rows are the system's own nDoFs.  One device only."""
    _ALGO = _capi.ALGO_REGRESSOR

    def __init__(self, input, device=0):
        super().__init__(input, device)
        self._Y = None

    def _tables(self):
        """(engine, expanded system or None) that serve this calculator."""
        if isinstance(self._device, (list, tuple)):
            raise NotImplementedError("the joint-torque regressor runs on one device")
        if self._input.hasWeldedBodies():
            return self._expanded()
        return self._engine, None

    def compute(self, q, qd, qdd):
        """compute(q, qd, qdd) for N states; returns getJointTorqueRegressorMatrix() ([nDoFs * 10 nBodies, N])."""
        nv, nq = self._input.getNumberOfDoFs(), self._input.getConfigurationMatrixSize()
        n = q.shape[1] if q.ndim == 2 else -1
        self._check("q", q, nq, n)
        self._check("qd", qd, nv, n)
        self._check("qdd", qdd, nv, n)
        eng, x = self._tables()
        cols = 10 * eng.nb
        if x is None:
            Y = self._empty_like(q, nv * cols, n)
            eng.joint_torque_regressor(q, qd, qdd, Y)
        else:
            # the held joints' configuration / DoF rows follow the system's own: the leading nv rows of Y are the caller's
            q2 = self._extended(q, x.n_extra_cfg, x.q_extra)
            qd2, qdd2 = self._extended(qd, x.n_extra_dof), self._extended(qdd, x.n_extra_dof)
            Y2 = self._empty_like(q2, (nv + x.n_extra_dof) * cols, n, match_ld=False)
            eng.joint_torque_regressor(q2, qd2, qdd2, Y2)
            Y = Y2[:nv * cols]
        self._Y = Y
        return Y

    def getJointTorqueRegressorMatrix(self):
        return self._Y

    def getInertialParameterVector(self):
        """[10 nBodies]: the model's own parameters in the column order of Y, pi_w = [m, 0, 0, 0, J_xx, J_xy, J_xz, J_yy, J_yz, J_zz]
        (CoM frame: first moment zero, J about the CoM).  Y @ pi = the joint efforts of InverseDynamicsCalculator.compute."""
        eng, x = self._tables()
        d = (self._input if x is None else x).tables().contents
        nb = d.n_bodies
        pi = np.zeros(10 * nb)
        for b in range(nb):
            w = d.wrench_index[b] if d.wrench_index else b
            pi[10 * w + _capi.REGRESSOR_M] = d.mass[b]
            for k, e in enumerate((0, 1, 2, 4, 5, 8)):
                pi[10 * w + _capi.REGRESSOR_I + k] = d.inertia[9 * b + e]
        return pi


class MultiBodyGravityGradientCalculator(_BatchedCalculator):
    """Mecano's MultiBodyGravityGradientCalculator for N states: the joint efforts that gravity and the external wrenches cause,
    tau_g(q), and their configuration gradient G(q) = d tau_g / dq (mecano_b200_gravity_gradient in include/mecano_b200.h: column j
    is the derivative along the step the state integrator takes with qd = e_j, so a floating base's columns are perturbations in
    its own frame; external wrenches are body-fixed).  G is not symmetric in general.

    getTauMatrix() is [nDoFs, N]; getTauGradientMatrix() is [nDoFs * nDoFs, N], entry (i, j) of state s at [i * nDoFs + j, s].
    Systems with fixed or ignored joints run on their welded tables (lumping does not change gravity torques), or, with external
    wrenches, on the expanded tables (see _BatchedCalculator._expanded), of which the system's own rows and columns are returned.
    One device only."""
    _ALGO = _capi.ALGO_GRAVITY_GRADIENT

    def __init__(self, input, device=0):
        super().__init__(input, device)
        self._tau = self._G = None

    def compute(self, q):
        """compute(q) for N states; returns getTauGradientMatrix() ([nDoFs * nDoFs, N])."""
        if isinstance(self._device, (list, tuple)):
            raise NotImplementedError("the gravity gradient runs on one device")
        nv, nq = self._input.getNumberOfDoFs(), self._input.getConfigurationMatrixSize()
        n = q.shape[1] if q.ndim == 2 else -1
        self._check("q", q, nq, n)
        if self._fext is not None:
            self._check("externalWrenches", self._fext, 6 * self._input.getNumberOfJoints(), n)
        if self._fext is not None and self._input.hasWeldedBodies():
            eng, x = self._expanded()
            q2 = self._extended(q, x.n_extra_cfg, x.q_extra)
            nv2 = nv + x.n_extra_dof
            tau2 = self._empty_like(q2, nv2, n, match_ld=False)
            G2 = self._empty_like(q2, nv2 * nv2, n, match_ld=False)
            eng.gravity_gradient(q2, tau2, G2, fext=self._extended(self._fext, 6 * x.n_extra_wrench_blocks))
            # the held joints' DoFs follow the system's own in both the rows and the columns
            self._tau = tau2[:nv]
            self._G = G2.reshape(nv2, nv2, n)[:nv, :nv].reshape(nv * nv, n)
            return self._G
        self._tau = self._empty_like(q, nv, n)
        self._G = self._empty_like(q, nv * nv, n)
        self._engine.gravity_gradient(q, self._tau, self._G, fext=self._fext)
        return self._G

    def getTauMatrix(self):
        return self._tau

    def getTauGradientMatrix(self):
        return self._G


class InverseDynamicsDerivativesCalculator(_BatchedCalculator):
    """The first-order partials of inverse dynamics for N states: tau(q, qd, qdd) of InverseDynamicsCalculator together with
    d tau / dq and d tau / dqd (mecano_b200_rnea_derivatives in include/mecano_b200.h: column j of d tau / dq is the derivative along
    the step the state integrator takes with qd = e_j, so a floating base's columns are perturbations in its own frame; external
    wrenches are body-fixed).  d tau / dqdd is the mass matrix (CompositeRigidBodyMassMatrixCalculator).  Mecano has no counterpart:
    the definition is this project's, the one of MultiBodyGravityGradientCalculator extended to a moving state.

    getJointTauMatrix() is [nDoFs, N]; getTauConfigurationGradientMatrix() and getTauVelocityGradientMatrix() are [nDoFs * nDoFs, N],
    entry (i, j) of state s at [i * nDoFs + j, s].  Systems with fixed or ignored joints run on their welded tables, or, with external
    wrenches, on the expanded tables (see _BatchedCalculator._expanded), of which the system's own rows and columns are returned.
    One device only."""
    _ALGO = _capi.ALGO_RNEA_DERIVATIVES

    def __init__(self, input, device=0):
        super().__init__(input, device)
        self._tau = self._dq = self._dqd = None

    def compute(self, q, qd, qdd):
        """compute(q, qd, qdd) for N states; returns getTauConfigurationGradientMatrix() ([nDoFs * nDoFs, N])."""
        if isinstance(self._device, (list, tuple)):
            raise NotImplementedError("the inverse-dynamics derivatives run on one device")
        nv, nq = self._input.getNumberOfDoFs(), self._input.getConfigurationMatrixSize()
        n = q.shape[1] if q.ndim == 2 else -1
        self._check("q", q, nq, n)
        self._check("qd", qd, nv, n)
        self._check("qdd", qdd, nv, n)
        if self._fext is not None:
            self._check("externalWrenches", self._fext, 6 * self._input.getNumberOfJoints(), n)
        if self._fext is not None and self._input.hasWeldedBodies():
            eng, x = self._expanded()
            q2 = self._extended(q, x.n_extra_cfg, x.q_extra)
            qd2, qdd2 = self._extended(qd, x.n_extra_dof), self._extended(qdd, x.n_extra_dof)
            nv2 = nv + x.n_extra_dof
            tau2 = self._empty_like(q2, nv2, n, match_ld=False)
            dq2 = self._empty_like(q2, nv2 * nv2, n, match_ld=False)
            dqd2 = self._empty_like(q2, nv2 * nv2, n, match_ld=False)
            eng.rnea_derivatives(q2, qd2, qdd2, tau2, dq2, dqd2, fext=self._extended(self._fext, 6 * x.n_extra_wrench_blocks))
            # the held joints' DoFs follow the system's own in both the rows and the columns
            self._tau = tau2[:nv]
            self._dq = dq2.reshape(nv2, nv2, n)[:nv, :nv].reshape(nv * nv, n)
            self._dqd = dqd2.reshape(nv2, nv2, n)[:nv, :nv].reshape(nv * nv, n)
            return self._dq
        self._tau = self._empty_like(q, nv, n)
        self._dq = self._empty_like(q, nv * nv, n)
        self._dqd = self._empty_like(q, nv * nv, n)
        self._engine.rnea_derivatives(q, qd, qdd, self._tau, self._dq, self._dqd, fext=self._fext)
        return self._dq

    def getJointTauMatrix(self):
        return self._tau

    def getTauConfigurationGradientMatrix(self):
        return self._dq

    def getTauVelocityGradientMatrix(self):
        return self._dqd


class ForwardDynamicsDerivativesCalculator(_BatchedCalculator):
    """The first-order partials of forward dynamics for N states: qdd(q, qd, tau) of ForwardDynamicsCalculator together with
    d qdd / dq, d qdd / dqd and d qdd / d tau = M^-1 (mecano_b200_aba_derivatives in include/mecano_b200.h: the conventions of
    InverseDynamicsDerivativesCalculator -- column j of d qdd / dq is the derivative along the step the state integrator takes with
    qd = e_j, so a floating base's columns are perturbations in its own frame; qd, tau and the body-fixed external wrenches are
    held).  These are A = [d qdd / dq, d qdd / dqd] and B = M^-1 of xdot = f(x, u), u = tau.  Mecano has no counterpart: the
    definition is this project's.

    getJointAccelerationMatrix() is [nDoFs, N] and bit for bit what ForwardDynamicsCalculator computes; the three matrices are
    [nDoFs * nDoFs, N], entry (i, j) of state s at [i * nDoFs + j, s].  Systems with fixed or ignored joints run on their welded
    tables; external wrenches on such systems are not supported (the locked-joint reduction changes M^-1).  Every joint is an
    EFFORT_SOURCE.  One device only.  kernelInfo() / setGridLimit() concern the inverse-dynamics derivatives kernel, the
    heaviest of the four launches."""
    _ALGO = _capi.ALGO_RNEA_DERIVATIVES

    def __init__(self, input, device=0):
        super().__init__(input, device)
        self._qdd = self._dq = self._dqd = self._minv = None

    def compute(self, q, qd, tau):
        """compute(q, qd, tau) for N states; returns getAccelerationConfigurationGradientMatrix() ([nDoFs * nDoFs, N])."""
        if isinstance(self._device, (list, tuple)):
            raise NotImplementedError("the forward-dynamics derivatives run on one device")
        nv, nq = self._input.getNumberOfDoFs(), self._input.getConfigurationMatrixSize()
        n = q.shape[1] if q.ndim == 2 else -1
        self._check("q", q, nq, n)
        self._check("qd", qd, nv, n)
        self._check("tau", tau, nv, n)
        if self._fext is not None:
            self._check("externalWrenches", self._fext, 6 * self._input.getNumberOfJoints(), n)
            if self._input.hasWeldedBodies():
                raise NotImplementedError("forward-dynamics derivatives with external wrenches on a system with fixed or ignored joints")
        self._qdd = self._empty_like(q, nv, n)
        self._dq = self._empty_like(q, nv * nv, n)
        self._dqd = self._empty_like(q, nv * nv, n)
        self._minv = self._empty_like(q, nv * nv, n)
        self._engine.aba_derivatives(q, qd, tau, self._qdd, self._dq, self._dqd, self._minv, fext=self._fext)
        return self._dq

    def getJointAccelerationMatrix(self):
        return self._qdd

    def getAccelerationConfigurationGradientMatrix(self):
        return self._dq

    def getAccelerationVelocityGradientMatrix(self):
        return self._dqd

    def getInverseMassMatrix(self):
        return self._minv


class MultiBodyDynamicsStep:
    """The three calculators on the same joint states behind one host call (mecano_b200_step_host / mecano_b200_multi_step_host):
    what a Mecano user does per control tick -- insertJointsState once (MultiBodySystemTools.java:1578), updateFramesRecursively()
    once (RigidBodyBasics.java:104-112), then InverseDynamicsCalculator.compute(qdd), ForwardDynamicsCalculator.compute(tau) and
    CompositeRigidBodyMassMatrixCalculator.getMassMatrix().  Host (numpy, ideally pinned) matrices; `device` may be a list of
    GPUs, in which case the batch is sliced across them.  Results are bit-identical to the three calculators called one by one."""

    def __init__(self, input, device=0):
        if isinstance(input, RigidBody):
            input = MultiBodySystem.toMultiBodySystemBasics(input)
        self._input = input
        self._engine = _make_engine(input, device)

    def setGravitationalAcceleration(self, *gravity):
        g = (0.0, 0.0, float(gravity[0])) if len(gravity) == 1 and np.isscalar(gravity[0]) else tuple(float(v) for v in (gravity[0] if len(gravity) == 1 else gravity))
        if len(g) != 3:
            raise ValueError("gravity must have 3 components")
        self._engine.set_gravity(*g)

    def setKernelVariant(self, variant):
        self._engine.set_variant({"auto": 0, "thread": 1, "warp": 2}[variant] if isinstance(variant, str) else int(variant))
        return self

    def getMassMatrixPackedIndex(self):
        return self._engine.packed_index()

    def getMassMatrixRows(self, packed=False):
        return self._engine.packed_size() if packed else self._engine.nv * self._engine.nv

    def compute(self, q, qd, qdd=None, tau=None, tauOut=None, qddOut=None, massMatrix=None, packed=False, stateMajor=False, ownedMassMatrix=False,
                massMatrixZerosPresent=False):
        """qdd -> tauOut (inverse dynamics), tau -> qddOut (forward dynamics), massMatrix (layout as getMassMatrix): each part runs
        if its matrices are given.  ownedMassMatrix=True (dense entry-major layout, no `massMatrix`): the step owns the dense
        matrix like Mecano's calculator does (getMassMatrix() returns a reference to the internal matrix,
        CompositeRigidBodyMassMatrixCalculator.java:344-348) -- one page-locked [nDoFs*nDoFs, N] buffer per batch shape, reused by
        later calls, whose structurally zero entries are written by the first call and from the second on neither recomputed nor
        sent over PCIe again (MECANO_B200_CRBA_ZEROS_PRESENT): the same dense matrix for about half the bytes on a humanoid.
        massMatrixZerosPresent=True is the same for a caller-owned dense entry-major `massMatrix`: the caller's statement that an
        earlier call for this tree filled this very buffer (so its structurally zero entries hold zeros)."""
        layout = _capi.CRBA_PACKED if packed else (_capi.CRBA_STATE_MAJOR if stateMajor else _capi.CRBA_ENTRY_MAJOR)
        if massMatrixZerosPresent:
            if massMatrix is None or packed or stateMajor or ownedMassMatrix:
                raise ValueError("massMatrixZerosPresent: a caller-owned dense entry-major massMatrix filled by an earlier call")
            layout |= _capi.CRBA_ZEROS_PRESENT
        if ownedMassMatrix:
            if massMatrix is not None or packed or stateMajor:
                raise ValueError("ownedMassMatrix: the dense entry-major matrix of the step itself (no massMatrix / packed / stateMajor)")
            nv, n = self._engine.nv, q.shape[1]
            ld = n if q.shape[0] < 2 else max(n, q.strides[0] // 8)
            key = (n, ld)
            if getattr(self, "_owned_key", None) != key:
                self._owned_key, self._owned_M, self._owned_primed = key, CompositeRigidBodyMassMatrixCalculator._new_owned(q, (nv * nv, n), ld), False
            massMatrix = self._owned_M
            if self._owned_primed:
                layout |= _capi.CRBA_ZEROS_PRESENT
        self._engine.step_host(q, qd, qdd_in=qdd, tau_in=tau, tau_out=tauOut, qdd_out=qddOut, M=massMatrix, layout=layout)
        if ownedMassMatrix:
            self._owned_primed = True  # (only once a call has completed: a failed first call has not written the zeros)
        return tauOut, qddOut, massMatrix


class MultiBodySystemStateIntegrator:
    """Batched mirror of M/tools/MultiBodySystemStateIntegrator.java (:26-70 constructor / setIntegrationDT, :365-470
    doubleIntegrateFromAcceleration): q, qd and the SixDoF rows of qdd of N states are updated in place on the GPU.  The
    reference reads and writes the joint objects of one system; here the system is given once and the state matrices
    ([nCfg, N], [nDoFs, N], [nDoFs, N], JointMatrixIndexProvider order) per call."""

    def __init__(self, input, dt=float("nan"), device=0, engine=None):
        if isinstance(input, RigidBody):
            input = MultiBodySystem.toMultiBodySystemBasics(input)
        self._input = input
        self._engine = engine if engine is not None else Engine(input.tables().contents, device, keepalive=input)
        self.setIntegrationDT(dt)

    def setIntegrationDT(self, dt):
        self._dt = float(dt)

    def getIntegrationDT(self):
        return self._dt

    def doubleIntegrateFromAcceleration(self, q, qd, qdd):
        nv, nq = self._input.getNumberOfDoFs(), self._input.getConfigurationMatrixSize()
        n = q.shape[1] if q.ndim == 2 else -1
        for name, m, rows in (("q", q, nq), ("qd", qd, nv), ("qdd", qdd, nv)):
            if m is None or m.ndim != 2 or m.shape[0] != rows or m.shape[1] != n:
                raise MatrixDimensionException("%s: expected a %d x %d matrix, got %s" % (name, rows, n, None if m is None else tuple(m.shape)))
        if self._dt != self._dt:
            raise ValueError("integration dt has not been set")
        if _is_torch(q):
            self._engine.integrate(self._dt, q, qd, qdd)
        else:
            self._engine.integrate_host(self._dt, q, qd, qdd)
        return q, qd
