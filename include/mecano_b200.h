/*
 * mecano_b200.h -- C ABI of the B200-native batched rigid-body dynamics engine.
 *
 * This is the drop-in boundary for Mecano's three recursive calculators evaluated at N joint
 * states in one call.  Mecano (pure Java) has no FFI of its own; the interface replaced is the
 * public API of the calculators ("M/" = /root/reference/src/main/java/us/ihmc/mecano/):
 *
 *   mecano_b200_create            <- new InverseDynamicsCalculator(MultiBodySystemReadOnly)      M/algorithms/InverseDynamicsCalculator.java:201-251
 *                                    new ForwardDynamicsCalculator(MultiBodySystemReadOnly)      M/algorithms/ForwardDynamicsCalculator.java:128-222
 *                                    new CompositeRigidBodyMassMatrixCalculator(...)             M/algorithms/CompositeRigidBodyMassMatrixCalculator.java:182-266
 *                                    (the "flatten the tree once" step; tables in JointMatrixIndexProvider order,
 *                                     M/multiBodySystem/interfaces/JointMatrixIndexProvider.java:71-101)
 *   mecano_b200_set_gravity       <- setGravitationalAcceleration(x, y, z)                       InverseDynamicsCalculator.java:397-403, ForwardDynamicsCalculator.java:313-319
 *   mecano_b200_rnea[_host]       <- InverseDynamicsCalculator.compute(DMatrix) + getJointTauMatrix()            :496-501, :567-570
 *                                    (+ setExternalWrench :469-472, setConsiderCoriolisAndCentrifugalForces /
 *                                     setConsiderJointAccelerations :291-306)
 *   mecano_b200_aba[_host]        <- ForwardDynamicsCalculator.compute(DMatrix) + getJointAccelerationMatrix()   :508-520, :556-567
 *   mecano_b200_crba[_host]       <- CompositeRigidBodyMassMatrixCalculator.reset() + getMassMatrix()            :286-291, :344-348
 *
 * The state (q, qd, qdd, tau), which Mecano keeps inside the joint objects and the frame tree
 * (OneDoFJoint.java:81-87, RigidBodyBasics.java:104-112), is an explicit argument here:
 * "set state -> updateFramesRecursively() -> compute()" is fused into each kernel.
 *
 * Buffers are DoF-major / state-minor:  x[k * ld + s], k = Mecano DoF (or configuration) row,
 * s = state, ld >= n_states.  A Java DMatrixRMaj(nDoFs, N) has exactly this layout.
 * SixDoF rows: configuration [qx qy qz qs x y z]; velocity-like rows [wx wy wz vx vy vz] in the
 * joint's frameAfterJoint (SixDoFJointReadOnly.java:21-26).  All spatial vectors angular-first.
 *
 * There is no CPU fallback: every compute entry point runs hand-written sm_100a kernels or fails.
 * All functions return 0 on success, <0 for an argument / topology error, >0 for a CUDA error
 * (the cudaError_t value); mecano_b200_last_error() gives the text.  Nothing throws across the ABI.
 */
#ifndef MECANO_B200_H
#define MECANO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MECANO_B200_VERSION 200

/* joint types (M/multiBodySystem/{RevoluteJoint,PrismaticJoint,SixDoFJoint,SphericalJoint,PlanarJoint}.java).
 * Rows of a joint in the matrices of the ABI (M/multiBodySystem/interfaces/*JointReadOnly.java):
 *   REVOLUTE / PRISMATIC   configuration [q]                   velocity-like [qd]
 *   SIXDOF                 configuration [qx qy qz qs x y z]   velocity-like [wx wy wz vx vy vz]  (SixDoFJointReadOnly.java:21-26)
 *   SPHERICAL              configuration [qx qy qz qs]         velocity-like [wx wy wz]           (SphericalJointReadOnly.java:31-71)
 *   PLANAR                 configuration [pitch x z]           velocity-like [wy vx vz]           (PlanarJointReadOnly.java:20-58)
 * velocity-like = velocity, acceleration, effort; all expressed in the joint's frameAfterJoint.  (FixedJoint has no rows: the
 * host model welds its successor into the parent body before the tables are built.) */
#define MECANO_B200_REVOLUTE 0
#define MECANO_B200_PRISMATIC 1
#define MECANO_B200_SIXDOF 2
#define MECANO_B200_SPHERICAL 3
#define MECANO_B200_PLANAR 4

/* status codes */
#define MECANO_B200_OK 0
#define MECANO_B200_ERR_INVALID_ARGUMENT (-1)
#define MECANO_B200_ERR_UNSUPPORTED_TOPOLOGY (-2)
#define MECANO_B200_ERR_SHAPE (-3)
#define MECANO_B200_ERR_NO_DEVICE (-4)
#define MECANO_B200_ERR_TOO_LARGE (-5)
#define MECANO_B200_ERR_JIT (-6) /* tree-specialised kernel could not be generated / compiled / loaded */

/* flags for mecano_b200_rnea (mirror InverseDynamicsCalculator.java:291-306) */
#define MECANO_B200_RNEA_NO_CORIOLIS 0x1u      /* setConsiderCoriolisAndCentrifugalForces(false) */
#define MECANO_B200_RNEA_NO_ACCELERATIONS 0x2u /* setConsiderJointAccelerations(false) */

/* mass-matrix layouts for mecano_b200_crba */
#define MECANO_B200_CRBA_ENTRY_MAJOR 0x0u /* M[(i*nv + j) * ld + s]   (default, coalesced) */
#define MECANO_B200_CRBA_STATE_MAJOR 0x1u /* M[s * nv*nv + i*nv + j]  (Mecano's per-state dense DMatrixRMaj) */
/* The entries coupling joints of unrelated branches are zero for every state (they depend on the topology only; half of the
 * matrix for a humanoid).  A Mecano calculator owns its mass matrix and hands out a reference to it
 * (CompositeRigidBodyMassMatrixCalculator.java:344-348); a caller that likewise reuses one buffer for one tree may pass this
 * flag from the second call on: the structurally zero entries are then neither written (device entry point) nor transferred
 * (host entry point, entry-major layout), everything else is recomputed.  The first call into a buffer must not set it. */
#define MECANO_B200_CRBA_ZEROS_PRESENT 0x2u
/* Packed layout: one row per UNIQUE entry that is not structurally zero, M[p * ld + s], p = 0 .. mecano_b200_crba_packed_size() - 1
 * (entry-major like the default, coalesced).  Mecano fills the dense symmetric matrix by writing every computed entry twice
 * (setSymmetricEntry, CompositeRigidBodyMassMatrixCalculator.java:700-707, :772-797) on top of massMatrix.zero() (:296); the packed
 * layout carries each computed entry once and no zeros: 362 rows instead of 1,369 for a 37-DoF humanoid, which is what the
 * host path (PCIe-bound) and a caller that scatters into its own DMatrixRMaj want.  mecano_b200_crba_packed_index() gives the
 * (row, column) of every packed row: M[row[p]][col[p]] = M[col[p]][row[p]] = packed[p]; rows are grouped by column, and
 * within a column ordered along the path from the root body to the column's joint.  Not combinable with STATE_MAJOR /
 * ZEROS_PRESENT; plain mass-matrix calls only (the by-product and fp32 entry points write the dense layout). */
#define MECANO_B200_CRBA_PACKED 0x4u

/* kernel selection */
#define MECANO_B200_VARIANT_AUTO 0
#define MECANO_B200_VARIANT_THREAD 1 /* one thread per state */
#define MECANO_B200_VARIANT_WARP 2   /* one warp-lane group per state (small batches / large trees) */

#define MECANO_B200_ALGO_RNEA 0
#define MECANO_B200_ALGO_ABA 1
#define MECANO_B200_ALGO_CRBA 2
#define MECANO_B200_ALGO_REGRESSOR 4 /* mecano_b200_kernel_info_get of mecano_b200_joint_torque_regressor (3: the Coriolis kernel) */
#define MECANO_B200_ALGO_GRAVITY_GRADIENT 5 /* mecano_b200_kernel_info_get of mecano_b200_gravity_gradient */
#define MECANO_B200_ALGO_RNEA_DERIVATIVES 6 /* mecano_b200_kernel_info_get of mecano_b200_rnea_derivatives */

/* Column order of a body's ten inertial parameters in the joint-torque regressor (mecano_b200_joint_torque_regressor): the
 * column of the mass, the first of the three first moments m c (x, y, z) and the first of the six moments of inertia about the
 * origin (xx, xy, xz, yy, yz, zz).  This order is this project's definition; the kernel, the bindings and the tests read it
 * from here. */
#define MECANO_B200_REGRESSOR_M 0
#define MECANO_B200_REGRESSOR_MC 1
#define MECANO_B200_REGRESSOR_I 4

typedef struct mecano_b200_handle mecano_b200_handle;

/*
 * Flattened, level-ordered description of one kinematic tree: what the Java host builds once from a
 * MultiBodySystemReadOnly.  Body b (0 <= b < n_bodies) is the successor of joint b; the root body
 * (elevator) is not listed and is referred to as parent -1.  Bodies must be listed so that
 * parent[b] < b (level order satisfies this).  level_start is optional (may be NULL).
 */
typedef struct mecano_b200_tree_desc
{
   int32_t struct_size; /* sizeof(mecano_b200_tree_desc), for ABI evolution */
   int32_t n_bodies;
   int32_t n_dofs;   /* MultiBodySystemTools.computeDegreesOfFreedom */
   int32_t n_cfg;    /* configuration rows: 1 per OneDoF joint, 7 per SixDoF, 4 per Spherical, 3 per Planar joint */
   int32_t n_levels; /* 0 if level_start == NULL */
   const int32_t *level_start; /* [n_levels + 1] first body of each tree level */
   const int32_t *parent;      /* [n_bodies] */
   const int32_t *joint_type;  /* [n_bodies] MECANO_B200_REVOLUTE / PRISMATIC / SIXDOF / SPHERICAL / PLANAR */
   const double *axis;         /* [n_bodies][3] unit joint axis in frameAfterJoint (one-DoF joints only) */
   const double *offset_rot;   /* [n_bodies][9] row-major rotation: frameBeforeJoint in the parent's frameAfterJoint */
   const double *offset_pos;   /* [n_bodies][3] */
   const double *com_rot;      /* [n_bodies][9] inertia pose: bodyFixedFrame (CoM frame) in frameAfterJoint */
   const double *com_pos;      /* [n_bodies][3] */
   const double *inertia;      /* [n_bodies][9] symmetric moment of inertia about the CoM, in bodyFixedFrame */
   const double *mass;         /* [n_bodies] */
   const int32_t *dof_offset;  /* [n_bodies] JointMatrixIndexProvider row of the joint's first DoF */
   const int32_t *cfg_offset;  /* [n_bodies] row of the joint's first configuration entry */
   const int32_t *wrench_index; /* [n_bodies] or NULL: body b's external wrench occupies rows [6 w, 6 w + 6) of fext, w = wrench_index[b]
                                   (NULL: w = b).  The Java host passes the joint's JointMatrixIndexProvider rank here so that fext
                                   is in Mecano joint order like every other matrix. */
} mecano_b200_tree_desc;

typedef struct mecano_b200_kernel_info
{
   int32_t variant;            /* MECANO_B200_VARIANT_THREAD / WARP actually selected for this batch size */
   int32_t block_threads;
   int32_t states_per_block;
   int32_t regs_per_thread;
   int32_t static_smem_bytes;
   int32_t dynamic_smem_bytes;
   int32_t local_bytes_per_thread;
   int32_t blocks_per_sm;      /* occupancy reported by the runtime */
   int32_t sm_count;
   int32_t stack_doubles;      /* per-state stack slots held in shared memory */
   int32_t max_depth;
   int32_t specialized;        /* 0: generic kernel (traversal program interpreted); 1: tree-specialised kernel compiled by
                                  mecano_b200_specialize(); 2: the same, loaded from the cubin cache */
   double bytes_per_state;     /* algorithmic HBM bytes per state (SURVEY.md 8d) */
   int32_t tmem_stack_slots;   /* per-state stack slots (16 bytes each) held in tensor memory instead of shared memory */
   int32_t reserved;
   double jit_seconds;         /* time mecano_b200_specialize() spent on this kernel (generate + NVRTC + load) */
} mecano_b200_kernel_info;

int mecano_b200_version(void);
int mecano_b200_device_count(void);

/* Build the constant tables / traversal programs for one tree on one device. */
int mecano_b200_create(const mecano_b200_tree_desc *desc, int device, mecano_b200_handle **out);
void mecano_b200_destroy(mecano_b200_handle *h);
const char *mecano_b200_last_error(const mecano_b200_handle *h); /* h may be NULL: error of the last failed create */

int mecano_b200_set_gravity(mecano_b200_handle *h, double gx, double gy, double gz);
int mecano_b200_set_variant(mecano_b200_handle *h, int variant);
/*
 * Optional fp32 variant.  MECANO_B200_PRECISION_FP32 makes the plain mecano_b200_rnea / aba / crba calls (device and host entry
 * points) compute in single precision; every buffer of the ABI stays fp64.  Mecano is double precision throughout: this is a
 * throughput option with its own, much looser tolerance (RNEA / CRBA 1e-5 relative, ABA 1e-4 on a 37-DoF humanoid; measured worst state of 2^20: 3e-6), reported
 * separately and never chosen implicitly.  Calls the variant does not cover (external wrenches, flags, by-products, trees
 * outside the humanoid-sized launch configuration) fail with MECANO_B200_ERR_UNSUPPORTED_TOPOLOGY instead of running in fp64.
 */
#define MECANO_B200_PRECISION_FP64 0
#define MECANO_B200_PRECISION_FP32 1
int mecano_b200_set_precision(mecano_b200_handle *h, int precision);
/*
 * Sharing the device between calculators that run at the same time on different streams (Mecano users run one calculator per
 * thread, MultiBodySystemFactories.java:310-348; here: one per stream).  The thread-per-state RNEA and ABA kernels are persistent
 * grids that by default fill every SM, and each of their blocks owns its SM (registers, tensor memory); max_blocks caps the
 * grid of `algo` (MECANO_B200_ALGO_*) so that a concurrent kernel -- typically the bandwidth-bound mass matrix next to the
 * FP64-bound forward dynamics -- finds free SMs.  0 = no cap.  Results do not depend on it.  (The warps of a persistent grid draw
 * their states, 32 at a time, from a counter owned by the handle -- a fresh one per launch out of a ring of 256 -- instead of taking
 * tiles in a fixed order; which warp evaluates a state has no influence on its result.)
 */
int mecano_b200_set_grid_limit(mecano_b200_handle *h, int algo, int max_blocks);

/*
 * Compile kernels specialised for this tree (bit mask of 1 << MECANO_B200_ALGO_*).  A Mecano calculator mirrors the body
 * tree into recursion-step objects in its constructor (InverseDynamicsCalculator.java:253-282); this is the same step taken
 * further: the traversal is unrolled into straight-line CUDA C++ with the tree's constants as literals and compiled with
 * NVRTC for sm_100a (seconds; cubins are cached under $MECANO_B200_CACHE, default ~/.cache/mecano_b200).  Optional: without
 * it every call runs the generic kernels, which interpret the same traversal program.  Calls with external wrenches or
 * non-default flags always use the generic kernels.  Unrolled code only pays while it fits the instruction caches: algorithms
 * whose estimated code size is too large (RNEA beyond ~20 bodies, ABA beyond ~9) are skipped and keep the generic kernel
 * (mecano_b200_kernel_info.specialized tells which one runs); CRBA is never specialised (HBM-bound).  Results of the two paths
 * agree to round-off (same routines, different instruction scheduling).
 */
#define MECANO_B200_SPECIALIZE_FORCE 0x100u /* also unroll trees whose code exceeds the instruction caches (slower; for measurements) */
int mecano_b200_specialize(mecano_b200_handle *h, uint32_t algo_mask);
int mecano_b200_n_dofs(const mecano_b200_handle *h);
int mecano_b200_n_cfg(const mecano_b200_handle *h);
int mecano_b200_n_bodies(const mecano_b200_handle *h);
/* Packed mass-matrix layout (MECANO_B200_CRBA_PACKED): number of packed rows, and the dense (row, col) of each (arrays of
 * mecano_b200_crba_packed_size() entries, either may be NULL). */
int mecano_b200_crba_packed_size(const mecano_b200_handle *h);
int mecano_b200_crba_packed_index(const mecano_b200_handle *h, int32_t *row, int32_t *col);

/*
 * Device-pointer entry points.  All pointers are device memory on the handle's device, 8-byte
 * aligned; `stream` is a cudaStream_t (NULL = default stream).  Calls are asynchronous.
 * fext (nullable): external wrench on each body expressed in that body's CoM frame,
 * [(6 * w + c) * ld + s], w = wrench_index[b] (default: b, the order of the tree description)
 * (InverseDynamicsCalculator.java:819, :946).
 */
int mecano_b200_rnea(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *qdd,
                     const double *fext, double *tau, uint32_t flags, void *stream);
int mecano_b200_aba(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *tau,
                    const double *fext, double *qdd, uint32_t flags, void *stream);
/*
 * Joint source modes of forward dynamics (ForwardDynamicsCalculator.JointSourceMode, ForwardDynamicsCalculator.java:45-57;
 * setJointSourceMode :400-403, resetJointSourceModes :438-444).  accel_source [n_bodies], in the order of the tree description:
 * non-zero = the joint of that body is an ACCELERATION_SOURCE (its acceleration is an input, its effort an output), zero =
 * EFFORT_SOURCE (the default).  NULL resets every joint to EFFORT_SOURCE.  A property of the handle like gravity: set it between
 * calls, not concurrently with them.
 *
 * mecano_b200_aba_sources = compute(jointTauInput, jointAccelerationInput) (:508-520) for N states:
 *   tau     [n_dofs][ld]  efforts; the rows of ACCELERATION_SOURCE joints are not read
 *   qdd_in  [n_dofs][ld]  accelerations; only the rows of ACCELERATION_SOURCE joints are read (may be NULL if there are none)
 *   qdd     [n_dofs][ld]  getJointAccelerationMatrix() (:556-564): computed for EFFORT_SOURCE joints, qdd_in repeated for the others
 *   tau_out [n_dofs][ld]  (nullable) getJointTauMatrix() (:566-590): tau repeated for EFFORT_SOURCE joints, computed for the others
 *                         (pass four, :1315-1363; costs one additional inverse-dynamics launch).  Must not alias tau.
 * With joints in ACCELERATION_SOURCE mode plain mecano_b200_aba is refused (it has no acceleration input).
 */
int mecano_b200_set_joint_source_modes(mecano_b200_handle *h, const int32_t *accel_source);
int mecano_b200_aba_sources(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *tau,
                            const double *qdd_in, const double *fext, double *qdd, double *tau_out, void *stream);
/*
 * RNEA with its by-products, the two per-body results InverseDynamicsCalculator keeps beside the joint efforts:
 *   body_acc     (nullable) getBodyAcceleration(body), InverseDynamicsCalculator.java:578-591: the spatial acceleration of each
 *                body (gravity included as the root's acceleration, :397-403) expressed in its CoM frame, angular part first;
 *   joint_wrench (nullable) getComputedJointWrench(joint), :593-602: the wrench its joint transmits to each body, expressed in
 *                the joint's frameAfterJoint, moment first.
 * Both are [(6 * w + c) * ld + s] with w = wrench_index[b], the row convention of fext.  Bodies welded into an ancestor (fixed
 * or ignored joints) have no rows written.  Always runs the generic thread-per-state kernel.
 */
int mecano_b200_rnea_full(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *qdd,
                          const double *fext, double *tau, double *body_acc, double *joint_wrench, uint32_t flags, void *stream);
int mecano_b200_crba(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, double *mass_matrix, uint32_t layout,
                     void *stream);

/*
 * Centroidal by-products of the mass-matrix calculator (CompositeRigidBodyMassMatrixCalculator.java:380-440, :801-839).
 * `frame` is the centroidal momentum frame (setCentroidalMomentumFrame, :380-387):
 *   MECANO_B200_FRAME_WORLD           the inertial frame of the system (the root body's frame);
 *   MECANO_B200_FRAME_CENTER_OF_MASS  axes of the inertial frame, origin at the centre of mass of the system in each state (what a
 *                                     CenterOfMassReferenceFrame handed to the Java calculator is).
 * mecano_b200_crba_centroidal = getMassMatrix() + getCentroidalMomentumMatrix() (:801-809) for N states:
 *   mass_matrix [n_dofs * n_dofs][ld]  entry-major, every entry written
 *   cmm         [6 * n_dofs][ld]       entry (r, j) of the 6 x n_dofs matrix at row r * n_dofs + j (the layout of Mecano's row-major
 *                                      DMatrixRMaj, state-minor); angular momentum rows first.  cmm * qd = momentum in `frame`
 *   com         [4][ld]                centre of mass in the root frame (x, y, z) and total mass
 * mecano_b200_centroidal_convective_term = getCentroidalConvectiveTerm() (:811-839), d/dt(cmm) qd:
 *   out         [6][ld]                moment first; `com` = the rows written by mecano_b200_crba_centroidal or
 *                                      mecano_b200_center_of_mass for the same q (needed for MECANO_B200_FRAME_CENTER_OF_MASS only,
 *                                      else may be NULL)
 * mecano_b200_center_of_mass = CenterOfMassCalculator.getCenterOfMass() + getTotalMass() (CenterOfMassCalculator.java:70-124), the
 * origin a CenterOfMassReferenceFrame moves to on update (CenterOfMassReferenceFrame.java:45-50), for N states: the `com` rows
 * alone, bit-identical to those of mecano_b200_crba_centroidal, without computing or writing a matrix
 */
#define MECANO_B200_FRAME_WORLD 0
#define MECANO_B200_FRAME_CENTER_OF_MASS 1
int mecano_b200_crba_centroidal(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, double *mass_matrix, double *cmm, double *com,
                                int frame, void *stream);
int mecano_b200_centroidal_convective_term(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *com,
                                           double *out, int frame, void *stream);
int mecano_b200_center_of_mass(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, double *com, void *stream);

/*
 * Mass matrix and Coriolis / centrifugal matrix together: getMassMatrix() + getCoriolisMatrix() after
 * setEnableCoriolisMatrixCalculation(true) (CompositeRigidBodyMassMatrixCalculator.java:278-281, :358-366, recursion :588-799,
 * FactorizedBodyInertia.java).  Both [n_dofs * n_dofs][ld], entry-major, every entry written; coriolis_matrix * qd = the joint
 * efforts of inverse dynamics with zero joint accelerations and no gravity.
 */
int mecano_b200_coriolis(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd, double *mass_matrix,
                         double *coriolis_matrix, void *stream);

/*
 * Joint-torque regressor (Mecano's JointTorqueRegressorCalculator): the matrix Y(q, qd, qdd) with tau = Y pi for ANY inertial
 * parameters pi of the bodies -- what system identification stacks over a log of states to fit masses, centres of mass and
 * inertias.  For a tree of n_bodies bodies (the root body, which is fixed, has no columns) and n_dofs DoFs:
 *   Y            [n_dofs * 10 n_bodies][ld]  entry (i, c) of state s at [(i * 10 n_bodies + c) * ld + s], every entry written
 *                                            (including the structural zeros: rows of joints off the path from the root to the
 *                                            column's body).  Row i = Mecano DoF row.  Column block w (ten columns) belongs to
 *                                            the body whose external-wrench rows are [6 w, 6 w + 6), w = wrench_index[b], the
 *                                            convention of fext / body_acc / joint_wrench.
 * The parameters of body w, in the column order of the MECANO_B200_REGRESSOR_* table: m, m cx, m cy, m cz, Ixx, Ixy, Ixz, Iyy,
 * Iyz, Izz, with c the centre of mass and I the moment of inertia about the origin, both expressed in the body's bodyFixedFrame
 * (the CoM frame of the tree description: com_rot, com_pos), the frame in which Mecano holds a body's SpatialInertia.  The
 * model's own parameters are therefore pi_w = [m, 0, 0, 0, J_xx, J_xy, J_xz, J_yy, J_yz, J_zz].  tau = Y pi is inverse dynamics
 * with the handle's gravity and without external wrenches.
 * Always runs the generic thread-per-state kernel, in fp64 (a handle set to fp32 refuses with MECANO_B200_ERR_UNSUPPORTED_TOPOLOGY);
 * the wrench_index ranks must be below n_bodies (MECANO_B200_ERR_SHAPE otherwise).  Y is large: 10 n_bodies n_dofs doubles per
 * state (94,720 bytes for a 32-body, 37-DoF humanoid).
 */
int mecano_b200_joint_torque_regressor(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *qdd,
                                       double *Y, void *stream);

/*
 * Gravity gradient (Mecano's MultiBodyGravityGradientCalculator): the joint efforts that gravity and the external wrenches cause,
 * tau_g(q), and their configuration gradient G(q) = d tau_g / dq -- what gravity compensation with joint stiffness, the stability
 * margin of a posture and the linearisation of the dynamics need.  For N states, with the handle's gravity:
 *   tau       [n_dofs][ld]            the joint efforts of mecano_b200_rnea at the same q and fext with qd = 0 and qdd = 0
 *   gradient  [n_dofs * n_dofs][ld]   entry (i, j) of G at [(i * n_dofs + j) * ld + s], entry-major like the mass matrix, every
 *                                     entry written; the entries that couple joints of unrelated branches (the structural zeros of
 *                                     the mass matrix) are 0.0.
 * Entry (i, j) is d/d eps tau_i(q (+) eps e_j) at eps = 0, where q (+) eps e_j is what mecano_b200_integrate does to q with dt = eps,
 * qd = e_j and qdd = 0: q + eps for a one-DoF joint; for SixDoF, spherical and planar joints a step along the body-frame velocity
 * coordinate j, in frameAfterJoint.  The columns of a floating base are therefore perturbations in its own frame, the convention
 * under which G is n_dofs x n_dofs.
 * fext (nullable): the convention of mecano_b200_rnea (rows [6 w, 6 w + 6), w = wrench_index[b], in the body's CoM frame): the
 * external wrenches are body-fixed and turn with their body.  With fext the wrench_index ranks must be below n_bodies
 * (MECANO_B200_ERR_SHAPE otherwise).
 * G is not symmetric in general; it is symmetric to round-off on trees of one-DoF joints without fext, where it is the Hessian of
 * the potential energy.  The floating-base and external-wrench conventions of Mecano's own calculator are unpinned (its source is
 * not at hand): the ones above are this project's definition.
 * Always runs the generic thread-per-state kernel, in fp64 (a handle set to fp32 refuses with MECANO_B200_ERR_UNSUPPORTED_TOPOLOGY).
 */
int mecano_b200_gravity_gradient(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *fext, double *tau,
                                 double *gradient, void *stream);

/*
 * Inverse-dynamics derivatives: the joint efforts tau(q, qd, qdd) of RNEA and their first-order partials d tau / dq and d tau / dqd
 * at a general state -- what MPC, iLQR / DDP and trajectory optimisation linearise along a trajectory.  The third partial,
 * d tau / dqdd, is the mass matrix (mecano_b200_crba); the forward-dynamics partials follow as dqdd / dx = -M^-1 d tau / dx.
 * For N states, with the handle's gravity:
 *   tau       [n_dofs][ld]            the joint efforts of mecano_b200_rnea on the same q, qd, qdd and fext, with no flags
 *   dtau_dq   [n_dofs * n_dofs][ld]   entry (i, j) at [(i * n_dofs + j) * ld + s], entry-major like the mass matrix
 *   dtau_dqd  [n_dofs * n_dofs][ld]   the same layout
 * Every entry of both matrices is written; the entries that couple joints of unrelated branches (the structural zeros of the mass
 * matrix) are 0.0.  Column j of dtau_dq follows the convention of mecano_b200_gravity_gradient: the derivative along the step
 * mecano_b200_integrate takes with dt = eps, qd = e_j and qdd = 0, so a floating base's columns are perturbations in its own frame;
 * qd and qdd are held.  Column j of dtau_dqd is d tau / d qd_j with q and qdd held.
 * fext (nullable): the convention of mecano_b200_rnea (rows [6 w, 6 w + 6), w = wrench_index[b], in the body's CoM frame): the
 * external wrenches are body-fixed and turn with their body.  With fext the wrench_index ranks must be below n_bodies
 * (MECANO_B200_ERR_SHAPE otherwise).
 * At qd = qdd = 0, dtau_dq is the gradient of mecano_b200_gravity_gradient (to round-off) and dtau_dqd is zero.  Mecano has no
 * counterpart of this call: the definition above is this project's.
 * Always runs the generic thread-per-state kernel, in fp64 (a handle set to fp32 refuses with MECANO_B200_ERR_UNSUPPORTED_TOPOLOGY).
 */
int mecano_b200_rnea_derivatives(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *qdd,
                                 const double *fext, double *tau, double *dtau_dq, double *dtau_dqd, void *stream);

/*
 * Forward-dynamics derivatives: the joint accelerations qdd(q, qd, tau) of ABA, their first-order partials d qdd / dq and d qdd / dqd,
 * and d qdd / d tau = M^-1 -- the A = [d qdd / dq, d qdd / dqd] and B = M^-1 of the dynamics xdot = f(x, u), u = tau, that iLQR / DDP,
 * MPC and batched-simulation gradients consume.  For N states, with the handle's gravity:
 *   qdd       [n_dofs][ld]            what mecano_b200_aba computes on the same q, qd, tau and fext, bit for bit
 *   dqdd_dq   [n_dofs * n_dofs][ld]   entry (i, j) at [(i * n_dofs + j) * ld + s], entry-major like the mass matrix
 *   dqdd_dqd  [n_dofs * n_dofs][ld]   the same layout
 *   minv      [n_dofs * n_dofs][ld]   the same layout
 * Every entry of the three matrices is written.  Unlike M, M^-1 has no structural zeros in general: only the entries between
 * branches that hang separately off the fixed root are zero (0.0), in minv and in both partials.  The conventions are those of
 * mecano_b200_rnea_derivatives: column j of dqdd_dq is the derivative along the step mecano_b200_integrate takes with qd = e_j, so a
 * floating base's columns are perturbations in its own frame; qd, tau and fext are held, and fext (nullable, the convention of
 * mecano_b200_rnea) is body-fixed.  Since ID(q, qd, FD(q, qd, tau)) = tau,
 *   dqdd_dq = -M^-1 dtau_dq(q, qd, qdd),   dqdd_dqd = -M^-1 dtau_dqd(q, qd, qdd),   minv = M^-1,
 * and this is how they are computed: mecano_b200_aba, mecano_b200_rnea_derivatives at its qdd, mecano_b200_crba, then one kernel that
 * factors M = L^T D L along the kinematic tree (no fill-in) and solves in place -- four launches on `stream`, no workspace.
 * Refusals: a handle set to fp32 (MECANO_B200_ERR_UNSUPPORTED_TOPOLOGY), a joint in ACCELERATION_SOURCE mode
 * (MECANO_B200_ERR_INVALID_ARGUMENT), with fext a wrench_index rank >= n_bodies (MECANO_B200_ERR_SHAPE), and a tree the
 * inverse-dynamics derivatives kernel does not fit (MECANO_B200_ERR_TOO_LARGE).  Mecano has no counterpart of this call.
 */
int mecano_b200_aba_derivatives(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *tau,
                                const double *fext, double *qdd, double *dqdd_dq, double *dqdd_dqd, double *minv, void *stream);

/*
 * Host-pointer entry points (what a JNI / Panama binding calls with DMatrixRMaj.data): inputs are
 * staged host -> device in chunks, the kernels run, results are copied back; the call returns when
 * the outputs are complete.  Pinned (page-locked) host memory makes the copies asynchronous and
 * overlapped; pageable memory works too.
 */
int mecano_b200_rnea_host(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *qdd,
                          const double *fext, double *tau, uint32_t flags);
int mecano_b200_rnea_full_host(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *qdd,
                               const double *fext, double *tau, double *body_acc, double *joint_wrench, uint32_t flags);
int mecano_b200_aba_host(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *tau,
                         const double *fext, double *qdd, uint32_t flags);
int mecano_b200_aba_sources_host(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *tau,
                                 const double *qdd_in, const double *fext, double *qdd, double *tau_out);
int mecano_b200_crba_host(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, double *mass_matrix, uint32_t layout);
/*
 * One host call for the three calculators on the same joint states -- what a controller or simulator does per tick with Mecano:
 * set the joint state once (MultiBodySystemTools.insertJointsState, M/tools/MultiBodySystemTools.java:1578), updateFramesRecursively()
 * once (RigidBodyBasics.java:104-112), then InverseDynamicsCalculator.compute(qdd) (:496), ForwardDynamicsCalculator.compute(tau)
 * (:508) and CompositeRigidBodyMassMatrixCalculator.getMassMatrix() (:344).  q and qd cross PCIe once per chunk instead of once
 * per calculator, and the three kernels run back to back on the resident chunk.
 *   qdd_in  [n_dofs][ld]  joint accelerations for inverse dynamics     -> tau_out    [n_dofs][ld]  (both NULL: skip RNEA)
 *   tau_in  [n_dofs][ld]  joint efforts for forward dynamics           -> qdd_out    [n_dofs][ld]  (both NULL: skip ABA)
 *   mass_matrix           layout as mecano_b200_crba_host (ENTRY_MAJOR [| ZEROS_PRESENT], STATE_MAJOR or PACKED)   (NULL: skip CRBA)
 * fext (nullable) applies to both dynamics calculators.  Results are bit-identical to the three separate calls.
 */
int mecano_b200_step_host(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *qdd_in,
                          const double *tau_in, const double *fext, double *tau_out, double *qdd_out, double *mass_matrix, uint32_t layout);

/*
 * Several GPUs of one box behind one call (SURVEY.md 8e).  States are independent, so a batch is cut into disjoint contiguous
 * slices of the state index, one per device; there is no exchange step and no collective (NCCL is not linked).  A multi-device
 * engine owns one handle (constant tables, traversal programs, staging buffers, two streams) per listed device; its host entry
 * points slice the state-minor matrices in place (a slice of a DoF-major matrix is the same matrix with an offset pointer and
 * the same ld: cudaMemcpy2DAsync does the strided copy), issue the chunks of all devices round-robin from the calling thread
 * and synchronise once at the end.  A device may be listed more than once (each entry gets its own handle and pipeline).
 * Results are bit-identical to the single-device call whatever the device list: every state is evaluated by the same
 * instruction sequence, and the thread- / warp-per-state choice of VARIANT_AUTO is made on the size of the whole batch.
 *   mecano_b200_multi_handle(m, i)   the handle of entry i, for the per-handle setters (variant, precision, source modes, ...);
 *                                    compute calls on it bypass the slicing
 *   mecano_b200_multi_slice          the slice [start, start + count) of an n_states batch that entry i evaluates
 */
typedef struct mecano_b200_multi mecano_b200_multi;
int mecano_b200_multi_create(const mecano_b200_tree_desc *desc, const int32_t *devices, int n_devices, mecano_b200_multi **out);
void mecano_b200_multi_destroy(mecano_b200_multi *m);
const char *mecano_b200_multi_last_error(const mecano_b200_multi *m);
int mecano_b200_multi_size(const mecano_b200_multi *m);
mecano_b200_handle *mecano_b200_multi_handle(mecano_b200_multi *m, int i);
int mecano_b200_multi_slice(const mecano_b200_multi *m, int64_t n_states, int i, int64_t *start, int64_t *count);
int mecano_b200_multi_set_gravity(mecano_b200_multi *m, double gx, double gy, double gz);
int mecano_b200_multi_rnea_host(mecano_b200_multi *m, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *qdd,
                                const double *fext, double *tau, uint32_t flags);
int mecano_b200_multi_aba_host(mecano_b200_multi *m, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *tau,
                               const double *fext, double *qdd, uint32_t flags);
int mecano_b200_multi_crba_host(mecano_b200_multi *m, int64_t n_states, int64_t ld, const double *q, double *mass_matrix, uint32_t layout);
int mecano_b200_multi_step_host(mecano_b200_multi *m, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *qdd_in,
                                const double *tau_in, const double *fext, double *tau_out, double *qdd_out, double *mass_matrix, uint32_t layout);
int mecano_b200_coriolis_host(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd, double *mass_matrix,
                              double *coriolis_matrix);
int mecano_b200_joint_torque_regressor_host(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd,
                                            const double *qdd, double *Y);
int mecano_b200_gravity_gradient_host(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *fext, double *tau,
                                      double *gradient);
int mecano_b200_rnea_derivatives_host(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *qdd,
                                      const double *fext, double *tau, double *dtau_dq, double *dtau_dqd);
int mecano_b200_aba_derivatives_host(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd, const double *tau,
                                     const double *fext, double *qdd, double *dqdd_dq, double *dqdd_dqd, double *minv);
int mecano_b200_crba_centroidal_host(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, double *mass_matrix, double *cmm,
                                     double *com, int frame);
int mecano_b200_centroidal_convective_term_host(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, const double *qd,
                                                const double *com, double *out, int frame);
int mecano_b200_center_of_mass_host(mecano_b200_handle *h, int64_t n_states, int64_t ld, const double *q, double *com);

/*
 * State integrator: MultiBodySystemStateIntegrator(dt).doubleIntegrateFromAcceleration(joints)
 * (M/tools/MultiBodySystemStateIntegrator.java:365-470; one-DoF joints :710-733, floating joints :503-560), the step that
 * follows ForwardDynamicsCalculator.compute() + writeComputedJointAccelerations() in a simulation loop, for N states:
 *   one-DoF:  q += dt qd + dt^2/2 qdd,  qd += dt qdd
 *   SixDoF:   SE(3) update of the pose from the body-frame twist / spatial acceleration; the twist and the linear rows of
 *             the acceleration are re-expressed in the new body frame exactly as the Java code leaves them in the joint
 * q [n_cfg][ld], qd [n_dofs][ld] and qdd [n_dofs][ld] are updated IN PLACE (qdd: SixDoF linear rows only).  Device / host
 * pointer variants like the calculators.  Keeping q, qd on the device between mecano_b200_aba and mecano_b200_integrate
 * gives batched simulation roll-outs with no host round trip.
 */
int mecano_b200_integrate(mecano_b200_handle *h, int64_t n_states, int64_t ld, double dt, double *q, double *qd, double *qdd, void *stream);
int mecano_b200_integrate_host(mecano_b200_handle *h, int64_t n_states, int64_t ld, double dt, double *q, double *qd, double *qdd);

/* Introspection for the benchmark / roofline report. */
int mecano_b200_kernel_info_get(mecano_b200_handle *h, int algo, int64_t n_states, mecano_b200_kernel_info *info);

/* Roofline denominators measured on the handle-less device: FP64 FMA chain (best of five short launches: the burst figure; back to
 * back for `seconds`, rate over the second half: the sustained figure under the board's power management) and a read+write copy. */
int mecano_b200_measure_fp64_peak(int device, double *tflops);
int mecano_b200_measure_fp64_sustained(int device, double seconds, double *tflops);
int mecano_b200_measure_hbm_peak(int device, double *gbytes_per_s);

/*
 * The CUDA C++ text of the tree-specialised kernel that mecano_b200_create() compiles for this tree (debugging,
 * build-time checks; works without a GPU).  tmem_slots = stack slots held in tensor memory (0 = shared memory only).
 * Writes at most `capacity` bytes (NUL-terminated) and reports the full size in *needed.
 */
int mecano_b200_generate_source(const mecano_b200_tree_desc *desc, int algo, int block_threads, int tmem_slots, char *buf, int64_t capacity,
                                int64_t *needed);

/* Generates the specialised source for (desc, algo) and compiles it with NVRTC to an sm_100a cubin without loading it:
 * the "does the run-time compiled path build" check; needs no GPU. */
int mecano_b200_jit_check(const mecano_b200_tree_desc *desc, int algo, int block_threads, int tmem_slots, int64_t *cubin_bytes);

/* Pinned host memory helpers for bindings that cannot allocate it themselves. */
int mecano_b200_host_alloc(void **ptr, int64_t bytes);
int mecano_b200_host_free(void *ptr);

#ifdef __cplusplus
}
#endif
#endif
