// calculators.hpp -- C++ mirror of Mecano's three calculators over the C ABI, batched over N states.
//
//   InverseDynamicsCalculator                 M/algorithms/InverseDynamicsCalculator.java:201-251, 291-306, 343-403, 469-472, 496-501, 567-570
//   ForwardDynamicsCalculator                 M/algorithms/ForwardDynamicsCalculator.java:128-196, 313-319, 508-520, 556-567
//   CompositeRigidBodyMassMatrixCalculator    M/algorithms/CompositeRigidBodyMassMatrixCalculator.java:182-233, 286-291, 344-348
//   JointTorqueRegressorCalculator            the inertial-parameter regressor of inverse dynamics (project definition, below)
//   MultiBodyGravityGradientCalculator        gravity torques and their configuration gradient (project definition, below)
//   InverseDynamicsDerivativesCalculator      d tau / dq and d tau / dqd of inverse dynamics (project definition, below)
//   ForwardDynamicsDerivativesCalculator      d qdd / dq, d qdd / dqd and M^-1 of forward dynamics (project definition, below)
//
// Same names, argument meaning and error behaviour (exceptions) as the reference, with two batching changes:
//   * compute(...) takes the joint state explicitly as nRows x N row-major matrices (what a Java
//     DMatrixRMaj(nDoFs, N) is) instead of reading it from the joint objects;
//   * results are written to caller-provided matrices (the reference returns internal references).
// All compute paths end in the CUDA kernels; there is no CPU implementation behind these classes.
#pragma once
#include <stdexcept>
#include <string>

#include "multibody.hpp"

namespace mecano
{
class MatrixDimensionException : public std::runtime_error // EJML's, thrown on shape errors (ForwardDynamicsCalculator.java:522-533)
{
 public:
   using std::runtime_error::runtime_error;
};

// Non-owning view of a rows x N row-major matrix (host or device memory).
struct MatrixView
{
   double *data = nullptr;
   int64_t rows = 0, cols = 0, ld = 0;
   MatrixView() = default;
   MatrixView(double *d, int64_t r, int64_t c) : data(d), rows(r), cols(c), ld(c) {}
   MatrixView(double *d, int64_t r, int64_t c, int64_t l) : data(d), rows(r), cols(c), ld(l) {}
};

enum class Memory { Host, Device };

class BatchedCalculatorBase
{
 public:
   BatchedCalculatorBase(const MultiBodySystem &input, int device) : input_(input), tables_(FlatTables::flatten(input))
   {
      tables_.bind(input.getNumberOfDoFs(), input.getConfigurationMatrixSize());
      const int rc = mecano_b200_create(&tables_.desc, device, &handle_);
      if (rc != MECANO_B200_OK)
         throw ScrewTheoryException(std::string("mecano_b200_create failed: ") + mecano_b200_last_error(nullptr));
   }
   virtual ~BatchedCalculatorBase() { mecano_b200_destroy(handle_); }
   BatchedCalculatorBase(const BatchedCalculatorBase &) = delete;
   BatchedCalculatorBase &operator=(const BatchedCalculatorBase &) = delete;

   const MultiBodySystem &getInput() const { return input_; }
   // setGravitationalAcceleration(double gravity): along z, usually -9.81
   void setGravitationalAcceleration(double gravity) { setGravitationalAcceleration(0.0, 0.0, gravity); }
   void setGravitationalAcceleration(double gx, double gy, double gz) { mecano_b200_set_gravity(handle_, gx, gy, gz); }
   void setGravitationalAcceleration(const Vector3D &g) { setGravitationalAcceleration(g.x, g.y, g.z); }
   // External wrenches for the next compute(): a (6 * nBodies) x N matrix, wrench of joint j's successor (j in
   // JointMatrixIndexProvider order) at rows [6 j, 6 j + 6), expressed in that body's CoM frame
   // (InverseDynamicsCalculator.java:469-472, :819).  Pass an empty view for setExternalWrenchesToZero().
   void setExternalWrenches(const MatrixView &fextInJointOrder) { fext_ = fextInJointOrder; }
   void setExternalWrenchesToZero() { fext_ = MatrixView(); }
   void setStream(void *cudaStream) { stream_ = cudaStream; }
   mecano_b200_handle *handle() const { return handle_; }
   const FlatTables &tables() const { return tables_; }

 protected:
   void check(int rc) const
   {
      if (rc != MECANO_B200_OK)
         throw std::runtime_error(std::string("mecano_b200: ") + mecano_b200_last_error(handle_));
   }
   void checkShape(const MatrixView &m, int64_t rows, int64_t cols, const char *what) const
   {
      if (!m.data || m.rows != rows || m.cols != cols || m.ld < cols)
         throw MatrixDimensionException(std::string(what) + ": expected " + std::to_string(rows) + " x " + std::to_string(cols));
   }
   const MultiBodySystem &input_;
   FlatTables tables_;
   mecano_b200_handle *handle_ = nullptr;
   MatrixView fext_;
   void *stream_ = nullptr;
};

class InverseDynamicsCalculator : public BatchedCalculatorBase
{
 public:
   explicit InverseDynamicsCalculator(const MultiBodySystem &input, int device = 0) : BatchedCalculatorBase(input, device) {}
   void setConsiderCoriolisAndCentrifugalForces(bool v) { coriolis_ = v; }
   void setConsiderJointAccelerations(bool v) { accelerations_ = v; }
   bool areCoriolisAndCentrifugalForcesConsidered() const { return coriolis_; }
   bool areJointAccelerationsConsidered() const { return accelerations_; }
   // compute(jointAccelerationMatrix) + getJointTauMatrix(), for N states
   void compute(const MatrixView &q, const MatrixView &qd, const MatrixView &qdd, const MatrixView &tauOut, Memory where = Memory::Device)
   {
      const int64_t n = q.cols, nv = input_.getNumberOfDoFs(), nq = input_.getConfigurationMatrixSize();
      checkShape(q, nq, n, "q");
      checkShape(qd, nv, n, "qd");
      checkShape(qdd, nv, n, "qdd");
      checkShape(tauOut, nv, n, "tau");
      if (fext_.data) checkShape(fext_, 6 * (int64_t)tables_.parent.size(), n, "externalWrenches");
      if (q.ld != qd.ld || q.ld != qdd.ld || q.ld != tauOut.ld || (fext_.data && fext_.ld != q.ld))
         throw MatrixDimensionException("all matrices of one call must share the same leading dimension");
      const uint32_t flags = (coriolis_ ? 0u : MECANO_B200_RNEA_NO_CORIOLIS) | (accelerations_ ? 0u : MECANO_B200_RNEA_NO_ACCELERATIONS);
      const int64_t rows = 6 * (int64_t)tables_.parent.size();
      if (bodyAcc_.data) checkShape(bodyAcc_, rows, n, "bodyAccelerations");
      if (jointWrench_.data) checkShape(jointWrench_, rows, n, "jointWrenches");
      if ((bodyAcc_.data && bodyAcc_.ld != q.ld) || (jointWrench_.data && jointWrench_.ld != q.ld))
         throw MatrixDimensionException("all matrices of one call must share the same leading dimension");
      if (!bodyAcc_.data && !jointWrench_.data)
      {
         if (where == Memory::Device)
            check(mecano_b200_rnea(handle_, n, q.ld, q.data, qd.data, qdd.data, fext_.data, tauOut.data, flags, stream_));
         else
            check(mecano_b200_rnea_host(handle_, n, q.ld, q.data, qd.data, qdd.data, fext_.data, tauOut.data, flags));
      }
      else if (where == Memory::Device)
         check(mecano_b200_rnea_full(handle_, n, q.ld, q.data, qd.data, qdd.data, fext_.data, tauOut.data, bodyAcc_.data, jointWrench_.data, flags, stream_));
      else
         check(mecano_b200_rnea_full_host(handle_, n, q.ld, q.data, qd.data, qdd.data, fext_.data, tauOut.data, bodyAcc_.data, jointWrench_.data, flags));
   }
   // Where the next compute() leaves getBodyAcceleration(body) / getComputedJointWrench(joint) (InverseDynamicsCalculator.java:
   // 578-602) of all N states: (6 * nJoints) x N matrices, rows [6 j, 6 j + 6) for joint j / its successor, accelerations in the
   // body's CoM frame, wrenches in the joint's frameAfterJoint.  Empty views (the default) skip them.
   void setByProductOutputs(const MatrixView &bodyAccelerations, const MatrixView &jointWrenches)
   {
      bodyAcc_ = bodyAccelerations;
      jointWrench_ = jointWrenches;
   }

 private:
   bool coriolis_ = true, accelerations_ = true;
   MatrixView bodyAcc_, jointWrench_;
};

class ForwardDynamicsCalculator : public BatchedCalculatorBase
{
 public:
   explicit ForwardDynamicsCalculator(const MultiBodySystem &input, int device = 0) : BatchedCalculatorBase(input, device) {}
   // compute(jointTauMatrix) + getJointAccelerationMatrix(), for N states
   void compute(const MatrixView &q, const MatrixView &qd, const MatrixView &tau, const MatrixView &qddOut, Memory where = Memory::Device)
   {
      const int64_t n = q.cols, nv = input_.getNumberOfDoFs(), nq = input_.getConfigurationMatrixSize();
      checkShape(q, nq, n, "q");
      checkShape(qd, nv, n, "qd");
      checkShape(tau, nv, n, "tau");
      checkShape(qddOut, nv, n, "qdd");
      if (fext_.data) checkShape(fext_, 6 * (int64_t)tables_.parent.size(), n, "externalWrenches");
      if (q.ld != qd.ld || q.ld != tau.ld || q.ld != qddOut.ld || (fext_.data && fext_.ld != q.ld))
         throw MatrixDimensionException("all matrices of one call must share the same leading dimension");
      if (where == Memory::Device)
         check(mecano_b200_aba(handle_, n, q.ld, q.data, qd.data, tau.data, fext_.data, qddOut.data, 0u, stream_));
      else
         check(mecano_b200_aba_host(handle_, n, q.ld, q.data, qd.data, tau.data, fext_.data, qddOut.data, 0u));
   }

   // ---- joint source modes (ForwardDynamicsCalculator.java:45-57, :400-465)
   enum class JointSourceMode { EFFORT_SOURCE, ACCELERATION_SOURCE };
   void setJointSourceMode(const Joint *joint, JointSourceMode mode)
   {
      const int j = input_.indexOf(joint);
      const int row = j < 0 ? -1 : tables_.body_of_joint[(size_t)j];
      if (row < 0)
         throw ScrewTheoryException("the joint is not considered by this calculator");
      accelSource_.resize(tables_.parent.size(), 0);
      accelSource_[(size_t)row] = mode == JointSourceMode::ACCELERATION_SOURCE ? 1 : 0;
      check(mecano_b200_set_joint_source_modes(handle_, accelSource_.data()));
   }
   void resetJointSourceModes()
   {
      accelSource_.assign(tables_.parent.size(), 0);
      check(mecano_b200_set_joint_source_modes(handle_, nullptr));
   }
   JointSourceMode getJointSourceMode(const Joint *joint) const
   {
      const int j = input_.indexOf(joint);
      const int row = j < 0 ? -1 : tables_.body_of_joint[(size_t)j];
      return row >= 0 && (size_t)row < accelSource_.size() && accelSource_[(size_t)row] ? JointSourceMode::ACCELERATION_SOURCE : JointSourceMode::EFFORT_SOURCE;
   }
   // compute(jointTauMatrix, jointAccelerationMatrix) (:508-520) for N states: qddIn is read at the rows of the
   // ACCELERATION_SOURCE joints only; qddOut = getJointAccelerationMatrix(), tauOut (may be empty) = getJointTauMatrix()
   void compute(const MatrixView &q, const MatrixView &qd, const MatrixView &tau, const MatrixView &qddIn, const MatrixView &qddOut,
                const MatrixView &tauOut, Memory where = Memory::Device)
   {
      const int64_t n = q.cols, nv = input_.getNumberOfDoFs(), nq = input_.getConfigurationMatrixSize();
      checkShape(q, nq, n, "q");
      checkShape(qd, nv, n, "qd");
      checkShape(tau, nv, n, "tau");
      if (qddIn.data) checkShape(qddIn, nv, n, "jointAccelerationInput");
      checkShape(qddOut, nv, n, "qdd");
      if (tauOut.data) checkShape(tauOut, nv, n, "tauOut");
      if (fext_.data) checkShape(fext_, 6 * (int64_t)tables_.parent.size(), n, "externalWrenches");
      if (q.ld != qd.ld || q.ld != tau.ld || q.ld != qddOut.ld || (fext_.data && fext_.ld != q.ld) || (qddIn.data && qddIn.ld != q.ld) ||
          (tauOut.data && tauOut.ld != q.ld))
         throw MatrixDimensionException("all matrices of one call must share the same leading dimension");
      if (where == Memory::Device)
         check(mecano_b200_aba_sources(handle_, n, q.ld, q.data, qd.data, tau.data, qddIn.data, fext_.data, qddOut.data, tauOut.data, stream_));
      else
         check(mecano_b200_aba_sources_host(handle_, n, q.ld, q.data, qd.data, tau.data, qddIn.data, fext_.data, qddOut.data, tauOut.data));
   }

 private:
   std::vector<int32_t> accelSource_;
};

class CompositeRigidBodyMassMatrixCalculator : public BatchedCalculatorBase
{
 public:
   explicit CompositeRigidBodyMassMatrixCalculator(const MultiBodySystem &input, int device = 0) : BatchedCalculatorBase(input, device) {}
   // reset() + getMassMatrix() for N states.  massMatrixOut is (nDoFs*nDoFs) x N (entry-major, default) or,
   // with stateMajor, N x (nDoFs*nDoFs): one Mecano-style dense nDoFs x nDoFs matrix per state.
   void getMassMatrix(const MatrixView &q, const MatrixView &massMatrixOut, bool stateMajor = false, Memory where = Memory::Device)
   {
      const int64_t n = q.cols, nv = input_.getNumberOfDoFs(), nq = input_.getConfigurationMatrixSize();
      checkShape(q, nq, n, "q");
      if (stateMajor)
         checkShape(massMatrixOut, n, nv * nv, "massMatrix");
      else
      {
         checkShape(massMatrixOut, nv * nv, n, "massMatrix");
         if (massMatrixOut.ld != q.ld) throw MatrixDimensionException("q and massMatrix must share the same leading dimension");
      }
      const uint32_t layout = stateMajor ? MECANO_B200_CRBA_STATE_MAJOR : MECANO_B200_CRBA_ENTRY_MAJOR;
      if (where == Memory::Device)
         check(mecano_b200_crba(handle_, n, q.ld, q.data, massMatrixOut.data, layout, stream_));
      else
         check(mecano_b200_crba_host(handle_, n, q.ld, q.data, massMatrixOut.data, layout));
   }

   // ---- Coriolis and centrifugal matrix (CompositeRigidBodyMassMatrixCalculator.java:278-281, :358-366)
   void setEnableCoriolisMatrixCalculation(bool enable) { coriolisEnabled_ = enable; }
   // getMassMatrix() + getCoriolisMatrix() for N states: both (nDoFs*nDoFs) x N, entry-major
   void getCoriolisMatrix(const MatrixView &q, const MatrixView &qd, const MatrixView &massMatrixOut, const MatrixView &coriolisMatrixOut,
                          Memory where = Memory::Device)
   {
      if (!coriolisEnabled_)
         throw std::runtime_error("Coriolis matrix calculation is disabled."); // UnsupportedOperationException, :360-361
      const int64_t n = q.cols, nv = input_.getNumberOfDoFs(), nq = input_.getConfigurationMatrixSize();
      checkShape(q, nq, n, "q");
      checkShape(qd, nv, n, "qd");
      checkShape(massMatrixOut, nv * nv, n, "massMatrix");
      checkShape(coriolisMatrixOut, nv * nv, n, "coriolisMatrix");
      if (qd.ld != q.ld || massMatrixOut.ld != q.ld || coriolisMatrixOut.ld != q.ld)
         throw MatrixDimensionException("all matrices of one call must share the same leading dimension");
      if (where == Memory::Device)
         check(mecano_b200_coriolis(handle_, n, q.ld, q.data, qd.data, massMatrixOut.data, coriolisMatrixOut.data, stream_));
      else
         check(mecano_b200_coriolis_host(handle_, n, q.ld, q.data, qd.data, massMatrixOut.data, coriolisMatrixOut.data));
   }

   // ---- centroidal by-products (CompositeRigidBodyMassMatrixCalculator.java:380-440, :801-839)
   enum class CentroidalMomentumFrame { World = MECANO_B200_FRAME_WORLD, CenterOfMass = MECANO_B200_FRAME_CENTER_OF_MASS };
   void setCentroidalMomentumFrame(CentroidalMomentumFrame f) { frame_ = f; }
   CentroidalMomentumFrame getCentroidalMomentumFrame() const { return frame_; }
   // getMassMatrix() + getCentroidalMomentumMatrix() for N states: massMatrixOut (nDoFs*nDoFs) x N entry-major, cmmOut (6*nDoFs) x N
   // (entry (r, j) at row r * nDoFs + j), comOut 4 x N (centre of mass in the root frame, total mass)
   void getCentroidalMomentumMatrix(const MatrixView &q, const MatrixView &massMatrixOut, const MatrixView &cmmOut, const MatrixView &comOut,
                                    Memory where = Memory::Device)
   {
      const int64_t n = q.cols, nv = input_.getNumberOfDoFs(), nq = input_.getConfigurationMatrixSize();
      checkShape(q, nq, n, "q");
      checkShape(massMatrixOut, nv * nv, n, "massMatrix");
      checkShape(cmmOut, 6 * nv, n, "centroidalMomentumMatrix");
      checkShape(comOut, 4, n, "centerOfMass");
      if (massMatrixOut.ld != q.ld || cmmOut.ld != q.ld || comOut.ld != q.ld)
         throw MatrixDimensionException("all matrices of one call must share the same leading dimension");
      if (where == Memory::Device)
         check(mecano_b200_crba_centroidal(handle_, n, q.ld, q.data, massMatrixOut.data, cmmOut.data, comOut.data, (int)frame_, stream_));
      else
         check(mecano_b200_crba_centroidal_host(handle_, n, q.ld, q.data, massMatrixOut.data, cmmOut.data, comOut.data, (int)frame_));
   }
   // the centre of mass and total mass alone (CenterOfMassCalculator.getCenterOfMass() / getTotalMass(), CenterOfMassCalculator.java:
   // 70-124), comOut 4 x N: no matrix computed or written, the rows getCentroidalMomentumMatrix() leaves bit for bit
   void getCenterOfMass(const MatrixView &q, const MatrixView &comOut, Memory where = Memory::Device)
   {
      const int64_t n = q.cols, nq = input_.getConfigurationMatrixSize();
      checkShape(q, nq, n, "q");
      checkShape(comOut, 4, n, "centerOfMass");
      if (comOut.ld != q.ld)
         throw MatrixDimensionException("all matrices of one call must share the same leading dimension");
      if (where == Memory::Device)
         check(mecano_b200_center_of_mass(handle_, n, q.ld, q.data, comOut.data, stream_));
      else
         check(mecano_b200_center_of_mass_host(handle_, n, q.ld, q.data, comOut.data));
   }
   // getCentroidalConvectiveTermMatrix() for N states: out 6 x N; com = the rows written by getCentroidalMomentumMatrix() or
   // getCenterOfMass() for the same q (read in the centre-of-mass frame only)
   void getCentroidalConvectiveTermMatrix(const MatrixView &q, const MatrixView &qd, const MatrixView &com, const MatrixView &out,
                                          Memory where = Memory::Device)
   {
      const int64_t n = q.cols, nv = input_.getNumberOfDoFs(), nq = input_.getConfigurationMatrixSize();
      checkShape(q, nq, n, "q");
      checkShape(qd, nv, n, "qd");
      checkShape(out, 6, n, "centroidalConvectiveTerm");
      if (com.data) checkShape(com, 4, n, "centerOfMass");
      if (qd.ld != q.ld || out.ld != q.ld || (com.data && com.ld != q.ld))
         throw MatrixDimensionException("all matrices of one call must share the same leading dimension");
      if (where == Memory::Device)
         check(mecano_b200_centroidal_convective_term(handle_, n, q.ld, q.data, qd.data, com.data, out.data, (int)frame_, stream_));
      else
         check(mecano_b200_centroidal_convective_term_host(handle_, n, q.ld, q.data, qd.data, com.data, out.data, (int)frame_));
   }

 private:
   CentroidalMomentumFrame frame_ = CentroidalMomentumFrame::World;
   bool coriolisEnabled_ = false;
};

// JointTorqueRegressorCalculator: the inertial-parameter regressor Y(q, qd, qdd) of inverse dynamics, tau = Y pi for any inertial
// parameters pi (mecano_b200_joint_torque_regressor: layout, column order MECANO_B200_REGRESSOR_*, frames).  Systems whose fixed /
// ignored joints are welded into other bodies are refused by the C ABI here (a welded body has no block of its own); the Python
// calculator runs them on the expanded tables.
class JointTorqueRegressorCalculator : public BatchedCalculatorBase
{
 public:
   explicit JointTorqueRegressorCalculator(const MultiBodySystem &input, int device = 0) : BatchedCalculatorBase(input, device) {}
   int64_t getNumberOfParameters() const { return 10 * (int64_t)tables_.parent.size(); }
   // compute(q, qd, qdd) + getJointTorqueRegressorMatrix(), for N states: (nDoFs * 10 nBodies) x N, entry-major
   void compute(const MatrixView &q, const MatrixView &qd, const MatrixView &qdd, const MatrixView &regressorOut, Memory where = Memory::Device)
   {
      const int64_t n = q.cols, nv = input_.getNumberOfDoFs(), nq = input_.getConfigurationMatrixSize();
      checkShape(q, nq, n, "q");
      checkShape(qd, nv, n, "qd");
      checkShape(qdd, nv, n, "qdd");
      checkShape(regressorOut, nv * getNumberOfParameters(), n, "jointTorqueRegressor");
      if (qd.ld != q.ld || qdd.ld != q.ld || regressorOut.ld != q.ld)
         throw MatrixDimensionException("all matrices of one call must share the same leading dimension");
      if (where == Memory::Device)
         check(mecano_b200_joint_torque_regressor(handle_, n, q.ld, q.data, qd.data, qdd.data, regressorOut.data, stream_));
      else
         check(mecano_b200_joint_torque_regressor_host(handle_, n, q.ld, q.data, qd.data, qdd.data, regressorOut.data));
   }
   // the model's own parameters in the column order of Y: [m, 0, 0, 0, J_xx, J_xy, J_xz, J_yy, J_yz, J_zz] per body (CoM frame)
   std::vector<double> getInertialParameterVector() const
   {
      const size_t nb = tables_.parent.size();
      std::vector<double> pi(10 * nb, 0.0);
      const int sym[6] = {0, 1, 2, 4, 5, 8};
      for (size_t b = 0; b < nb; b++)
      {
         const size_t w = tables_.wrench_index.empty() ? b : (size_t)tables_.wrench_index[b];
         if (w >= nb)
            throw std::runtime_error("getInertialParameterVector: the system has welded bodies (fixed / ignored joints)");
         pi[10 * w + MECANO_B200_REGRESSOR_M] = tables_.mass[b];
         for (int k = 0; k < 6; k++)
            pi[10 * w + MECANO_B200_REGRESSOR_I + k] = tables_.inertia[9 * b + sym[k]];
      }
      return pi;
   }
};

// MultiBodyGravityGradientCalculator: the joint efforts tau_g(q) that gravity and the external wrenches cause, and their configuration
// gradient G = d tau_g / dq (mecano_b200_gravity_gradient: layout, floating-base and external-wrench conventions).  For systems
// without welded bodies (fixed / ignored joints): with external wrenches the C ABI refuses their tables, whose wrench ranks count
// the welded joints; the Python calculator runs them on the expanded tables.
class MultiBodyGravityGradientCalculator : public BatchedCalculatorBase
{
 public:
   explicit MultiBodyGravityGradientCalculator(const MultiBodySystem &input, int device = 0) : BatchedCalculatorBase(input, device) {}
   // compute(q) + getTauMatrix() (nDoFs x N) + getTauGradientMatrix() ((nDoFs * nDoFs) x N, entry (i, j) at row i * nDoFs + j)
   void compute(const MatrixView &q, const MatrixView &tauOut, const MatrixView &gradientOut, Memory where = Memory::Device)
   {
      const int64_t n = q.cols, nv = input_.getNumberOfDoFs(), nq = input_.getConfigurationMatrixSize();
      checkShape(q, nq, n, "q");
      checkShape(tauOut, nv, n, "tau");
      checkShape(gradientOut, nv * nv, n, "tauGradient");
      if (fext_.data) checkShape(fext_, 6 * (int64_t)tables_.parent.size(), n, "externalWrenches");
      if (tauOut.ld != q.ld || gradientOut.ld != q.ld || (fext_.data && fext_.ld != q.ld))
         throw MatrixDimensionException("all matrices of one call must share the same leading dimension");
      if (where == Memory::Device)
         check(mecano_b200_gravity_gradient(handle_, n, q.ld, q.data, fext_.data, tauOut.data, gradientOut.data, stream_));
      else
         check(mecano_b200_gravity_gradient_host(handle_, n, q.ld, q.data, fext_.data, tauOut.data, gradientOut.data));
   }
};

// InverseDynamicsDerivativesCalculator: the joint efforts tau(q, qd, qdd) and their partials d tau / dq, d tau / dqd
// (mecano_b200_rnea_derivatives: layout, floating-base and external-wrench conventions).  For systems without welded bodies (fixed /
// ignored joints) with external wrenches, as MultiBodyGravityGradientCalculator.
class InverseDynamicsDerivativesCalculator : public BatchedCalculatorBase
{
 public:
   explicit InverseDynamicsDerivativesCalculator(const MultiBodySystem &input, int device = 0) : BatchedCalculatorBase(input, device) {}
   // compute(q, qd, qdd) + getJointTauMatrix() (nDoFs x N) + getTauConfigurationGradientMatrix() / getTauVelocityGradientMatrix()
   // ((nDoFs * nDoFs) x N each, entry (i, j) at row i * nDoFs + j)
   void compute(const MatrixView &q, const MatrixView &qd, const MatrixView &qdd, const MatrixView &tauOut, const MatrixView &dqOut,
                const MatrixView &dqdOut, Memory where = Memory::Device)
   {
      const int64_t n = q.cols, nv = input_.getNumberOfDoFs(), nq = input_.getConfigurationMatrixSize();
      checkShape(q, nq, n, "q");
      checkShape(qd, nv, n, "qd");
      checkShape(qdd, nv, n, "qdd");
      checkShape(tauOut, nv, n, "tau");
      checkShape(dqOut, nv * nv, n, "tauConfigurationGradient");
      checkShape(dqdOut, nv * nv, n, "tauVelocityGradient");
      if (fext_.data) checkShape(fext_, 6 * (int64_t)tables_.parent.size(), n, "externalWrenches");
      if (qd.ld != q.ld || qdd.ld != q.ld || tauOut.ld != q.ld || dqOut.ld != q.ld || dqdOut.ld != q.ld || (fext_.data && fext_.ld != q.ld))
         throw MatrixDimensionException("all matrices of one call must share the same leading dimension");
      if (where == Memory::Device)
         check(mecano_b200_rnea_derivatives(handle_, n, q.ld, q.data, qd.data, qdd.data, fext_.data, tauOut.data, dqOut.data, dqdOut.data, stream_));
      else
         check(mecano_b200_rnea_derivatives_host(handle_, n, q.ld, q.data, qd.data, qdd.data, fext_.data, tauOut.data, dqOut.data, dqdOut.data));
   }
};

// ForwardDynamicsDerivativesCalculator: the joint accelerations qdd(q, qd, tau) and their partials d qdd / dq, d qdd / dqd and
// d qdd / d tau = M^-1 (mecano_b200_aba_derivatives: layout, floating-base and external-wrench conventions).  Systems with fixed /
// ignored joints run on their welded tables; with external wrenches the call refuses them (their wrench ranks count the welded
// bodies).
class ForwardDynamicsDerivativesCalculator : public BatchedCalculatorBase
{
 public:
   explicit ForwardDynamicsDerivativesCalculator(const MultiBodySystem &input, int device = 0) : BatchedCalculatorBase(input, device) {}
   // compute(q, qd, tau) + getJointAccelerationMatrix() (nDoFs x N) + getAccelerationConfigurationGradientMatrix() /
   // getAccelerationVelocityGradientMatrix() / getInverseMassMatrix() ((nDoFs * nDoFs) x N each, entry (i, j) at row i * nDoFs + j)
   void compute(const MatrixView &q, const MatrixView &qd, const MatrixView &tau, const MatrixView &qddOut, const MatrixView &dqOut,
                const MatrixView &dqdOut, const MatrixView &minvOut, Memory where = Memory::Device)
   {
      const int64_t n = q.cols, nv = input_.getNumberOfDoFs(), nq = input_.getConfigurationMatrixSize();
      checkShape(q, nq, n, "q");
      checkShape(qd, nv, n, "qd");
      checkShape(tau, nv, n, "tau");
      checkShape(qddOut, nv, n, "qdd");
      checkShape(dqOut, nv * nv, n, "accelerationConfigurationGradient");
      checkShape(dqdOut, nv * nv, n, "accelerationVelocityGradient");
      checkShape(minvOut, nv * nv, n, "inverseMassMatrix");
      if (fext_.data) checkShape(fext_, 6 * (int64_t)tables_.parent.size(), n, "externalWrenches");
      if (qd.ld != q.ld || tau.ld != q.ld || qddOut.ld != q.ld || dqOut.ld != q.ld || dqdOut.ld != q.ld || minvOut.ld != q.ld ||
          (fext_.data && fext_.ld != q.ld))
         throw MatrixDimensionException("all matrices of one call must share the same leading dimension");
      if (where == Memory::Device)
         check(mecano_b200_aba_derivatives(handle_, n, q.ld, q.data, qd.data, tau.data, fext_.data, qddOut.data, dqOut.data, dqdOut.data, minvOut.data,
                                           stream_));
      else
         check(mecano_b200_aba_derivatives_host(handle_, n, q.ld, q.data, qd.data, tau.data, fext_.data, qddOut.data, dqOut.data, dqdOut.data,
                                                minvOut.data));
   }
};
} // namespace mecano
