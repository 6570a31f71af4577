/**
 * @file ContactRolloutBatch.h
 * Batched forms of the steps either side of the contact model (no reference equivalent as a
 * class; the per-system semantics are those of FloatingBaseSystemKinematics + ForwardEuler and of
 * FloatingBaseDynamicalSystem::dynamics from the bias forces on,
 * src/System/src/FloatingBaseSystemDynamics.cpp:188-248).  Host code is C++17 and reaches the GPU
 * only through the C ABI (include/blf_ccm.h).
 */
#ifndef BIPEDAL_LOCOMOTION_SYSTEM_CONTACT_ROLLOUT_BATCH_H
#define BIPEDAL_LOCOMOTION_SYSTEM_CONTACT_ROLLOUT_BATCH_H

#include <cstddef>
#include <cstdint>
#include <memory>

#include <BipedalLocomotion/ContactModels/ContinuousContactModelBatch.h>
#include <BipedalLocomotion/GenericContainer/DeviceSoA.h>

namespace BipedalLocomotion
{
namespace System
{

class ContactRolloutBatch
{
public:
    struct Result
    {
        double cost;
        std::int64_t index; /**< -1 when there is nothing to compare */
    };

    /** Shares the device handle (and the uniform contact parameters) of `model`. */
    explicit ContactRolloutBatch(std::shared_ptr<ContactModels::CudaDevice> device);
    ~ContactRolloutBatch();
    ContactRolloutBatch(const ContactRolloutBatch&) = delete;
    ContactRolloutBatch& operator=(const ContactRolloutBatch&) = delete;

    /** One ForwardEuler step of FloatingBaseSystemKinematics for every system:
     * twists 6 planes, positions 3 planes and rotations 9 planes (row-major) updated in place. */
    bool eulerStep(double rho, double dT, const GenericContainer::DeviceSoA& twists,
                   GenericContainer::DeviceSoA& positions, GenericContainer::DeviceSoA& rotations,
                   void* stream = nullptr);

    /**
     * Fused sampling-MPC rollout (integrate -> contact model -> cost); layouts in
     * include/blf_ccm.h, blf_ccm_rollout_integrate_cost.  twists: 6 planes of horizon*chains
     * (time-major), positions/rotations/nullPoses: 3/9/12 planes of chains = nRollouts*feet.
     * Optional trajectories per `outputs` (ContinuousContactModelBatch::Output bits 1|2|4),
     * optional final pose; costs (device, nRollouts) may be nullptr; best = 16 device bytes.
     */
    bool rollout(std::size_t nRollouts, int feet, int horizon, double dT, double rho,
                 const GenericContainer::DeviceSoA& twists, const GenericContainer::DeviceSoA& positions,
                 const GenericContainer::DeviceSoA& rotations, const GenericContainer::DeviceSoA& nullPoses,
                 const GenericContainer::DeviceSoA* parameters, unsigned outputs,
                 GenericContainer::DeviceSoA* wrench, GenericContainer::DeviceSoA* autonomousDynamics,
                 double* controlMatrix, GenericContainer::DeviceSoA* finalPositions,
                 GenericContainer::DeviceSoA* finalRotations, const iDynTree::Wrench& referenceWrench,
                 double forceWeight, double torqueWeight, std::int64_t indexBase, double* costs,
                 void* best, void* stream = nullptr);
    /** Cost-only form that copies the arg-min pair to the host (synchronises the stream). */
    bool rollout(std::size_t nRollouts, int feet, int horizon, double dT, double rho,
                 const GenericContainer::DeviceSoA& twists, const GenericContainer::DeviceSoA& positions,
                 const GenericContainer::DeviceSoA& rotations, const GenericContainer::DeviceSoA& nullPoses,
                 const GenericContainer::DeviceSoA* parameters, const iDynTree::Wrench& referenceWrench,
                 double forceWeight, double torqueWeight, Result& result);

    /**
     * Reverse mode of the rollouts' cost (blf_ccm_rollout_cost_vjp; no reference counterpart): for
     * the cotangents gradCost (device, nRollouts) of the costs `rollout` computes from the same
     * inputs, writes gradCost^T dcost/d(input) into the requested outputs -- twistGradient 6 planes
     * of horizon*chains (time-major), positionGradient + rotationGradient 3 + 9 planes (both or
     * neither), nullPoseGradient 12, parameterGradient 4 planes of chains (each chain's share).
     * nullptr = not requested; at least one must be given.  Outputs must not alias inputs.
     */
    bool rolloutCostGradient(std::size_t nRollouts, int feet, int horizon, double dT, double rho,
                             const GenericContainer::DeviceSoA& twists,
                             const GenericContainer::DeviceSoA& positions,
                             const GenericContainer::DeviceSoA& rotations,
                             const GenericContainer::DeviceSoA& nullPoses,
                             const GenericContainer::DeviceSoA* parameters,
                             const iDynTree::Wrench& referenceWrench, double forceWeight,
                             double torqueWeight, const double* gradCost,
                             GenericContainer::DeviceSoA* twistGradient,
                             GenericContainer::DeviceSoA* positionGradient,
                             GenericContainer::DeviceSoA* rotationGradient,
                             GenericContainer::DeviceSoA* nullPoseGradient,
                             GenericContainer::DeviceSoA* parameterGradient, void* stream = nullptr);

    /**
     * Cost-only rollouts with every plane in HOST memory (blf_ccm_rollout_integrate_cost_host):
     * twistPlanes[6] of horizon*chains doubles (time-major), positionPlanes[3], rotationPlanes[9],
     * nullPosePlanes[12] (third rotation column may be null) and optional parameterPlanes[4] of
     * chains doubles.  Uploads are pipelined with the kernels; costs (host, nRollouts) may be
     * nullptr.  Returns when `result` is written.
     */
    bool rolloutHost(std::size_t nRollouts, int feet, int horizon, double dT, double rho,
                     const double* const* twistPlanes, const double* const* positionPlanes,
                     const double* const* rotationPlanes, const double* const* nullPosePlanes,
                     const double* const* parameterPlanes, const iDynTree::Wrench& referenceWrench,
                     double forceWeight, double torqueWeight, double* costs, Result& result);

    /**
     * knownCoefficient[s] = base[s] + sum_c J_c^T wrench_c  (FloatingBaseSystemDynamics.cpp:199-226)
     * states: 30 planes of nSystems*contactsPerSystem contacts; jacobians: device array of
     * 6 x columns row-major blocks per contact; base (may be nullptr, may alias out) and out:
     * nSystems x columns row-major.
     */
    bool generalizedForce(std::size_t nSystems, int contactsPerSystem, int columns,
                          const GenericContainer::DeviceSoA& states,
                          const GenericContainer::DeviceSoA* parameters, const double* jacobians,
                          const double* base, double* out, GenericContainer::DeviceSoA* wrench = nullptr,
                          void* stream = nullptr);

    /**
     * Last step of FloatingBaseDynamicalSystem::dynamics (FloatingBaseSystemDynamics.cpp:226-243):
     * acceleration[s] = (massMatrices[s] + regularization).llt().solve(known[s] (+ jointTorques[s] on
     * the tail)).  Device arrays: massMatrices nSystems x columns x columns row-major (the lower
     * triangle is read), regularization columns x columns or nullptr (what
     * setMassMatrixRegularization stores), known / acceleration nSystems x columns (may alias),
     * jointTorques nSystems x (columns - 6) or nullptr.
     */
    bool massMatrixSolve(std::size_t nSystems, int columns, const double* massMatrices,
                         const double* regularization, const double* known, const double* jointTorques,
                         double* acceleration, void* stream = nullptr);

    /**
     * dynamics() from the bias forces on (:188-248), the rigid-body quantities supplied by the caller:
     * acceleration = (M + regularization).llt().solve(-biasForces + sum_c J_c^T wrench_c + [0; jointTorques]).
     * states / parameters / jacobians / wrench as generalizedForce; biasForces nSystems x columns
     * = [base wrench; joint torques] of generalizedBiasForces.
     */
    bool floatingBaseAcceleration(std::size_t nSystems, int contactsPerSystem, int columns,
                                  const GenericContainer::DeviceSoA& states,
                                  const GenericContainer::DeviceSoA* parameters, const double* jacobians,
                                  const double* biasForces, const double* jointTorques,
                                  const double* massMatrices, const double* regularization,
                                  double* acceleration, GenericContainer::DeviceSoA* wrench = nullptr,
                                  void* stream = nullptr);

    /**
     * The base part of FloatingBaseSystemKinematics::dynamics / FloatingBaseDynamicalSystem::dynamics
     * (FloatingBaseSystemKinematics.cpp:60-70, FloatingBaseSystemDynamics.cpp:134-140) for device arrays:
     * twists nSystems x 6, rotations nSystems x 9 row-major -> linearVelocities nSystems x 3,
     * rotationRates nSystems x 9.
     */
    bool kinematicsDynamics(std::size_t nSystems, double rho, const double* twists, const double* rotations,
                            double* linearVelocities, double* rotationRates, void* stream = nullptr);

    /**
     * One ForwardEuler step of FloatingBaseDynamicalSystem (ForwardEuler.tpp:19-49 over the state tuple
     * of FloatingBaseSystemDynamics.h:33-52), in place, every derivative at the state before the step:
     * basePosition += velocity.head<3>() dT, baseRotation += (rotation rate of
     * FloatingBaseSystemDynamics.cpp:139-145 with the Baumgarte parameter rho) dT, jointPositions +=
     * velocity.tail dT, velocity += acceleration dT.  Device arrays: acceleration / velocity nSystems x
     * columns ([base (6); joints]), jointPositions nSystems x (columns - 6) (nullptr when columns == 6),
     * basePositions nSystems x 3, baseRotations nSystems x 9 row-major.
     */
    bool floatingBaseEulerStep(std::size_t nSystems, int columns, double rho, double dT,
                               const double* acceleration, double* velocity, double* jointPositions,
                               double* basePositions, double* baseRotations, void* stream = nullptr);

private:
    std::shared_ptr<ContactModels::CudaDevice> m_device;
    void* m_best{nullptr};
};

} // namespace System
} // namespace BipedalLocomotion

#endif // BIPEDAL_LOCOMOTION_SYSTEM_CONTACT_ROLLOUT_BATCH_H
