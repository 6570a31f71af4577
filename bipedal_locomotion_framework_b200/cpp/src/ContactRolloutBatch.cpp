/**
 * @file ContactRolloutBatch.cpp
 * Thin C++17 layer over blf_sys_kinematics_euler_step_soa, blf_ccm_rollout_integrate_cost,
 * blf_ccm_rollout_cost_vjp and
 * blf_ccm_generalized_force_soa.
 */
#include <iostream>

#include <BipedalLocomotion/System/ContactRolloutBatch.h>

#include "blf_ccm.h"

using namespace BipedalLocomotion::System;
using namespace BipedalLocomotion::GenericContainer;
using BipedalLocomotion::ContactModels::CudaDevice;

namespace
{
blf_ccm_handle* raw(const std::shared_ptr<CudaDevice>& d)
{
    return d ? static_cast<blf_ccm_handle*>(d->handle()) : nullptr;
}

bool report(int rc, const char* where)
{
    if (rc == BLF_CCM_OK) return true;
    std::cerr << "[ContactRolloutBatch::" << where << "] " << blf_ccm_last_error() << std::endl;
    return false;
}

bool planes(const DeviceSoA& s, std::size_t want, std::size_t size, const char* what, const char* where)
{
    if (s.planes() == want && s.size() == size) return true;
    std::cerr << "[ContactRolloutBatch::" << where << "] " << what << " must have " << want
              << " planes of " << size << " doubles." << std::endl;
    return false;
}
} // namespace

ContactRolloutBatch::ContactRolloutBatch(std::shared_ptr<CudaDevice> device) : m_device(std::move(device)) {}

ContactRolloutBatch::~ContactRolloutBatch()
{
    if (m_best != nullptr && m_device != nullptr) blf_ccm_device_free(raw(m_device), m_best);
}

bool ContactRolloutBatch::eulerStep(double rho, double dT, const DeviceSoA& twists, DeviceSoA& positions,
                                    DeviceSoA& rotations, void* stream)
{
    if (m_device == nullptr) return report(BLF_CCM_ERR_INVALID_HANDLE, "eulerStep");
    const std::size_t n = twists.size();
    if (!planes(twists, 6, n, "twists", "eulerStep") || !planes(positions, 3, n, "positions", "eulerStep")
        || !planes(rotations, 9, n, "rotations", "eulerStep"))
        return false;
    return report(blf_sys_kinematics_euler_step_soa(raw(m_device), static_cast<std::int64_t>(n), rho, dT,
                                                    twists.planePointers(), positions.planePointers(),
                                                    rotations.planePointers(), stream),
                  "eulerStep");
}

bool ContactRolloutBatch::rollout(std::size_t nRollouts, int feet, int horizon, double dT, double rho,
                                  const DeviceSoA& twists, const DeviceSoA& positions,
                                  const DeviceSoA& rotations, const DeviceSoA& nullPoses,
                                  const DeviceSoA* parameters, unsigned outputs, DeviceSoA* wrench,
                                  DeviceSoA* autonomousDynamics, double* controlMatrix,
                                  DeviceSoA* finalPositions, DeviceSoA* finalRotations,
                                  const iDynTree::Wrench& referenceWrench, double forceWeight,
                                  double torqueWeight, std::int64_t indexBase, double* costs, void* best,
                                  void* stream)
{
    if (m_device == nullptr) return report(BLF_CCM_ERR_INVALID_HANDLE, "rollout");
    if (feet < 1 || horizon < 1)
    {
        std::cerr << "[ContactRolloutBatch::rollout] feet and horizon must be positive." << std::endl;
        return false;
    }
    const std::size_t chains = nRollouts * static_cast<std::size_t>(feet);
    if (!planes(twists, 6, chains * static_cast<std::size_t>(horizon), "twists", "rollout")
        || !planes(positions, 3, chains, "positions", "rollout")
        || !planes(rotations, 9, chains, "rotations", "rollout")
        || !planes(nullPoses, 12, chains, "nullPoses", "rollout"))
        return false;
    const double weights[2] = {forceWeight, torqueWeight};
    return report(blf_ccm_rollout_integrate_cost(
                      raw(m_device), static_cast<std::int64_t>(nRollouts), feet, horizon, dT, rho,
                      twists.planePointers(), positions.planePointers(), rotations.planePointers(),
                      nullPoses.planePointers(), parameters ? parameters->planePointers() : nullptr,
                      outputs, wrench ? wrench->planePointers() : nullptr,
                      autonomousDynamics ? autonomousDynamics->planePointers() : nullptr, controlMatrix,
                      finalPositions ? finalPositions->planePointers() : nullptr,
                      finalRotations ? finalRotations->planePointers() : nullptr, referenceWrench.data(),
                      weights, indexBase, costs, best, stream),
                  "rollout");
}

bool ContactRolloutBatch::rolloutCostGradient(std::size_t nRollouts, int feet, int horizon, double dT,
                                              double rho, const DeviceSoA& twists, const DeviceSoA& positions,
                                              const DeviceSoA& rotations, const DeviceSoA& nullPoses,
                                              const DeviceSoA* parameters, const iDynTree::Wrench& referenceWrench,
                                              double forceWeight, double torqueWeight, const double* gradCost,
                                              DeviceSoA* twistGradient, DeviceSoA* positionGradient,
                                              DeviceSoA* rotationGradient, DeviceSoA* nullPoseGradient,
                                              DeviceSoA* parameterGradient, void* stream)
{
    const char* where = "rolloutCostGradient";
    if (m_device == nullptr) return report(BLF_CCM_ERR_INVALID_HANDLE, where);
    if (feet < 1 || horizon < 1)
    {
        std::cerr << "[ContactRolloutBatch::rolloutCostGradient] feet and horizon must be positive." << std::endl;
        return false;
    }
    const std::size_t chains = nRollouts * static_cast<std::size_t>(feet);
    const std::size_t steps = chains * static_cast<std::size_t>(horizon);
    if (!planes(twists, 6, steps, "twists", where) || !planes(positions, 3, chains, "positions", where)
        || !planes(rotations, 9, chains, "rotations", where) || !planes(nullPoses, 12, chains, "nullPoses", where)
        || (twistGradient && !planes(*twistGradient, 6, steps, "twistGradient", where))
        || (positionGradient && !planes(*positionGradient, 3, chains, "positionGradient", where))
        || (rotationGradient && !planes(*rotationGradient, 9, chains, "rotationGradient", where))
        || (nullPoseGradient && !planes(*nullPoseGradient, 12, chains, "nullPoseGradient", where))
        || (parameterGradient && !planes(*parameterGradient, 4, chains, "parameterGradient", where)))
        return false;
    const double weights[2] = {forceWeight, torqueWeight};
    auto out = [](DeviceSoA* s) { return s ? s->planePointers() : nullptr; };
    return report(blf_ccm_rollout_cost_vjp(
                      raw(m_device), static_cast<std::int64_t>(nRollouts), feet, horizon, dT, rho,
                      twists.planePointers(), positions.planePointers(), rotations.planePointers(),
                      nullPoses.planePointers(), parameters ? parameters->planePointers() : nullptr,
                      referenceWrench.data(), weights, gradCost, out(twistGradient), out(positionGradient),
                      out(rotationGradient), out(nullPoseGradient), out(parameterGradient), stream),
                  where);
}

bool ContactRolloutBatch::rollout(std::size_t nRollouts, int feet, int horizon, double dT, double rho,
                                  const DeviceSoA& twists, const DeviceSoA& positions,
                                  const DeviceSoA& rotations, const DeviceSoA& nullPoses,
                                  const DeviceSoA* parameters, const iDynTree::Wrench& referenceWrench,
                                  double forceWeight, double torqueWeight, Result& result)
{
    if (m_device == nullptr) return report(BLF_CCM_ERR_INVALID_HANDLE, "rollout");
    blf_ccm_handle* h = raw(m_device);
    if (m_best == nullptr && !report(blf_ccm_device_alloc(h, 16, &m_best), "rollout")) return false;
    if (!rollout(nRollouts, feet, horizon, dT, rho, twists, positions, rotations, nullPoses, parameters, 0u,
                 nullptr, nullptr, nullptr, nullptr, nullptr, referenceWrench, forceWeight, torqueWeight, 0,
                 nullptr, m_best, nullptr))
        return false;
    struct
    {
        double cost;
        std::int64_t index;
    } pair;
    if (!report(blf_ccm_copy_d2h(h, &pair, m_best, 16, nullptr), "rollout")) return false;
    if (!report(blf_ccm_stream_synchronize(h, nullptr), "rollout")) return false;
    result.cost = pair.cost;
    result.index = pair.index;
    return true;
}

bool ContactRolloutBatch::rolloutHost(std::size_t nRollouts, int feet, int horizon, double dT, double rho,
                                      const double* const* twistPlanes,
                                      const double* const* positionPlanes,
                                      const double* const* rotationPlanes,
                                      const double* const* nullPosePlanes,
                                      const double* const* parameterPlanes,
                                      const iDynTree::Wrench& referenceWrench, double forceWeight,
                                      double torqueWeight, double* costs, Result& result)
{
    if (m_device == nullptr) return report(BLF_CCM_ERR_INVALID_HANDLE, "rolloutHost");
    const double weights[2] = {forceWeight, torqueWeight};
    std::int64_t index = -1;
    if (!report(blf_ccm_rollout_integrate_cost_host(raw(m_device), static_cast<std::int64_t>(nRollouts),
                                                    feet, horizon, dT, rho, twistPlanes, positionPlanes,
                                                    rotationPlanes, nullPosePlanes, parameterPlanes,
                                                    referenceWrench.data(), weights, costs, &result.cost,
                                                    &index),
                "rolloutHost"))
        return false;
    result.index = index;
    return true;
}

bool ContactRolloutBatch::generalizedForce(std::size_t nSystems, int contactsPerSystem, int columns,
                                           const DeviceSoA& states, const DeviceSoA* parameters,
                                           const double* jacobians, const double* base, double* out,
                                           DeviceSoA* wrench, void* stream)
{
    if (m_device == nullptr) return report(BLF_CCM_ERR_INVALID_HANDLE, "generalizedForce");
    if (contactsPerSystem < 1
        || !planes(states, 30, nSystems * static_cast<std::size_t>(contactsPerSystem), "states",
                   "generalizedForce"))
        return false;
    return report(blf_ccm_generalized_force_soa(raw(m_device), static_cast<std::int64_t>(nSystems),
                                                contactsPerSystem, columns, states.planePointers(),
                                                parameters ? parameters->planePointers() : nullptr,
                                                jacobians, base, out,
                                                wrench ? wrench->planePointers() : nullptr, stream),
                  "generalizedForce");
}

bool ContactRolloutBatch::massMatrixSolve(std::size_t nSystems, int columns, const double* massMatrices,
                                          const double* regularization, const double* known,
                                          const double* jointTorques, double* acceleration, void* stream)
{
    if (m_device == nullptr) return report(BLF_CCM_ERR_INVALID_HANDLE, "massMatrixSolve");
    return report(blf_sys_mass_matrix_solve(raw(m_device), static_cast<std::int64_t>(nSystems), columns,
                                            massMatrices, regularization, known, jointTorques, acceleration,
                                            stream),
                  "massMatrixSolve");
}

bool ContactRolloutBatch::floatingBaseAcceleration(std::size_t nSystems, int contactsPerSystem, int columns,
                                                   const DeviceSoA& states, const DeviceSoA* parameters,
                                                   const double* jacobians, const double* biasForces,
                                                   const double* jointTorques, const double* massMatrices,
                                                   const double* regularization, double* acceleration,
                                                   DeviceSoA* wrench, void* stream)
{
    if (m_device == nullptr) return report(BLF_CCM_ERR_INVALID_HANDLE, "floatingBaseAcceleration");
    if (contactsPerSystem < 1
        || !planes(states, 30, nSystems * static_cast<std::size_t>(contactsPerSystem), "states",
                   "floatingBaseAcceleration"))
        return false;
    return report(blf_sys_floating_base_acceleration(
                      raw(m_device), static_cast<std::int64_t>(nSystems), contactsPerSystem, columns,
                      states.planePointers(), parameters ? parameters->planePointers() : nullptr, jacobians,
                      biasForces, jointTorques, massMatrices, regularization, acceleration,
                      wrench ? wrench->planePointers() : nullptr, stream),
                  "floatingBaseAcceleration");
}

bool ContactRolloutBatch::kinematicsDynamics(std::size_t nSystems, double rho, const double* twists,
                                             const double* rotations, double* linearVelocities,
                                             double* rotationRates, void* stream)
{
    if (m_device == nullptr) return report(BLF_CCM_ERR_INVALID_HANDLE, "kinematicsDynamics");
    return report(blf_sys_kinematics_dynamics(raw(m_device), static_cast<std::int64_t>(nSystems), rho, twists,
                                              rotations, linearVelocities, rotationRates, stream),
                  "kinematicsDynamics");
}

bool ContactRolloutBatch::floatingBaseEulerStep(std::size_t nSystems, int columns, double rho, double dT,
                                                const double* acceleration, double* velocity,
                                                double* jointPositions, double* basePositions,
                                                double* baseRotations, void* stream)
{
    if (m_device == nullptr) return report(BLF_CCM_ERR_INVALID_HANDLE, "floatingBaseEulerStep");
    return report(blf_sys_floating_base_euler_step(raw(m_device), static_cast<std::int64_t>(nSystems), columns,
                                                   rho, dT, acceleration, velocity, jointPositions,
                                                   basePositions, baseRotations, stream),
                  "floatingBaseEulerStep");
}
