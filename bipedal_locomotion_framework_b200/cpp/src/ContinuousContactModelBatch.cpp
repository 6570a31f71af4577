/**
 * @file ContinuousContactModelBatch.cpp
 * Batched entry point: thin C++17 layer over the C ABI (include/blf_ccm.h).
 */
#include <iostream>
#include <vector>

#include <BipedalLocomotion/ContactModels/ContinuousContactModelBatch.h>

#include "blf_ccm.h"

using namespace BipedalLocomotion::ContactModels;
using namespace BipedalLocomotion::GenericContainer;
using namespace BipedalLocomotion::ParametersHandler;

static_assert(sizeof(ContactParameters) == sizeof(blf_ccm_params), "ContactParameters layout");
static_assert(unsigned(ContinuousContactModelBatch::ContactWrench) == BLF_CCM_WRENCH
                  && unsigned(ContinuousContactModelBatch::AutonomousDynamics) == BLF_CCM_AUTODYN
                  && unsigned(ContinuousContactModelBatch::ControlMatrix) == BLF_CCM_CTRL
                  && unsigned(ContinuousContactModelBatch::Regressor) == BLF_CCM_REGRESSOR,
              "output bits");

namespace
{
blf_ccm_handle* raw(const std::shared_ptr<CudaDevice>& d)
{
    return d ? static_cast<blf_ccm_handle*>(d->handle()) : nullptr;
}

bool report(int rc, const char* where)
{
    if (rc == BLF_CCM_OK) return true;
    std::cerr << "[ContinuousContactModelBatch::" << where << "] " << blf_ccm_last_error() << std::endl;
    return false;
}
} // namespace

ContinuousContactModelBatch::ContinuousContactModelBatch(int device) : m_device(CudaDevice::open(device)) {}

ContinuousContactModelBatch::ContinuousContactModelBatch(std::shared_ptr<CudaDevice> device)
    : m_device(std::move(device))
{
}

ContinuousContactModelBatch::~ContinuousContactModelBatch()
{
    if (m_best != nullptr && m_device != nullptr) blf_ccm_device_free(raw(m_device), m_best);
}

bool ContinuousContactModelBatch::initialize(std::weak_ptr<IParametersHandler> weakHandler)
{
    auto handler = weakHandler.lock();
    if (handler == nullptr)
    {
        std::cerr << "[ContinuousContactModelBatch::initialize] The parameter handler is corrupted. "
                     "Please make sure that the handler exists."
                  << std::endl;
        return false;
    }
    double length, width, spring, damper;
    const struct
    {
        const char* key;
        double* value;
    } keys[] = {{"length", &length}, {"width", &width}, {"spring_coeff", &spring}, {"damper_coeff", &damper}};
    for (const auto& k : keys)
        if (!handler->getParameter(k.key, *k.value))
        {
            std::cerr << "[ContinuousContactModelBatch::initialize] Unable to get the variable named "
                      << k.key << "." << std::endl;
            return false;
        }
    if (m_device == nullptr)
    {
        std::cerr << "[ContinuousContactModelBatch::initialize] The CUDA backend is not available and "
                     "there is no CPU evaluation path."
                  << std::endl;
        return false;
    }
    return report(blf_ccm_set_uniform_params(raw(m_device), length, width, spring, damper), "initialize");
}

bool ContinuousContactModelBatch::loadParameterTable(std::weak_ptr<IParametersHandler> weakHandler,
                                                     DeviceSoA& parameters)
{
    auto handler = weakHandler.lock();
    if (handler == nullptr)
    {
        std::cerr << "[ContinuousContactModelBatch::loadParameterTable] The parameter handler is "
                     "corrupted. Please make sure that the handler exists."
                  << std::endl;
        return false;
    }
    const char* keys[4] = {"length", "width", "spring_coeff", "damper_coeff"};
    std::vector<double> column[4];
    for (int k = 0; k < 4; ++k)
    {
        if (!handler->getParameter(keys[k], column[k], BipedalLocomotion::GenericContainer::VectorResizeMode::Resizable))
        {
            std::cerr << "[ContinuousContactModelBatch::loadParameterTable] Unable to get the vector "
                         "named "
                      << keys[k] << "." << std::endl;
            return false;
        }
        if (column[k].size() != column[0].size())
        {
            std::cerr << "[ContinuousContactModelBatch::loadParameterTable] The vector named " << keys[k]
                      << " has " << column[k].size() << " elements, " << keys[0] << " has "
                      << column[0].size() << "." << std::endl;
            return false;
        }
    }
    if (m_device == nullptr)
    {
        std::cerr << "[ContinuousContactModelBatch::loadParameterTable] The CUDA backend is not "
                     "available and there is no CPU evaluation path."
                  << std::endl;
        return false;
    }
    DeviceSoA table(m_device, 4, column[0].size());
    if (!table.valid()) return report(BLF_CCM_ERR_CUDA, "loadParameterTable");
    for (int k = 0; k < 4; ++k)
        if (!table.upload(static_cast<std::size_t>(k), column[k].data())) return false;
    parameters = std::move(table);
    return true;
}

bool ContinuousContactModelBatch::evaluate(const DeviceSoA& states, const DeviceSoA* parameters,
                                           unsigned outputs, DeviceSoA* wrench,
                                           DeviceSoA* autonomousDynamics, double* controlMatrix,
                                           DeviceSoA* regressor, void* stream)
{
    if (m_device == nullptr) return report(BLF_CCM_ERR_INVALID_HANDLE, "evaluate");
    if (states.planes() != NumberOfPlanes)
    {
        std::cerr << "[ContinuousContactModelBatch::evaluate] states must have 30 planes." << std::endl;
        return false;
    }
    return report(blf_ccm_eval_batch_soa(raw(m_device), static_cast<std::int64_t>(states.size()),
                                         states.planePointers(),
                                         parameters ? parameters->planePointers() : nullptr, outputs,
                                         wrench ? wrench->planePointers() : nullptr,
                                         autonomousDynamics ? autonomousDynamics->planePointers() : nullptr,
                                         controlMatrix,
                                         regressor ? regressor->planePointers() : nullptr, stream),
                  "evaluate");
}

bool ContinuousContactModelBatch::wrenchGradient(const DeviceSoA& states, const DeviceSoA* parameters,
                                                 const DeviceSoA& wrenchCotangent,
                                                 DeviceSoA* stateGradient, DeviceSoA* parameterGradient,
                                                 void* stream)
{
    if (m_device == nullptr) return report(BLF_CCM_ERR_INVALID_HANDLE, "wrenchGradient");
    const bool shapes = states.planes() == NumberOfPlanes && wrenchCotangent.planes() == 6
                        && wrenchCotangent.size() == states.size()
                        && (parameters == nullptr || (parameters->planes() == 4 && parameters->size() == states.size()))
                        && (stateGradient == nullptr
                            || (stateGradient->planes() == NumberOfPlanes && stateGradient->size() == states.size()))
                        && (parameterGradient == nullptr
                            || (parameterGradient->planes() == 4 && parameterGradient->size() == states.size()));
    if (!shapes)
    {
        std::cerr << "[ContinuousContactModelBatch::wrenchGradient] states and stateGradient must have 30 "
                     "planes, wrenchCotangent 6, parameters and parameterGradient 4, all of the same size."
                  << std::endl;
        return false;
    }
    return report(blf_ccm_wrench_vjp_soa(raw(m_device), static_cast<std::int64_t>(states.size()),
                                         states.planePointers(),
                                         parameters ? parameters->planePointers() : nullptr,
                                         wrenchCotangent.planePointers(),
                                         stateGradient ? stateGradient->planePointers() : nullptr,
                                         parameterGradient ? parameterGradient->planePointers() : nullptr,
                                         stream),
                  "wrenchGradient");
}

bool ContinuousContactModelBatch::evaluate(std::size_t n, const iDynTree::Twist* twists,
                                           const iDynTree::Transform* transforms,
                                           const iDynTree::Transform* nullForceTransforms,
                                           const ContactParameters* parameters, unsigned outputs,
                                           iDynTree::Wrench* wrenches,
                                           iDynTree::Vector6* autonomousDynamics,
                                           iDynTree::Matrix6x6* controlMatrices, double* regressors)
{
    if (m_device == nullptr) return report(BLF_CCM_ERR_INVALID_HANDLE, "evaluate");
    return report(blf_ccm_eval_batch_host(raw(m_device), static_cast<std::int64_t>(n),
                                          reinterpret_cast<const double*>(twists),
                                          reinterpret_cast<const double*>(transforms),
                                          reinterpret_cast<const double*>(nullForceTransforms),
                                          reinterpret_cast<const blf_ccm_params*>(parameters), outputs,
                                          reinterpret_cast<double*>(wrenches),
                                          reinterpret_cast<double*>(autonomousDynamics),
                                          reinterpret_cast<double*>(controlMatrices), regressors),
                  "evaluate");
}

bool ContinuousContactModelBatch::rolloutCostArgmin(const DeviceSoA& states, const DeviceSoA* parameters,
                                                    std::size_t rolloutLength,
                                                    const iDynTree::Wrench& referenceWrench,
                                                    double forceWeight, double torqueWeight,
                                                    std::int64_t indexBase, double* costs, void* best,
                                                    void* stream)
{
    if (m_device == nullptr) return report(BLF_CCM_ERR_INVALID_HANDLE, "rolloutCostArgmin");
    if (rolloutLength == 0 || states.size() % rolloutLength != 0)
    {
        std::cerr << "[ContinuousContactModelBatch::rolloutCostArgmin] The batch size must be a "
                     "multiple of the rollout length."
                  << std::endl;
        return false;
    }
    const double weights[2] = {forceWeight, torqueWeight};
    return report(blf_ccm_rollout_cost_argmin_soa(raw(m_device),
                                                  static_cast<std::int64_t>(states.size() / rolloutLength),
                                                  static_cast<std::int64_t>(rolloutLength),
                                                  states.planePointers(),
                                                  parameters ? parameters->planePointers() : nullptr, 0u,
                                                  nullptr, nullptr, nullptr, referenceWrench.data(),
                                                  weights, indexBase, costs, best, stream),
                  "rolloutCostArgmin");
}

bool ContinuousContactModelBatch::rolloutCostArgmin(const DeviceSoA& states, const DeviceSoA* parameters,
                                                    std::size_t rolloutLength,
                                                    const iDynTree::Wrench& referenceWrench,
                                                    double forceWeight, double torqueWeight,
                                                    RolloutResult& result)
{
    if (m_device == nullptr) return report(BLF_CCM_ERR_INVALID_HANDLE, "rolloutCostArgmin");
    blf_ccm_handle* h = raw(m_device);
    if (m_best == nullptr && !report(blf_ccm_device_alloc(h, 16, &m_best), "rolloutCostArgmin")) return false;
    if (!rolloutCostArgmin(states, parameters, rolloutLength, referenceWrench, forceWeight, torqueWeight,
                           0, nullptr, m_best, nullptr))
        return false;
    struct
    {
        double cost;
        std::int64_t index;
    } pair;
    if (!report(blf_ccm_copy_d2h(h, &pair, m_best, 16, nullptr), "rolloutCostArgmin")) return false;
    if (!report(blf_ccm_stream_synchronize(h, nullptr), "rolloutCostArgmin")) return false;
    result.cost = pair.cost;
    result.index = pair.index;
    return true;
}
