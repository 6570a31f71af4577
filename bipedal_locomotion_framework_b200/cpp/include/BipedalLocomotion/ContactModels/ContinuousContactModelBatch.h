/**
 * @file ContinuousContactModelBatch.h
 * Batched entry point of the continuous contact model: millions of contact states per call, the
 * way a sampling-based MPC rollout or a contact-rich simulator consumes the model.  It has no
 * reference equivalent (the reference evaluates one object per state); the per-state semantics are
 * exactly those of ContinuousContactModel (setState + setNullForceTransform + getters).
 *
 * Host code stays C++17 and reaches the GPU only through the C ABI (include/blf_ccm.h).
 */
#ifndef BIPEDAL_LOCOMOTION_CONTACT_MODELS_CONTINUOUS_CONTACT_MODEL_BATCH_H
#define BIPEDAL_LOCOMOTION_CONTACT_MODELS_CONTINUOUS_CONTACT_MODEL_BATCH_H

#include <cstddef>
#include <cstdint>
#include <memory>

#include <BipedalLocomotion/ContactModels/ContactModel.h>
#include <BipedalLocomotion/GenericContainer/DeviceSoA.h>

namespace BipedalLocomotion
{
namespace ContactModels
{

/** RAII owner of one C-ABI handle (one CUDA device).  Shared by models, batches and containers. */
class CudaDevice
{
    struct Impl;
    std::unique_ptr<Impl> m_impl;

public:
    /** nullptr (and a message on std::cerr) when the device cannot be opened. */
    static std::shared_ptr<CudaDevice> open(int device);
    /** Device the per-instance facades (ContinuousContactModel, RecursiveLeastSquare,
     * FloatingBaseSystemKinematics) open in initialize(): the value given to setDefaultIndex, else
     * $BLF_CCM_DEVICE, else 0. */
    static int defaultIndex();
    static void setDefaultIndex(int device);
    ~CudaDevice();
    void* handle() const; /**< blf_ccm_handle* */
    int index() const;
    std::int64_t kernelLaunches() const;
    const char* lastError() const;

private:
    CudaDevice();
};

/** Per-contact parameters (same keys as ContinuousContactModel::initialize). */
struct ContactParameters
{
    double length;
    double width;
    double springCoeff;
    double damperCoeff;
};

class ContinuousContactModelBatch
{
public:
    enum Output : unsigned
    {
        ContactWrench = 1,
        AutonomousDynamics = 2,
        ControlMatrix = 4,
        Regressor = 8,
        All = 7
    };

    /** Plane order of the structure-of-arrays state (30 planes). */
    enum Plane : unsigned
    {
        LinearVelocity = 0,   // 0-2
        AngularVelocity = 3,  // 3-5
        Position = 6,         // 6-8
        Rotation = 9,         // 9-17 row-major
        NullForcePosition = 18, // 18-20
        NullForceRotation = 21, // 21-29 row-major
        NumberOfPlanes = 30
    };

    struct RolloutResult
    {
        double cost;
        std::int64_t index; /**< -1 when there is nothing to compare */
    };

    explicit ContinuousContactModelBatch(int device = 0);
    explicit ContinuousContactModelBatch(std::shared_ptr<CudaDevice> device);
    ~ContinuousContactModelBatch();
    ContinuousContactModelBatch(const ContinuousContactModelBatch&) = delete;
    ContinuousContactModelBatch& operator=(const ContinuousContactModelBatch&) = delete;

    /** Same four required double parameters as ContinuousContactModel; they apply to every contact
     * of evaluations that pass no per-contact parameters. */
    bool initialize(std::weak_ptr<ParametersHandler::IParametersHandler> handler);

    std::shared_ptr<CudaDevice> device() const { return m_device; }

    /**
     * Per-contact parameter table -> the four device planes `evaluate` takes as `parameters`.
     * The handler (typically a group of a `.ini` file read with ParametersHandler::loadIniFile,
     * the reference's on-disk configuration format) must hold the four keys of initialize() as
     * equally long std::vector<double>: "length", "width", "spring_coeff", "damper_coeff".
     * On success `parameters` owns 4 planes of that length.  No range validation, as initialize().
     */
    bool loadParameterTable(std::weak_ptr<ParametersHandler::IParametersHandler> handler,
                            GenericContainer::DeviceSoA& parameters);

    /**
     * Device-resident structure-of-arrays evaluation (asynchronous on `stream`).
     * @param states 30 planes (Plane order); planes that cannot affect `outputs` may be null
     * @param parameters 4 planes length,width,spring,damper or nullptr for the uniform ones
     * @param wrench 6 planes, autonomousDynamics 6 planes, controlMatrix dense n*36 row-major
     *        device array, regressor 12 planes; each may be nullptr when not requested
     */
    bool evaluate(const GenericContainer::DeviceSoA& states,
                  const GenericContainer::DeviceSoA* parameters, unsigned outputs,
                  GenericContainer::DeviceSoA* wrench,
                  GenericContainer::DeviceSoA* autonomousDynamics, double* controlMatrix,
                  GenericContainer::DeviceSoA* regressor, void* stream = nullptr);

    /**
     * Reverse mode of the contact wrench (asynchronous on `stream`): for per-contact cotangents
     * of the wrench, the vector-Jacobian products with respect to the state and the parameters.
     * @param states 30 planes (Plane order); planes no requested gradient reads may be null
     * @param parameters 4 planes length,width,spring,damper or nullptr for the uniform ones
     * @param wrenchCotangent 6 planes force xyz, torque xyz; a null plane counts as zero
     * @param stateGradient 30 planes or nullptr; every non-null plane is written (R02, R12 and the
     *        null-force rotation's third column with +0.0), the others are neither computed nor written
     * @param parameterGradient 4 planes or nullptr: each contact's gradient with respect to
     *        length, width, spring, damper (with uniform parameters, their sum over contacts)
     */
    bool wrenchGradient(const GenericContainer::DeviceSoA& states,
                        const GenericContainer::DeviceSoA* parameters,
                        const GenericContainer::DeviceSoA& wrenchCotangent,
                        GenericContainer::DeviceSoA* stateGradient,
                        GenericContainer::DeviceSoA* parameterGradient, void* stream = nullptr);

    /**
     * Host arrays of iDynTree objects in, host arrays of iDynTree objects out (what a loop over
     * ContactModel instances would produce).  Copies and kernels are pipelined; returns when the
     * results are in host memory.
     */
    bool evaluate(std::size_t n, const iDynTree::Twist* twists, const iDynTree::Transform* transforms,
                  const iDynTree::Transform* nullForceTransforms, const ContactParameters* parameters,
                  unsigned outputs, iDynTree::Wrench* wrenches,
                  iDynTree::Vector6* autonomousDynamics, iDynTree::Matrix6x6* controlMatrices,
                  double* regressors = nullptr);

    /**
     * Sampling-MPC epilogue on a rollout-major device batch: evaluates, reduces
     * cost[r] = sum_e wf |force - ref.force|^2 + wt |torque - ref.torque|^2 and returns the local
     * arg-min (index offset by indexBase) -- one kernel launch.  `best` is 16 device bytes
     * {double cost, int64 index}; costs (device, nRollouts) may be nullptr.
     */
    bool rolloutCostArgmin(const GenericContainer::DeviceSoA& states,
                           const GenericContainer::DeviceSoA* parameters, std::size_t rolloutLength,
                           const iDynTree::Wrench& referenceWrench, double forceWeight,
                           double torqueWeight, std::int64_t indexBase, double* costs, void* best,
                           void* stream = nullptr);
    /** Same, then copies the pair to the host (synchronises the stream). */
    bool rolloutCostArgmin(const GenericContainer::DeviceSoA& states,
                           const GenericContainer::DeviceSoA* parameters, std::size_t rolloutLength,
                           const iDynTree::Wrench& referenceWrench, double forceWeight,
                           double torqueWeight, RolloutResult& result);

private:
    std::shared_ptr<CudaDevice> m_device;
    void* m_best{nullptr}; /**< 16 device bytes for the synchronous rolloutCostArgmin */
};

} // namespace ContactModels
} // namespace BipedalLocomotion

#endif // BIPEDAL_LOCOMOTION_CONTACT_MODELS_CONTINUOUS_CONTACT_MODEL_BATCH_H
