/**
 * @file DeviceSoA.h
 * Device-side structure-of-arrays container: the GPU companion of GenericContainer::Vector.
 *
 * Owns `planes` arrays of `size` doubles in one device allocation; every plane starts on a
 * 256-byte boundary so the 128-bit / bulk-copy paths of the C ABI are always taken.  Memory is
 * reached only through the C ABI (blf_ccm_device_alloc / blf_ccm_copy_*), so this header needs no
 * CUDA toolkit.  Like GenericContainer::Vector it can also be a non-owning view over planes the
 * caller allocated (e.g. a simulator's own state buffers).
 */
#ifndef BIPEDAL_LOCOMOTION_GENERIC_CONTAINER_DEVICE_SOA_H
#define BIPEDAL_LOCOMOTION_GENERIC_CONTAINER_DEVICE_SOA_H

#include <cstddef>
#include <memory>
#include <vector>

namespace BipedalLocomotion
{
namespace ContactModels
{
class CudaDevice;
}

namespace GenericContainer
{

class DeviceSoA
{
    std::shared_ptr<ContactModels::CudaDevice> m_device;
    void* m_base{nullptr};
    std::size_t m_size{0};
    std::size_t m_pitch{0}; /**< doubles between consecutive planes */
    std::vector<double*> m_planes;
    bool m_owning{true};

public:
    DeviceSoA() = default;
    /** Owning container of `planes` x `size` doubles.  `compressible`: request Compute Data
     * Compression for the allocation (blf_ccm_device_alloc_compressible; plain memory where the
     * device does not grant it), for data with many zeros such as the dense n x 36 control matrix
     * (one plane of 36 n doubles). */
    DeviceSoA(std::shared_ptr<ContactModels::CudaDevice> device, std::size_t planes, std::size_t size,
              bool compressible = false);
    /** Non-owning view over existing device planes. */
    DeviceSoA(std::shared_ptr<ContactModels::CudaDevice> device, const std::vector<double*>& planes,
              std::size_t size);
    ~DeviceSoA();
    DeviceSoA(const DeviceSoA&) = delete;
    DeviceSoA& operator=(const DeviceSoA&) = delete;
    DeviceSoA(DeviceSoA&& other) noexcept;
    DeviceSoA& operator=(DeviceSoA&& other) noexcept;

    bool valid() const { return !m_planes.empty() && (m_size == 0 || m_planes[0] != nullptr); }
    std::size_t size() const { return m_size; }
    std::size_t planes() const { return m_planes.size(); }
    double* plane(std::size_t i) { return m_planes[i]; }
    const double* plane(std::size_t i) const { return m_planes[i]; }
    /** Host array of device pointers, as the C ABI takes it. */
    const double* const* planePointers() const { return m_planes.data(); }
    double* const* planePointers() { return m_planes.data(); }

    /** Copy `size()` doubles from / to host memory for one plane (synchronous). */
    bool upload(std::size_t plane, const double* host);
    bool download(std::size_t plane, double* host) const;
    /**
     * Transpose host array-of-structures rows into the planes: element j of row i goes to
     * plane (firstPlane + j)[i].  `stride` = doubles per row (6 for Twist, 12 for Transform).
     */
    bool uploadRows(std::size_t firstPlane, std::size_t stride, const double* hostRows);
    bool downloadRows(std::size_t firstPlane, std::size_t stride, double* hostRows) const;
};

} // namespace GenericContainer
} // namespace BipedalLocomotion

#endif // BIPEDAL_LOCOMOTION_GENERIC_CONTAINER_DEVICE_SOA_H
