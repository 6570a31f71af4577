/**
 * @file DeviceSoA.cpp
 * Device-side structure-of-arrays container over the C ABI's memory helpers.
 */
#include <cstdint>
#include <iostream>
#include <utility>
#include <vector>

#include <BipedalLocomotion/ContactModels/ContinuousContactModelBatch.h>
#include <BipedalLocomotion/GenericContainer/DeviceSoA.h>

#include "blf_ccm.h"

using namespace BipedalLocomotion::GenericContainer;
using BipedalLocomotion::ContactModels::CudaDevice;

namespace
{
blf_ccm_handle* raw(const std::shared_ptr<CudaDevice>& d)
{
    return static_cast<blf_ccm_handle*>(d->handle());
}
} // namespace

DeviceSoA::DeviceSoA(std::shared_ptr<CudaDevice> device, std::size_t planes, std::size_t size,
                     bool compressible)
    : m_device(std::move(device)), m_size(size), m_owning(true)
{
    if (m_device == nullptr || planes == 0) return;
    m_pitch = (size + 31) / 32 * 32; // planes start on 256-byte boundaries
    if (m_pitch == 0) m_pitch = 32;
    const std::uint64_t bytes = planes * m_pitch * sizeof(double);
    const int rc = compressible ? blf_ccm_device_alloc_compressible(raw(m_device), bytes, &m_base, nullptr)
                                : blf_ccm_device_alloc(raw(m_device), bytes, &m_base);
    if (rc != BLF_CCM_OK)
    {
        std::cerr << "[DeviceSoA::DeviceSoA] " << blf_ccm_last_error() << std::endl;
        m_base = nullptr;
        return;
    }
    m_planes.resize(planes);
    for (std::size_t i = 0; i < planes; ++i) m_planes[i] = static_cast<double*>(m_base) + i * m_pitch;
}

DeviceSoA::DeviceSoA(std::shared_ptr<CudaDevice> device, const std::vector<double*>& planes,
                     std::size_t size)
    : m_device(std::move(device)), m_size(size), m_planes(planes), m_owning(false)
{
}

DeviceSoA::~DeviceSoA()
{
    if (m_owning && m_base != nullptr && m_device != nullptr)
        blf_ccm_device_free(raw(m_device), m_base);
}

DeviceSoA::DeviceSoA(DeviceSoA&& o) noexcept { *this = std::move(o); }

DeviceSoA& DeviceSoA::operator=(DeviceSoA&& o) noexcept
{
    if (this == &o) return *this;
    if (m_owning && m_base != nullptr && m_device != nullptr)
        blf_ccm_device_free(raw(m_device), m_base);
    m_device = std::move(o.m_device);
    m_base = o.m_base;
    m_size = o.m_size;
    m_pitch = o.m_pitch;
    m_planes = std::move(o.m_planes);
    m_owning = o.m_owning;
    o.m_base = nullptr;
    o.m_size = 0;
    o.m_planes.clear();
    return *this;
}

bool DeviceSoA::upload(std::size_t plane, const double* host)
{
    if (plane >= m_planes.size() || m_device == nullptr) return false;
    blf_ccm_handle* h = raw(m_device);
    return blf_ccm_copy_h2d(h, m_planes[plane], host, m_size * sizeof(double), nullptr) == BLF_CCM_OK
           && blf_ccm_stream_synchronize(h, nullptr) == BLF_CCM_OK;
}

bool DeviceSoA::download(std::size_t plane, double* host) const
{
    if (plane >= m_planes.size() || m_device == nullptr) return false;
    blf_ccm_handle* h = raw(m_device);
    return blf_ccm_copy_d2h(h, host, m_planes[plane], m_size * sizeof(double), nullptr) == BLF_CCM_OK
           && blf_ccm_stream_synchronize(h, nullptr) == BLF_CCM_OK;
}

bool DeviceSoA::uploadRows(std::size_t firstPlane, std::size_t stride, const double* hostRows)
{
    if (firstPlane + stride > m_planes.size()) return false;
    std::vector<double> column(m_size);
    for (std::size_t j = 0; j < stride; ++j)
    {
        for (std::size_t i = 0; i < m_size; ++i) column[i] = hostRows[i * stride + j];
        if (!upload(firstPlane + j, column.data())) return false;
    }
    return true;
}

bool DeviceSoA::downloadRows(std::size_t firstPlane, std::size_t stride, double* hostRows) const
{
    if (firstPlane + stride > m_planes.size()) return false;
    std::vector<double> column(m_size);
    for (std::size_t j = 0; j < stride; ++j)
    {
        if (!download(firstPlane + j, column.data())) return false;
        for (std::size_t i = 0; i < m_size; ++i) hostRows[i * stride + j] = column[i];
    }
    return true;
}
